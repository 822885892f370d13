"""Drop-in for `sitrack.ncio` (reference: sitrack/ncio.py).  Host-side I/O stays Python.

netCDF4 is imported lazily (it is not installed in the build image).  Every reader and
the writer also accept `.npz` files holding the SAME variable names, dtypes and leading
singleton dimensions, so the whole CLI runs on synthetic data without netCDF:
  mesh_mask : tmask glamt gphit glamf gphif glamu gphiu glamv gphiv e1t e2t
  SI3 file  : time_counter siconc u_ice v_ice
  buoy file : time id_buoy latitude longitude y_pos x_pos [mask] [time_pos]
The km coordinates of the grid come from the device projection kernel
(ConvertGeo2CartesianNPSkm -> st_latlon2xy) instead of cartopy.
"""
import math
import os
import re
import shutil
import sys
import tempfile
import zipfile

import numpy as np

from .util import chck4f, ConvertGeo2CartesianNPSkm
from .util import epoch2clock as e2c

__all__ = ["tunits_default", "FillValue", "GetModelGrid", "GetModelUVGrid", "GetSeedMask",
           "GetModelSeaIceConc", "ncSaveCloudBuoys", "LoadNCtime", "LoadNCdata", "SeedFileTimeInfo",
           "ModelFileTimeInfo", "open_dataset", "CloudBuoyWriter", "DeformationWriter",
           "DeformationScalingWriter", "DeformationGridWriter", "DispersionWriter", "FsleWriter", "SampleWriter"]

tunits_default = 'seconds since 1970-01-01 00:00:00'     # ncio.py:15
FillValue = -9999.                                       # ncio.py:19

_TIME_VARS = ("time", "time_counter", "time_pos")
_DIM_OF = {"time_counter": "time_counter", "time": "time", "id_buoy": "buoy"}


def _die(msg):
    print(msg)
    raise SystemExit(0)


class _Var:
    """Array with a `.units` attribute, indexable like a netCDF4 variable."""

    def __init__(self, data, units=None):
        self._d, self.units = data, units

    def __getitem__(self, key):
        return self._d[key]

    shape = property(lambda self: self._d.shape)


class _Dim:
    def __init__(self, size):
        self.size = size


class _NpzDataset:
    """Read-only stand-in for netCDF4.Dataset over an .npz with the same variable names."""

    def __init__(self, fn):
        self._z = np.load(fn, allow_pickle=False)
        names = self._z.files
        self.variables = {n: _Var(self._z[n], tunits_default if n in _TIME_VARS else None) for n in names}
        self.dimensions = {d: _Dim(self._z[v].shape[0]) for v, d in _DIM_OF.items() if v in names}

    def close(self):
        self._z.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def open_dataset(fn):
    """netCDF4.Dataset(fn), or the npz stand-in when `fn` ends in .npz."""
    if str(fn).endswith(".npz"):
        return _NpzDataset(fn)
    try:
        import netCDF4
    except ImportError as e:
        raise ImportError("netCDF4 is needed to read '%s' (or pass the .npz equivalent)" % fn) from e
    return netCDF4.Dataset(fn)


def _plane(var):
    """The horizontal (Nj,Ni) plane of a mesh_mask variable: first time record / first level, as the reference
    indexes them (ncio.py:28-36: `[0,0,:,:]` for the masks, `[0,:,:]` for coordinates and scale factors).  A real
    NEMO mesh_mask stores tmask / fmask as (t,z,y,x) with z > 1; only the surface plane is read."""
    nd = len(var.shape)
    return np.asarray(var[(0,) * (nd - 2) + (slice(None), slice(None))])


def _keep_mask(a):
    """netCDF4 hands out masked arrays; keep the mask when it hides something (the reference does, and its
    np.min / np.max then skip the fill values, ncio.py:341), plain ndarray otherwise."""
    return a if isinstance(a, np.ma.MaskedArray) and np.ma.is_masked(a) else np.asarray(a)


def _read_planes(fn, names):
    chck4f(fn)
    with open_dataset(fn) as ds:
        return [_plane(ds.variables[n]) for n in names]


def _to_km(lat, lon):
    return ConvertGeo2CartesianNPSkm(lat, np.mod(lon, 360.))


def GetModelGrid(fNCmeshmask, alsoF=False):
    """ncio.py:22-63 -> kmaskt, latT, lonT(0..360), Yt, Xt, Yf, Xf [km], ResKM [, kmaskf, latF, lonF]"""
    want = ['tmask', 'glamt', 'gphit', 'glamf', 'gphif', 'e1t', 'e2t'] + (['fmask'] if alsoF else [])
    got = dict(zip(want, _read_planes(fNCmeshmask, want)))
    kmaskt = np.array(got['tmask'], dtype='i1')
    lonT, lonF = np.mod(got['glamt'], 360.), np.mod(got['glamf'], 360.)
    Yt, Xt = _to_km(got['gphit'], lonT)
    Yf, Xf = _to_km(got['gphif'], lonF)
    e1, e2 = got['e1t'] / 1000., got['e2t'] / 1000.
    res = np.asarray(np.sqrt(e1 * e1 + e2 * e2), dtype=np.float64)
    base = (kmaskt, got['gphit'], lonT, Yt, Xt, Yf, Xf, res)
    return base + (got['fmask'], got['gphif'], lonF) if alsoF else base


def GetModelUVGrid(fNCmeshmask):
    """ncio.py:66-92 -> Yv, Xv, Yu, Xu [km]"""
    lonV, latV, lonU, latU = _read_planes(fNCmeshmask, ['glamv', 'gphiv', 'glamu', 'gphiu'])
    return _to_km(latV, lonV) + _to_km(latU, lonU)


def GetSeedMask(fFSmask, mvar='tmask'):
    chck4f(fFSmask)
    with open_dataset(fFSmask) as ds:
        return np.array(ds.variables[mvar][:, :], dtype='i1')


def GetModelSeaIceConc(fNCsi3, name='siconc', krec=0, expected_shape=[]):
    chck4f(fNCsi3)
    print('    * [GetModelSeaIceConc]: reading "%s" at record %d in %s !' % (name, krec, fNCsi3))
    with open_dataset(fNCsi3) as ds:
        sic = np.asarray(ds.variables[name][krec, :, :])
    if len(expected_shape) > 0 and sic.shape != tuple(expected_shape):
        _die('ERROR [GetModelSeaIceConc]: wrong shape for sea-ice concentration read: %s, expected: %s'
             % (sic.shape, expected_shape))
    return sic


class _OutFile:
    """One output file of the writers below, created with its dimensions `dims` (name -> size; `time` is unlimited
    on netCDF4) and global attributes About, Author, Origin (corigin, if given) and `attrs`.

    netCDF4 when it imports and the name does not end in .npz; otherwise `<name>.npz` with the same variables, each an
    on-disk .npy member (numpy memmap) in a temporary directory next to the output, zipped (deflate) at close, never
    held in memory.  The .npz also holds the `attrs` as members, a 0-d string member `<name>_units` for every variable
    with units and, with `fill` given, a `FillValue` member of fill's type; npz_attrs=False (the cloud-of-buoys file,
    which mirrors the reference's file that LoadNCdata reads back) leaves out all of these.  Variables are `_v[name]`,
    written by index like netCDF4 variables."""

    def __init__(self, cf_out, who, dims, about, corigin=None, fill=None, npz_attrs=True, **attrs):
        print('\n *** [%s]: About to generate file: %s ...' % (who, cf_out))
        nc = None
        if not str(cf_out).endswith(".npz"):
            try:
                import netCDF4 as nc
            except ImportError:
                cf_out += ".npz"
                print('      (netCDF4 not available: writing ' + cf_out + ' with the same variables)')
        self.cf_out, self._nc, self.dims, self.fill, self._npz_attrs = cf_out, nc, dims, fill, npz_attrs
        self._v = {}
        if nc is None:
            self._tmp = tempfile.mkdtemp(prefix=".sitrack_", dir=os.path.dirname(os.path.abspath(cf_out)) or ".")
            if npz_attrs:
                if fill is not None:
                    attrs['FillValue'] = fill
                for n, a in attrs.items():
                    np.save(os.path.join(self._tmp, n + ".npy"), a)
        else:
            f = self._f = nc.Dataset(cf_out, 'w', format='NETCDF4')
            for d, n in dims.items():
                f.createDimension(d, None if d == 'time' else n)
            for n, a in attrs.items():
                setattr(f, n, a)
            if corigin:
                f.Origin = corigin
            f.About = about
            f.Author = 'Generated with `%s` of `sitrack` (L. Brodeau, 2023)' % os.path.basename(sys.argv[0])

    def var(self, name, dtype, dims, units=None, fill=False, zlib=False, data=None):
        """Variable `name` over the dimensions `dims`; fill: with the file's fill value; zlib: compressed on netCDF4
        (every .npz member is); data: its whole content."""
        if self._nc is None:
            v = np.lib.format.open_memmap(os.path.join(self._tmp, name + ".npy"), mode='w+', dtype=dtype,
                                          shape=tuple(self.dims[d] for d in dims))
            if units is not None and self._npz_attrs:
                np.save(os.path.join(self._tmp, name + "_units.npy"), np.array(units))
        else:
            kw = dict(fill_value=self.fill) if fill else {}
            v = self._f.createVariable(name, dtype, dims, **kw, **(dict(zlib=True, complevel=9) if zlib else {}))
            if units is not None:
                v.units = units
        if data is not None:
            v[:] = data
        self._v[name] = v

    def close(self):
        if self._nc is not None:
            self._f.close()
        else:
            for v in self._v.values():
                v.flush()
            self._v = {}
            with zipfile.ZipFile(self.cf_out, 'w', zipfile.ZIP_DEFLATED, allowZip64=True) as z:
                for fn in sorted(os.listdir(self._tmp)):
                    z.write(os.path.join(self._tmp, fn), arcname=fn)         # streamed from disk
            shutil.rmtree(self._tmp, ignore_errors=True)
        print('      ===> ' + self.cf_out + ' saved!')

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


# (variable, dtype, units) of the buoy-cloud file, ncio.py:153-172
_CLOUD_VARS = [
    ('latitude', 'f4', 'degrees north'), ('longitude', 'f4', 'degrees south'),      # sic (ncio.py:164)
    ('y_pos', 'f4', 'km'), ('x_pos', 'f4', 'km'),
]


class CloudBuoyWriter(_OutFile):
    """Record-by-record writer of a cloud-of-buoys file: the variables, dtypes and attributes of ncSaveCloudBuoys
    (reference ncio.py:131-197), one `write(jt, ...)` per trajectory row, so that a run never has to hold the
    (Nt+1, nP, 2) series the reference allocates (si3_part_tracker.py:326-328; SURVEY section 5 "output volume").
    netCDF4 (unlimited `time` dimension, rows appended as they come) or an .npz with the same variables and no other
    member (see _OutFile)."""

    def __init__(self, cf_out, ntime, pIDs, with_mask=False, with_time_pos=False, tunits=tunits_default,
                 fillVal=FillValue, corigin=None):
        self.ntime, self.nP = int(ntime), int(np.shape(pIDs)[0])
        super().__init__(cf_out, 'ncSaveCloudBuoys', dict(time=self.ntime, buoy=self.nP), 'Lagrangian sea-ice drift',
                         corigin, fill=fillVal, npz_attrs=False)
        self.names = [n for n, _, _ in _CLOUD_VARS] + (['mask'] if with_mask else []) + (['time_pos'] if with_time_pos else [])
        self.var('time', 'i4', ('time',), units=tunits)
        self.var('buoy', 'i4', ('buoy',), data=np.arange(self.nP, dtype='i8'))
        self.var('id_buoy', 'i8', ('buoy',), units='ID of buoy', data=np.asarray(pIDs))
        for name, dt, units in _CLOUD_VARS:
            self.var(name, dt, ('time', 'buoy'), units=units, fill=True, zlib=True)
        if with_mask:
            self.var('mask', 'i1', ('time', 'buoy'), zlib=True)
        if with_time_pos:
            self.var('time_pos', 'i4', ('time', 'buoy'), units=tunits, fill=True, zlib=True)

    def write(self, jt, time, y, x, lat, lon, mask=None, time_pos=None):
        """Row jt of every variable ((nP,) arrays, any float dtype: stored as f4 like the reference's file)."""
        self._v['time'][jt] = time
        row = dict(latitude=lat, longitude=lon, y_pos=y, x_pos=x, mask=mask, time_pos=time_pos)
        for n in self.names:
            self._v[n][jt, :] = np.asarray(row[n])


class DeformationWriter(_OutFile):
    """Window-by-window writer of the strain rates of buoy triangles (sitrack_b200.deform, TrackEngine.track's
    `deform`).  Dimensions time (windows), triangle, vertex = 3; variables
      time_start, time_end (time) i4          first and last date of each window [tunits]
      vertices (triangle,vertex) i4           indices into the `buoy` axis of the tracking file
      id_vertices (triangle,vertex) i8        IDs of those buoys
      divergence, shear, vorticity (time,triangle) f4 [day-1]; area f4 [km2]; y_ctr, x_ctr f4 [km]
    each output with `units` and the fill value `fillVal` for invalid triangles.  netCDF4 or an .npz with the same
    variables, `<name>_units` and an f4 `FillValue` (see _OutFile)."""

    def __init__(self, cf_out, ntime, tri, pIDs, tunits=tunits_default, fillVal=FillValue, corigin=None):
        from .deform import DEFORM_NAMES, DEFORM_UNITS
        tri = np.asarray(tri).reshape(-1, 3)
        self.ntime, self.nT = int(ntime), tri.shape[0]
        self.names = DEFORM_NAMES
        ids = np.asarray(pIDs).astype('i8')[tri] if self.nT else np.zeros((0, 3), 'i8')
        super().__init__(cf_out, 'DeformationWriter', dict(time=self.ntime, triangle=self.nT, vertex=3),
                         'Sea-ice deformation rates of buoy triangles', corigin, fill=np.float32(fillVal))
        for n in ('time_start', 'time_end'):
            self.var(n, 'i4', ('time',), units=tunits)
        self.var('vertices', 'i4', ('triangle', 'vertex'), data=tri)
        self.var('id_vertices', 'i8', ('triangle', 'vertex'), units='ID of buoy', data=ids)
        for n in self.names:
            self.var(n, 'f4', ('time', 'triangle'), units=DEFORM_UNITS[n], fill=True, zlib=True)

    def write(self, jw, time_start, time_end, out):
        """Window jw: out = dict of (nT,) arrays over the six outputs."""
        self._v['time_start'][jw] = time_start
        self._v['time_end'][jw] = time_end
        for n in self.names:
            self._v[n][jw, :] = np.asarray(out[n], dtype=np.float32)


class DeformationScalingWriter(_OutFile):
    """Window-by-window writer of the per-scale statistics of coarse-grained deformation (sitrack_b200.deform_scales,
    TrackEngine.track's `deform` with `scales`).  Dimensions time (windows), scale, bin, bin_edge; variables
      time_start, time_end (time) i4                       first and last date of each window [tunits]
      scale_km (scale) f8                                  box side [km]; fillVal for the triangles (scale 0)
      bin_edges (bin_edge) f8                              histogram edges [day-1]
      n (time,scale) i8                                    cells (boxes or triangles) that count
      L_eff, eps_tot, eps_tot2, eps_tot3 (time,scale) f8   means of sqrt(area) [km] and of eps_tot^q [day-q],
                                                           fillVal where n = 0
      hist_total, hist_divergence, hist_shear (time,scale,bin) i8   counts of eps_tot, |div|, shear per bin,
                                                           bin k = [edge k-1, edge k), underflow and overflow first/last
    with `units` on every variable.  netCDF4 or an .npz with the same variables, `<name>_units` and an f8
    `FillValue` (see _OutFile)."""

    MEANS = (("L_eff", "sum_L_eff", "km"), ("eps_tot", "sum_eps_tot", "day-1"), ("eps_tot2", "sum_eps_tot2", "day-2"),
             ("eps_tot3", "sum_eps_tot3", "day-3"))
    HISTS = ("hist_total", "hist_divergence", "hist_shear")

    def __init__(self, cf_out, ntime, scale_km, bin_edges, tunits=tunits_default, fillVal=FillValue, corigin=None):
        scale_km, bin_edges = np.asarray(scale_km, 'f8'), np.asarray(bin_edges, 'f8')
        self.ntime, self.ns, self.nbin = int(ntime), scale_km.size, bin_edges.size + 1
        super().__init__(cf_out, 'DeformationScalingWriter',
                         dict(time=self.ntime, scale=self.ns, bin=self.nbin, bin_edge=bin_edges.size),
                         'Per-scale statistics of sea-ice deformation coarse-grained over material boxes of buoy '
                         'triangles', corigin, fill=np.float64(fillVal))
        for n in ('time_start', 'time_end'):
            self.var(n, 'i4', ('time',), units=tunits)
        self.var('n', 'i8', ('time', 'scale'), units='1')
        for n, _, u in self.MEANS:
            self.var(n, 'f8', ('time', 'scale'), units=u, fill=True)
        for h in self.HISTS:
            self.var(h, 'i8', ('time', 'scale', 'bin'), units='1')
        self.var('scale_km', 'f8', ('scale',), units='km', data=scale_km)
        self.var('bin_edges', 'f8', ('bin_edge',), units='day-1', data=bin_edges)

    def write(self, jw, time_start, time_end, stats):
        """Window jw: stats = the dict of sitrack_b200.CoarseGrainedRates / track(deform=dict(scales=...))."""
        n = np.asarray(stats['n'], 'i8')
        self._v['time_start'][jw] = time_start
        self._v['time_end'][jw] = time_end
        self._v['n'][jw, :] = n
        with np.errstate(all='ignore'):
            for name, key, _ in self.MEANS:
                self._v[name][jw, :] = np.where(n > 0, np.asarray(stats[key], 'f8') / np.maximum(n, 1), self.fill)
        for h in self.HISTS:
            self._v[h][jw, :, :] = np.asarray(stats[h], 'i8')


class DeformationGridWriter(_OutFile):
    """Window-by-window writer of deformation coarse-grained over the cells of a fixed Eulerian grid
    (sitrack_b200.deform_grid, TrackEngine.track's `deform` with `grid`).  Dimensions time (windows) and, per level
    s = 1..levels, y<s>, x<s>; variables
      time_start, time_end (time) i4                       first and last date of each window [tunits]
      y<s> (y<s>), x<s> (x<s>) f8                          cell-centre coordinates [km] on the tracking plane
      <name>_<s> (time,y<s>,x<s>) f4                       divergence, shear, vorticity, total [day-1], L_eff [km],
                                                           y_ctr, x_ctr [km]; fillVal where the cell does not count
    with `units` on every variable and the attributes L_km (cell side per level), cover and origin ([y, x] km of the
    grid's corner); corigin, if given, as `Origin`.  netCDF4 or an .npz with the same variables, `L_km`, `cover`,
    `origin`, `<name>_units` and an f4 `FillValue` (see _OutFile)."""

    UNITS = dict(divergence='day-1', shear='day-1', vorticity='day-1', total='day-1', L_eff='km', y_ctr='km',
                 x_ctr='km')

    def __init__(self, cf_out, ntime, G, tunits=tunits_default, fillVal=FillValue, corigin=None):
        from .deform_scales import BOX_NAMES
        self.ntime, self.levels, self.names = int(ntime), G.levels, BOX_NAMES
        dims = dict(time=self.ntime)
        for s, (nj, ni) in enumerate(G.shapes):
            dims['y%d' % (s + 1)], dims['x%d' % (s + 1)] = nj, ni
        super().__init__(cf_out, 'DeformationGridWriter', dims,
                         'Sea-ice deformation of buoy triangles coarse-grained over the cells of a fixed grid', corigin,
                         fill=np.float32(fillVal), L_km=np.asarray(G.L_km, 'f8'), cover=float(G.cover),
                         origin=np.asarray(G.origin, 'f8'))
        for n in ('time_start', 'time_end'):
            self.var(n, 'i4', ('time',), units=tunits)
        for s, (y, x) in enumerate(G.centres(s) for s in range(G.levels)):
            dy, dx = 'y%d' % (s + 1), 'x%d' % (s + 1)
            self.var(dy, 'f8', (dy,), units='km', data=y)
            self.var(dx, 'f8', (dx,), units='km', data=x)
            for n in self.names:
                self.var(self.field(n, s), 'f4', ('time', dy, dx), units=self.UNITS[n], fill=True, zlib=True)

    @staticmethod
    def field(n, s):
        return '%s_%d' % (n, s + 1)

    def write(self, jw, time_start, time_end, fields):
        """Window jw: fields = per level dicts of (nj_s, ni_s) planes (sitrack_b200.GriddedRates, track's grid_sink)."""
        self._v['time_start'][jw] = time_start
        self._v['time_end'][jw] = time_end
        for s in range(self.levels):
            for n in self.names:
                self._v[self.field(n, s)][jw, :, :] = np.asarray(fields[s][n], dtype=np.float32)


class DispersionWriter(_OutFile):
    """Window-by-window writer of the per-lag, per-class statistics of pair dispersion (sitrack_b200.dispersion,
    TrackEngine.track's `dispersion`).  Dimensions time (windows), lag, class, bin, class_edge, bin_edge; variables
      time_start, time_end (time) i4                 first and last date of each window [tunits]
      lag_days (lag) f8                              time lag [day]
      r_edges (class_edge) f8                        initial-separation class edges [km]
      bin_edges (bin_edge) f8                        stretch-rate histogram edges [day-1]
      n (time,lag,class) i8                          pairs that count
      sum_r0, sum_dr, sum_dr2, sum_dD2 (time,lag,class) f8   sums of r0 [km], dr [km], dr^2 [km2], dD2 [km2]
      hist_stretch (time,lag,class,bin) i8           counts of the stretch rate |dr| / (r0 tau) per bin
    with `units` on every variable.  Sums, not means, so that windows add up to ensembles; no variable has a fill value
    (a lag not reached yet has zero counts and sums).  netCDF4 or an .npz with the same variables and `<name>_units`
    (see _OutFile)."""

    SUMS = (("sum_r0", "km"), ("sum_dr", "km"), ("sum_dr2", "km2"), ("sum_dD2", "km2"))

    def __init__(self, cf_out, ntime, lag_days, r_edges, bin_edges, tunits=tunits_default, corigin=None):
        lag_days, r_edges, bin_edges = (np.asarray(a, 'f8') for a in (lag_days, r_edges, bin_edges))
        self.ntime = int(ntime)
        super().__init__(cf_out, 'DispersionWriter',
                         dict(time=self.ntime, lag=lag_days.size, **{'class': r_edges.size + 1}, bin=bin_edges.size + 1,
                              class_edge=r_edges.size, bin_edge=bin_edges.size),
                         'Two-particle dispersion of buoy pairs over time lags, by initial separation', corigin)
        for n in ('time_start', 'time_end'):
            self.var(n, 'i4', ('time',), units=tunits)
        self.var('n', 'i8', ('time', 'lag', 'class'), units='1')
        for n, u in self.SUMS:
            self.var(n, 'f8', ('time', 'lag', 'class'), units=u)
        self.var('hist_stretch', 'i8', ('time', 'lag', 'class', 'bin'), units='1')
        self.var('lag_days', 'f8', ('lag',), units='day', data=lag_days)
        self.var('r_edges', 'f8', ('class_edge',), units='km', data=r_edges)
        self.var('bin_edges', 'f8', ('bin_edge',), units='day-1', data=bin_edges)

    def write(self, jw, time_start, time_end, stats):
        """Window jw: stats = the dict of sitrack_b200.PairDispersion / track(dispersion=...)."""
        self._v['time_start'][jw] = time_start
        self._v['time_end'][jw] = time_end
        self._v['n'][jw] = np.asarray(stats['n'], 'i8')
        for n, _ in self.SUMS:
            self._v[n][jw] = np.asarray(stats[n], 'f8')
        self._v['hist_stretch'][jw] = np.asarray(stats['hist_stretch'], 'i8')


class FsleWriter(_OutFile):
    """Window-by-window writer of the exit-time statistics of finite-size Lyapunov exponents (sitrack_b200.fsle,
    TrackEngine.track's `fsle`).  Dimensions time (windows), threshold (K), transition (K-1), tau_bin, plus level
    (K+1) and tau_edge; variables
      time_start, time_end (time) i4                 first and last date of each window [tunits]
      delta_km (threshold) f8                        separation thresholds [km]
      tau_edges (tau_edge) f8                        exit-time histogram edges [sample]
      n_start (time,level) i8                        pairs that started with that many thresholds reached
      n, n_censored (time,transition) i8             exit times recorded; timed transitions cut by a pair's end
      sum_tau, sum_tau2 (time,transition) i8         sums of the exit times [sample] and of their squares [sample2]
      hist_tau (time,transition,tau_bin) i8          counts of the exit times per bin
    with `units` on every variable and the global attribute sample_days (the length of one sample in days).  Sums,
    not means, so that windows add up to the run; no variable has a fill value.  netCDF4 or an .npz with the same
    variables, `<name>_units` and `sample_days` (see _OutFile)."""

    COUNTS = (("n", "1"), ("sum_tau", "sample"), ("sum_tau2", "sample2"), ("n_censored", "1"))

    def __init__(self, cf_out, ntime, deltas_km, tau_edges, sample_days, tunits=tunits_default, corigin=None):
        deltas_km, tau_edges = np.asarray(deltas_km, 'f8'), np.asarray(tau_edges, 'f8')
        self.ntime, K = int(ntime), deltas_km.size
        super().__init__(cf_out, 'FsleWriter',
                         dict(time=self.ntime, threshold=K, transition=K - 1, tau_bin=tau_edges.size + 1,
                              level=K + 1, tau_edge=tau_edges.size),
                         'Finite-size Lyapunov exponents of buoy pairs: exit times between separation thresholds',
                         corigin, sample_days=float(sample_days))
        for n in ('time_start', 'time_end'):
            self.var(n, 'i4', ('time',), units=tunits)
        self.var('n_start', 'i8', ('time', 'level'), units='1')
        for n, u in self.COUNTS:
            self.var(n, 'i8', ('time', 'transition'), units=u)
        self.var('hist_tau', 'i8', ('time', 'transition', 'tau_bin'), units='1')
        self.var('delta_km', 'f8', ('threshold',), units='km', data=deltas_km)
        self.var('tau_edges', 'f8', ('tau_edge',), units='sample', data=tau_edges)

    def write(self, jw, time_start, time_end, stats):
        """Window jw: stats = a window's dict of sitrack_b200.FiniteSizeLyapunov / track(fsle=...)."""
        self._v['time_start'][jw] = time_start
        self._v['time_end'][jw] = time_end
        for n in ('n_start', 'hist_tau') + tuple(n for n, _ in self.COUNTS):
            self._v[n][jw] = np.asarray(stats[n], 'i8')


class SampleWriter(_OutFile):
    """Row-by-row writer of SI3 fields sampled along the trajectories (sitrack_b200.sample, TrackEngine.track's
    `sample`).  Dimensions time (sampled rows), buoy (the tracking file's buoy axis); variables
      time (time) i4                 the date of each sampled row [tunits]
      id_buoy (buoy) i8              IDs of the buoys
      <name> (time,buoy) f4          one per field, named like the SI3 variable, with its units when given and the
                                     fill value fillVal where the buoy is masked or the value is missing
    and the global attributes interp ("cell" or "bilinear") and every (records between sampled rows).  netCDF4 or an
    .npz with the same variables, `<name>_units`, `interp`, `every` and an f4 `FillValue` (see _OutFile)."""

    def __init__(self, cf_out, ntime, pIDs, names, interp, every, units=None, tunits=tunits_default,
                 fillVal=FillValue, corigin=None):
        self.ntime, self.nP, self.names = int(ntime), int(np.shape(pIDs)[0]), list(names)
        units = units or {}
        super().__init__(cf_out, 'SampleWriter', dict(time=self.ntime, buoy=self.nP),
                         'SI3 fields sampled along Lagrangian sea-ice trajectories', corigin, fill=np.float32(fillVal),
                         interp=str(interp), every=int(every))
        self.var('time', 'i4', ('time',), units=tunits)
        self.var('id_buoy', 'i8', ('buoy',), units='ID of buoy', data=np.asarray(pIDs))
        for n in self.names:
            self.var(n, 'f4', ('time', 'buoy'), units=units.get(n), fill=True, zlib=True)

    def write(self, js, time, values):
        """Sampled row js: values = {name: (nP,) f4} (sitrack_b200.SampleFields / track(sample=...))."""
        self._v['time'][js] = time
        for n in self.names:
            self._v[n][js, :] = np.asarray(values[n], 'f4')


def ncSaveCloudBuoys(cf_out, ptime, pIDs, pY, pX, pLat, pLon, mask=[], xtime=[],
                     tunits=tunits_default, fillVal=FillValue, corigin=None):
    """ncio.py:131-197: time i4, buoy i4, id_buoy i8, latitude/longitude/y_pos/x_pos f4 (time,buoy)
    [+ mask i1, time_pos i4].  netCDF4 when available and the name does not end in .npz, otherwise an
    .npz with the same variables and dtypes.  (Whole arrays in, like upstream; CloudBuoyWriter streams.)"""
    shp = (np.shape(ptime)[0], np.shape(pIDs)[0])
    fields = dict(latitude=pLat, longitude=pLon, y_pos=pY, x_pos=pX)
    if any(np.shape(a) != shp for a in fields.values()):
        _die('ERROR [ncSaveCloudBuoys]: one of the 2D arrays has a wrong shape!!!')
    wm, wt = np.shape(mask) == shp, np.shape(xtime) == shp
    with CloudBuoyWriter(cf_out, shp[0], pIDs, with_mask=wm, with_time_pos=wt, tunits=tunits, fillVal=fillVal,
                         corigin=corigin) as w:
        for jt in range(shp[0]):
            w.write(jt, ptime[jt], pY[jt], pX[jt], pLat[jt], pLon[jt], mask=mask[jt] if wm else None,
                    time_pos=xtime[jt] if wt else None)
    return 0


def _need(ds, kind, names, who):
    have = ds.dimensions if kind == 'dimensions' else ds.variables
    for n in names:
        if n not in have:
            _die(' ERROR [%s()]: no %s `%s` found into input file!' % (who, kind, n))


def _check_tunits(v, who):
    u = getattr(v, "units", tunits_default)
    if u is not None and u != tunits_default:
        _die(' ERROR [%s()]: we expect "%s" as units for the time record vector, yet we have: %s'
             % (who, tunits_default, u))


def LoadNCtime(cfile, ltime2d=False, iverbose=0):
    """ncio.py:199-239 -> Nt, time [, time_pos]"""
    chck4f(cfile)
    with open_dataset(cfile) as ds:
        _need(ds, 'dimensions', ['time'], 'LoadNCtime')
        _need(ds, 'variables', ['time'] + (['time_pos'] if ltime2d else []), 'LoadNCtime')
        Nt = ds.dimensions['time'].size
        _check_tunits(ds.variables['time'], 'LoadNCtime')
        print('    * [LoadNCtime] => reading "time" (%d records) in file %s' % (Nt, os.path.basename(cfile)))
        t1d = _keep_mask(ds.variables['time'][:])
        if not ltime2d:
            return Nt, t1d
        _check_tunits(ds.variables['time_pos'], 'LoadNCtime')
        t2d = _keep_mask(ds.variables['time_pos'][:, :])
    if t2d.shape[0] != Nt:
        _die(' ERROR [LoadNCtime()]: array `time_pos` has not the same number of records as `time`!!!')
    return Nt, t1d, t2d


def LoadNCdata(cfile, krec=-1, lmask=False, lGetTimePos=False, iverbose=0):
    """ncio.py:243-326 -> time, IDs, LatLon (..,nP,2) with lon in 0..360, YX (..,nP,2) [, mask][, time_pos]"""
    chck4f(cfile)
    with open_dataset(cfile) as ds:
        _need(ds, 'dimensions', ['time', 'buoy'], 'LoadNCdata')
        _need(ds, 'variables', ['id_buoy', 'latitude', 'longitude', 'y_pos', 'x_pos']
              + (['time_pos'] if lGetTimePos else []), 'LoadNCdata')
        Nt, nP = ds.dimensions['time'].size, ds.dimensions['buoy'].size
        _check_tunits(ds.variables['time'], 'LoadNCdata')
        rec = krec if krec >= 0 else slice(None)
        grab = lambda n: np.array(ds.variables[n][rec, :])
        ztime = np.asarray(ds.variables['time'][rec])
        ids = np.array(ds.variables['id_buoy'][:], dtype=int)
        lat, lon, y, x = (grab(n) for n in ('latitude', 'longitude', 'y_pos', 'x_pos'))
        tail = ([grab('mask')] if lmask else []) + ([grab('time_pos')] if lGetTimePos else [])
    geo = np.stack([lat, np.mod(lon, 360.)], axis=-1).astype(np.float64)     # f4 -> f8 like the reference
    yx = np.stack([y, x], axis=-1).astype(np.float64)
    return tuple([ztime, ids, geo, yx] + tail)


def SeedFileTimeInfo(fSeedNc, ltime2d=False, iverbose=0):
    """ncio.py:329-352 -> idate0, idateN (rounded to the hour), SeedName, SeedBatch, time_pos"""
    base = os.path.basename(fSeedNc)
    name = re.sub(r'\.(nc|npz)$', '', base.replace('SELECTION_', ''))
    batch = base.split('_')[2]
    chck4f(fSeedNc)
    if ltime2d:
        _, _, t2d = LoadNCtime(fSeedNc, ltime2d=True, iverbose=iverbose)
        first, last = np.min(t2d), np.max(t2d)
    else:
        n, t1d = LoadNCtime(fSeedNc, iverbose=iverbose)
        first, last, t2d = t1d[0], t1d[n - 1], []
    print('    * [SeedFileTimeInfo] => earliest and latest time position in the SEED file: %s - %s' % (e2c(first), e2c(last)))
    first, last = int(math.floor(first / 3600.) * 3600.), int(math.ceil(last / 3600.) * 3600.)
    print('    * [SeedFileTimeInfo]  ==> will actually use rounded to the hour! => %s - %s' % (e2c(first), e2c(last)))
    return first, last, name, batch, t2d


def ModelFileTimeInfo(fModelNc, iverbose=0):
    """ncio.py:356-384 -> Nt, time_counter (i4), idate0, idateN, CONF, EXP (both from the FILE NAME)"""
    with open_dataset(fModelNc) as ds:
        Nt = ds.dimensions['time_counter'].size
        _check_tunits(ds.variables['time_counter'], 'ModelFileTimeInfo')
        tmod = np.array(ds.variables['time_counter'][:], dtype='i4')
    print('    * [ModelFileTimeInfo] => %d records in input MODEL file!' % Nt)
    t0, tN = np.min(tmod), np.max(tmod)
    print('    * [ModelFileTimeInfo] => earliest and latest time position in the MODEL file: %s - %s' % (e2c(t0), e2c(tN)))
    parts = os.path.basename(fModelNc).split('_')
    conf, second = parts[0], parts[1].split('-')
    if len(second) == 1:                       # "<CONF>-<EXP>_1h_..." rather than "<CONF>_<x>-<EXP>_..."
        second = parts[0].split('-')
        conf = second[0]
    print('    * [ModelFileTimeInfo] => NEMO config and experiment =', conf, second[1], '\n')
    return Nt, tmod, t0, tN, conf, second[1]
