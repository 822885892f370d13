"""The five output files of ncio, pinned as they read back: every member of each .npz (name, dtype, shape, and the
value of 0-d members), and every dimension, variable (dtype, shape, fill value, units) and global attribute of each
netCDF4 file, written through the in-memory stand-in of test_cli."""
import contextlib
import io
import os
import sys
import types
import zipfile

import numpy as np
import pytest

TU = "seconds since 1970-01-01 00:00:00"
FILL = -9999.0
KINDS = ("cloud", "deform", "scaling", "grid", "dispersion")


def _write_all(d, ext):
    """Each of the five files from small fixed inputs, named <kind><ext> in d."""
    import sitrack_b200 as sit
    ids = np.array([10, 11, 12, 13])
    f = lambda k: os.path.join(d, k + ext)
    with contextlib.redirect_stdout(io.StringIO()):
        with sit.CloudBuoyWriter(f("cloud"), 3, ids, with_mask=True, with_time_pos=True, corigin="ORG") as w:
            for jt in range(3):
                w.write(jt, 100 + jt, np.ones(4), np.ones(4), np.ones(4), np.ones(4), mask=np.ones(4, "i1"),
                        time_pos=np.ones(4, "i4"))
        with sit.DeformationWriter(f("deform"), 2, np.array([[0, 1, 2], [2, 1, 3]]), ids, corigin="ORG") as w:
            for jw in range(2):
                w.write(jw, jw, jw + 1, {n: np.full(2, 0.5) for n in sit.DEFORM_NAMES})
        with sit.DeformationScalingWriter(f("scaling"), 2, [FILL, 10.0, 20.0], [0.01, 0.1, 1.0], corigin="ORG") as w:
            for jw in range(2):
                w.write(jw, jw, jw + 1, dict(n=np.array([4, 2, 0]), sum_L_eff=np.ones(3), sum_eps_tot=np.ones(3),
                                             sum_eps_tot2=np.ones(3), sum_eps_tot3=np.ones(3), hist_total=np.ones((3, 4)),
                                             hist_divergence=np.ones((3, 4)), hist_shear=np.ones((3, 4))))
        G = sit.EulerianGrid((0.0, -4.0), 2.0, (3, 4), 2, cover=0.25)
        with sit.DeformationGridWriter(f("grid"), 2, G, corigin="ORG") as w:
            for jw in range(2):
                w.write(jw, jw, jw + 1, [{n: np.ones(G.shapes[s]) for n in sit.BOX_NAMES} for s in range(2)])
        with sit.DispersionWriter(f("dispersion"), 2, [0.25, 0.5], [10.0, 100.0], [1.0, 2.0, 3.0], corigin="ORG") as w:
            for jw in range(2):
                w.write(jw, jw, jw + 1, dict(n=np.ones((2, 3)), sum_r0=np.ones((2, 3)), sum_dr=np.ones((2, 3)),
                                             sum_dr2=np.ones((2, 3)), sum_dD2=np.ones((2, 3)),
                                             hist_stretch=np.ones((2, 3, 4))))


def _units(**kw):
    """The 0-d `<name>_units` members of an .npz."""
    return {n + "_units": ("<U%d" % len(u), (), u) for n, u in kw.items()}


_FIELDS = dict(divergence="day-1", shear="day-1", vorticity="day-1", total="day-1", L_eff="km", y_ctr="km", x_ctr="km")
_GRID_SHAPES = {1: (3, 4), 2: (2, 2)}

NPZ = dict(
    cloud=dict(time=("<i4", (3,)), buoy=("<i4", (4,)), id_buoy=("<i8", (4,)), latitude=("<f4", (3, 4)),
               longitude=("<f4", (3, 4)), y_pos=("<f4", (3, 4)), x_pos=("<f4", (3, 4)), mask=("|i1", (3, 4)),
               time_pos=("<i4", (3, 4))),
    deform=dict(time_start=("<i4", (2,)), time_end=("<i4", (2,)), vertices=("<i4", (2, 3)), id_vertices=("<i8", (2, 3)),
                FillValue=("<f4", (), FILL),
                **{n: ("<f4", (2, 2)) for n in ("divergence", "shear", "vorticity", "area", "y_ctr", "x_ctr")},
                **_units(time_start=TU, time_end=TU, id_vertices="ID of buoy", divergence="day-1", shear="day-1",
                         vorticity="day-1", area="km2", y_ctr="km", x_ctr="km")),
    scaling=dict(time_start=("<i4", (2,)), time_end=("<i4", (2,)), scale_km=("<f8", (3,)), bin_edges=("<f8", (3,)),
                 n=("<i8", (2, 3)), FillValue=("<f8", (), FILL),
                 **{n: ("<f8", (2, 3)) for n in ("L_eff", "eps_tot", "eps_tot2", "eps_tot3")},
                 **{n: ("<i8", (2, 3, 4)) for n in ("hist_total", "hist_divergence", "hist_shear")},
                 **_units(time_start=TU, time_end=TU, scale_km="km", bin_edges="day-1", n="1", L_eff="km",
                          eps_tot="day-1", eps_tot2="day-2", eps_tot3="day-3", hist_total="1", hist_divergence="1",
                          hist_shear="1")),
    grid=dict(time_start=("<i4", (2,)), time_end=("<i4", (2,)), FillValue=("<f4", (), FILL), L_km=("<f8", (2,)),
              cover=("<f8", (), 0.25), origin=("<f8", (2,)),
              y1=("<f8", (3,)), x1=("<f8", (4,)), y2=("<f8", (2,)), x2=("<f8", (2,)),
              **{"%s_%d" % (n, s): ("<f4", (2,) + sh) for n in _FIELDS for s, sh in _GRID_SHAPES.items()},
              **_units(time_start=TU, time_end=TU, y1="km", x1="km", y2="km", x2="km",
                       **{"%s_%d" % (n, s): u for n, u in _FIELDS.items() for s in _GRID_SHAPES})),
    dispersion=dict(time_start=("<i4", (2,)), time_end=("<i4", (2,)), lag_days=("<f8", (2,)), r_edges=("<f8", (2,)),
                    bin_edges=("<f8", (3,)), n=("<i8", (2, 2, 3)), hist_stretch=("<i8", (2, 2, 3, 4)),
                    **{n: ("<f8", (2, 2, 3)) for n in ("sum_r0", "sum_dr", "sum_dr2", "sum_dD2")},
                    **_units(time_start=TU, time_end=TU, lag_days="day", r_edges="km", bin_edges="day-1", n="1",
                             hist_stretch="1", sum_r0="km", sum_dr="km", sum_dr2="km2", sum_dD2="km2")),
)

# netCDF4: dims, variables {name: (dtype, shape, fill value, units)}, global attributes other than Author
NC = dict(
    cloud=({"time": None, "buoy": 4},
           dict(time=("<i4", (3,), None, TU), buoy=("<i4", (4,), None, None), id_buoy=("<i8", (4,), None, "ID of buoy"),
                latitude=("<f4", (3, 4), FILL, "degrees north"), longitude=("<f4", (3, 4), FILL, "degrees south"),
                y_pos=("<f4", (3, 4), FILL, "km"), x_pos=("<f4", (3, 4), FILL, "km"), mask=("|i1", (3, 4), None, None),
                time_pos=("<i4", (3, 4), FILL, TU)),
           dict(Origin="ORG", About="Lagrangian sea-ice drift")),
    deform=({"time": None, "triangle": 2, "vertex": 3},
            dict(time_start=("<i4", (2,), None, TU), time_end=("<i4", (2,), None, TU),
                 vertices=("<i4", (2, 3), None, None), id_vertices=("<i8", (2, 3), None, "ID of buoy"),
                 divergence=("<f4", (2, 2), FILL, "day-1"), shear=("<f4", (2, 2), FILL, "day-1"),
                 vorticity=("<f4", (2, 2), FILL, "day-1"), area=("<f4", (2, 2), FILL, "km2"),
                 y_ctr=("<f4", (2, 2), FILL, "km"), x_ctr=("<f4", (2, 2), FILL, "km")),
            dict(Origin="ORG", About="Sea-ice deformation rates of buoy triangles")),
    scaling=({"time": None, "scale": 3, "bin": 4, "bin_edge": 3},
             dict(time_start=("<i4", (2,), None, TU), time_end=("<i4", (2,), None, TU),
                  scale_km=("<f8", (3,), None, "km"), bin_edges=("<f8", (3,), None, "day-1"),
                  n=("<i8", (2, 3), None, "1"), L_eff=("<f8", (2, 3), FILL, "km"), eps_tot=("<f8", (2, 3), FILL, "day-1"),
                  eps_tot2=("<f8", (2, 3), FILL, "day-2"), eps_tot3=("<f8", (2, 3), FILL, "day-3"),
                  **{n: ("<i8", (2, 3, 4), None, "1") for n in ("hist_total", "hist_divergence", "hist_shear")}),
             dict(Origin="ORG", About="Per-scale statistics of sea-ice deformation coarse-grained over material boxes "
                                      "of buoy triangles")),
    grid=({"time": None, "y1": 3, "x1": 4, "y2": 2, "x2": 2},
          dict(time_start=("<i4", (2,), None, TU), time_end=("<i4", (2,), None, TU),
               y1=("<f8", (3,), None, "km"), x1=("<f8", (4,), None, "km"), y2=("<f8", (2,), None, "km"),
               x2=("<f8", (2,), None, "km"),
               **{"%s_%d" % (n, s): ("<f4", (2,) + sh, FILL, u) for n, u in _FIELDS.items()
                  for s, sh in _GRID_SHAPES.items()}),
          dict(Origin="ORG", About="Sea-ice deformation of buoy triangles coarse-grained over the cells of a fixed grid",
               L_km=np.array([2.0, 4.0]), cover=0.25, origin=np.array([0.0, -4.0]))),
    dispersion=({"time": None, "lag": 2, "class": 3, "bin": 4, "class_edge": 2, "bin_edge": 3},
                dict(time_start=("<i4", (2,), None, TU), time_end=("<i4", (2,), None, TU),
                     lag_days=("<f8", (2,), None, "day"), r_edges=("<f8", (2,), None, "km"),
                     bin_edges=("<f8", (3,), None, "day-1"), n=("<i8", (2, 2, 3), None, "1"),
                     hist_stretch=("<i8", (2, 2, 3, 4), None, "1"), sum_r0=("<f8", (2, 2, 3), None, "km"),
                     sum_dr=("<f8", (2, 2, 3), None, "km"), sum_dr2=("<f8", (2, 2, 3), None, "km2"),
                     sum_dD2=("<f8", (2, 2, 3), None, "km2")),
                dict(Origin="ORG", About="Two-particle dispersion of buoy pairs over time lags, by initial separation")),
)


@pytest.fixture(scope="module")
def npz_dir(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("npz"))
    _write_all(d, ".npz")
    return d


@pytest.mark.parametrize("kind", KINDS)
def test_npz_members(npz_dir, kind):
    assert sorted(os.listdir(npz_dir)) == sorted(k + ".npz" for k in KINDS)       # no scratch directory left behind
    z = np.load(os.path.join(npz_dir, kind + ".npz"))
    got = {n: (z[n].dtype.str, z[n].shape) + ((z[n].item(),) if z[n].ndim == 0 else ()) for n in z.files}
    assert got == NPZ[kind]
    with zipfile.ZipFile(os.path.join(npz_dir, kind + ".npz")) as f:
        assert {i.compress_type for i in f.infolist()} == {zipfile.ZIP_DEFLATED}


@pytest.fixture(scope="module")
def nc_files(tmp_path_factory):
    from test_cli import _FakeNC
    fake = types.ModuleType("netCDF4"); fake.Dataset = _FakeNC.Dataset
    mp = pytest.MonkeyPatch()
    mp.setitem(sys.modules, "netCDF4", fake)
    d = str(tmp_path_factory.mktemp("nc"))
    try:
        _write_all(d, ".nc")
    finally:
        mp.undo()
    assert not os.listdir(d)
    return {k: _FakeNC.files[os.path.join(d, k + ".nc")] for k in KINDS}


@pytest.mark.parametrize("kind", KINDS)
def test_netcdf_dims_variables_and_attributes(nc_files, kind):
    ds = nc_files[kind]
    dims, variables, attrs = NC[kind]
    assert ds._dims == dims
    got = {n: (v.dtype.str, v.a.shape, v.fill, getattr(v, "units", None)) for n, v in ds.variables.items()}
    assert got == variables
    attrs = dict(attrs, Author="Generated with `%s` of `sitrack` (L. Brodeau, 2023)" % os.path.basename(sys.argv[0]))
    assert sorted(ds.attrs) == sorted(attrs)
    for k, v in attrs.items():
        assert type(ds.attrs[k]) is type(v) and np.array_equal(ds.attrs[k], v), k
