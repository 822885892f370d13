"""Buoy-triangle deformation coarse-grained over the cells of a fixed Eulerian grid, rebuilt every window: dense
per-level fields and per-scale statistics (the gridded products of RGPS and of model-observation comparisons, and
scaling statistics over boxes whose side stays what its label says).

Definitions (DESIGN.md section 12).  EulerianGrid fixes, for the whole run, square cells of side L0 on the
NorthPolarStereo plane of the rows: level-1 cell (bj, bi) covers [oy + bj L0, oy + (bj+1) L0) x [ox + bi L0,
ox + (bi+1) L0); level s has side L0 2^(s-1) and key (bj, bi) >> (s-1).  In every window a triangle is binned when it is
valid (section 10) and its mid-time centroid lies in the grid, in the level-1 cell holding it (a centroid on an edge
belongs to the upper cell).  From there the sums, box outputs, cover rule and statistics are those of section 11
(sitrack_b200.deform_scales) over the cells, with scale 0 the binned triangles.  Membership, sort and segmentation run
on the device (csrc/st_deform_grid.cu); only the fields and statistics reach the host.  No CPU fallback.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_c, check
from .deform import _upload_rows, check_mesh
from .deform_scales import BOX_NAMES, _Levels, stats_dict

__all__ = ["EulerianGrid", "GriddedRates", "MAX_GRID_SIDE"]

MAX_GRID_SIDE = 2 ** 20


class EulerianGrid(_Levels):
    """A fixed grid of shape = (nj, ni) level-1 cells (1..2^20 each) of side L0_km from origin_yx = (oy, ox) km, with
    `levels` (1..20) levels of sides L0_km * 2^s.  A cell counts when the area of its binned triangles is at least
    cover * L_s^2.  `bins`: histogram edges [1/day] (f8, strictly increasing; default DEFAULT_BIN_EDGES).

    Attributes: origin (2,) f8, L0_km, shape (nj, ni), levels, cover, L_km (levels,), min_area (levels,), scale_km
    (levels+1,) with FillValue for the triangle scale, shapes [levels] (nj_s, ni_s) with nj_s = ((nj-1) >> s) + 1,
    bin_edges."""

    def __init__(self, origin_yx, L0_km, shape, levels, cover=0.5, bins=None):
        o = np.asarray(origin_yx, np.float64).ravel()
        if o.shape != (2,) or not np.isfinite(o).all():
            raise ValueError("EulerianGrid: origin_yx must be two finite numbers (oy, ox) km, got %r" % (origin_yx,))
        sh = tuple(shape) if np.ndim(shape) == 1 else ()
        if len(sh) != 2 or any(int(n) != n or not 1 <= n <= MAX_GRID_SIDE for n in sh):
            raise ValueError("EulerianGrid: shape must be two integers (nj, ni) in 1..%d, got %r" % (MAX_GRID_SIDE, shape))
        super().__init__("EulerianGrid", L0_km, levels, cover, bins)
        self.origin, self.shape = o, (int(sh[0]), int(sh[1]))
        self.shapes = [(((self.shape[0] - 1) >> s) + 1, ((self.shape[1] - 1) >> s) + 1) for s in range(self.levels)]

    def centres(self, s):
        """(y_km (nj_s,), x_km (ni_s,)) cell-centre coordinates of level s (0-based)."""
        nj, ni = self.shapes[s]
        L = self.L_km[s]
        return self.origin[0] + (np.arange(nj) + 0.5) * L, self.origin[1] + (np.arange(ni) + 0.5) * L

    def field_size(self):
        """f4 words of the fields of one window: sum_s 7 nj_s ni_s."""
        return sum(7 * nj * ni for nj, ni in self.shapes)


class _GridPlan:
    """The device buffers of a grid pass over a mesh `slots` ((nT,3) buoy indices as stored on the device, in the
    caller's triangle order): mesh, edges and scratch."""

    def __init__(self, torch, dev, G, slots):
        self.torch, self.G, self.L = torch, G, _lib.lib()
        slots = np.asarray(slots).reshape(-1, 3)
        if slots.shape[0] == 0:
            raise ValueError("the mesh has no triangle")
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        self.tri_t = t(slots, np.int32)
        self.edges_t = t(G.bin_edges, np.float64)
        self.min_area = as_c(G.min_area, np.float64)
        nb = C.c_int64()
        with torch.cuda.device(dev):
            check(self.L.st_deform_grid_scratch_bytes(int(self.tri_t.shape[0]), G.levels, G.shape[0], G.shape[1],
                                                      G.bin_edges.size, C.byref(nb)), None)
        self.scratch_bytes = nb.value
        self.scratch = torch.empty((nb.value + 7) // 8, dtype=torch.float64, device=dev)
        self.S = G.levels + 1

    def outputs(self, pin=False):
        """(moments (S,4) f8, hist (S,3,len(edges)+1) i8, fields (sum_s 7 nj_s ni_s,) f4, nbox (levels,) i8) on the
        device, or pinned on the host."""
        kw = dict(pin_memory=True) if pin else dict(device=self.scratch.device)
        T = self.torch
        return (T.empty((self.S, 4), dtype=T.float64, **kw), T.empty((self.S, 3, self.G.bin_edges.size + 1), dtype=T.int64, **kw),
                T.empty((self.G.field_size(),), dtype=T.float32, **kw), T.empty((self.G.levels,), dtype=T.int64, **kw))

    def launch(self, ctx, yx0_t, m0_t, yx1_t, m1_t, dt_days, mom_t, hist_t, fields_t, nbox_t, stream):
        """st_deform_grid_dev (async on `stream`)."""
        G = self.G
        check(self.L.st_deform_grid_dev(
            ctx, int(self.tri_t.shape[0]), self.tri_t.data_ptr(), yx0_t.data_ptr(), m0_t.data_ptr(), yx1_t.data_ptr(),
            m1_t.data_ptr(), float(dt_days), G.levels, G.shape[0], G.shape[1], float(G.origin[0]), float(G.origin[1]),
            G.L0_km, self.min_area.ctypes.data, G.bin_edges.size, self.edges_t.data_ptr(), self.scratch.data_ptr(),
            self.scratch_bytes, mom_t.data_ptr(), hist_t.data_ptr(), fields_t.data_ptr(), nbox_t.data_ptr(),
            C.c_void_p(stream.cuda_stream)), ctx)

    def window(self, ctx, origins, yx1_t, m1_t, dt_days, outs, stream):
        """TrackEngine.track's pass over one window: origins = [(yx0_t, m0_t, 1)]."""
        (yx0_t, m0_t, _), = origins
        self.launch(ctx, yx0_t, m0_t, yx1_t, m1_t, dt_days, *outs, stream)

    def results(self, outs):
        """(fields, stats) of the window from its pinned outputs."""
        mom, hist, fields, _ = (o.numpy() for o in outs)
        return split_fields(self.G, fields), stats_dict(self.G, mom, hist)


def split_fields(G, flat):
    """The flat f4 field buffer of one window -> per level dict of (nj_s, ni_s) f4 BOX_NAMES planes (copies) and the
    cell-centre coordinates y_km, x_km."""
    flat = np.asarray(flat)
    out, o = [], 0
    for s, (nj, ni) in enumerate(G.shapes):
        d = {}
        for n in BOX_NAMES:
            d[n] = flat[o:o + nj * ni].reshape(nj, ni).copy()
            o += nj * ni
        d["y_km"], d["x_km"] = G.centres(s)
        out.append(d)
    return out


def GriddedRates(pYX0, pYX1, mask0, mask1, tri, G, dt_days, device=None):
    """Deformation of the triangles `tri` (nT,3) coarse-grained over the cells of the EulerianGrid G between positions
    pYX0 and pYX1 ((nP,2) [y,x] km) with masks mask0, mask1 (nP,), dt_days apart.  Host arrays in and out; computed on
    the GPU.

    -> (fields, stats).  fields: per level a dict of (nj_s, ni_s) f4 BOX_NAMES planes (divergence, shear, vorticity,
    total = eps_tot [1/day], L_eff [km], y_ctr, x_ctr [km, mid-time centroid]; FillValue where a cell has no binned
    triangle or does not count) and y_km (nj_s,), x_km (ni_s,) cell centres.  stats: as CoarseGrainedRates' (scale 0 =
    the binned triangles)."""
    if not isinstance(G, EulerianGrid):
        raise TypeError("G must be an EulerianGrid")
    torch, dev, nP, rows = _upload_rows(pYX0, pYX1, mask0, mask1, dt_days, device)
    with torch.cuda.device(dev):
        plan = _GridPlan(torch, dev, G, check_mesh(tri, nP))
        mom, hist, fields, nbox = plan.outputs()
        plan.launch(None, *rows, dt_days, mom, hist, fields, nbox, torch.cuda.current_stream(dev))
        f, mom, hist = fields.cpu().numpy(), mom.cpu().numpy(), hist.cpu().numpy()
    return split_fields(G, f), stats_dict(G, mom, hist)
