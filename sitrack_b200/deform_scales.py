"""Buoy-triangle deformation coarse-grained over spatial scales, and per-scale statistics of it (the spatial scaling
of sea-ice deformation: <eps_tot^q> against L, Marsan et al. 2004; Rampal et al. 2008; Bouchat et al. 2022).

Definitions (DESIGN.md section 11).  BoxHierarchy builds, once per run on the host, square material boxes over the
mesh: a triangle belongs to the level-1 box (side L0) holding its build-time centroid, level s+1 boxes (side 2 L_s)
are unions of four level-s boxes, and boxes keep their triangles as the ice moves.  Between two rows, a box's velocity
gradient is the sum over its valid triangles of their edge line integrals over the sum of their areas (Green's
theorem: interior edges cancel), so it is the RGPS rate of the union.  A box counts when its area is at least
cover * L_s^2.  Per scale (0 = the triangles themselves) the statistics are n, sums of L_eff = sqrt(area), eps_tot,
eps_tot^2, eps_tot^3 (eps_tot = sqrt(div^2 + shear^2)) and histograms of eps_tot, |div| and shear on fixed edges.
The sums are computed on the device (csrc/st_deform_scale.cu) in a fixed order: bit-identical run to run and
whatever order the buoys are stored in.  No CPU fallback.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_c, check
from .deform import _upload_rows, check_mesh

__all__ = ["BoxHierarchy", "CoarseGrainedRates", "BOX_NAMES", "DEFAULT_BIN_EDGES", "MAX_LEVELS"]

FillValue = -9999.0
BOX_NAMES = ("divergence", "shear", "vorticity", "total", "L_eff", "y_ctr", "x_ctr")
DEFAULT_BIN_EDGES = np.array([10.0 ** (k / 10.0) for k in range(-50, 11)])   # 1e-5 ... 1e1 day-1, 10 bins per decade
MAX_LEVELS = 20
MAX_EDGES = 4096


def check_edges(edges, default, limit, what):
    """(n,) f8 histogram or class edges (`default` when None): 1..limit finite, strictly increasing values."""
    e = as_c(default if edges is None else edges, np.float64).ravel()
    if not 1 <= e.size <= limit or not np.isfinite(e).all() or (np.diff(e) <= 0).any():
        raise ValueError("%s must be 1..%d finite, strictly increasing edges" % (what, limit))
    return e


class _Levels:
    """What BoxHierarchy and EulerianGrid share, checked (ValueError prefixed by `who`): `levels` (1..MAX_LEVELS)
    levels of square cells of sides L_km = L0_km * 2^s, a cell counting when its area is at least min_area =
    cover * L_s^2, scale_km = (FillValue for the triangles, L_km...) and histogram edges bin_edges (`bins`, f8,
    strictly increasing; default DEFAULT_BIN_EDGES)."""

    def __init__(self, who, L0_km, levels, cover, bins):
        if not (np.isfinite(L0_km) and L0_km > 0):
            raise ValueError("%s: L0_km must be finite and positive, got %r" % (who, L0_km))
        if int(levels) != levels or not 1 <= levels <= MAX_LEVELS:
            raise ValueError("%s: levels must be an integer in 1..%d, got %r" % (who, MAX_LEVELS, levels))
        if not (np.isfinite(cover) and cover > 0):
            raise ValueError("%s: cover must be positive, got %r" % (who, cover))
        self.bin_edges = check_edges(bins, DEFAULT_BIN_EDGES, MAX_EDGES, who + ": bins")
        self.levels, self.L0_km, self.cover = int(levels), float(L0_km), float(cover)
        self.L_km = self.L0_km * 2.0 ** np.arange(self.levels)
        self.min_area = np.float64(self.cover) * self.L_km * self.L_km
        self.scale_km = np.r_[FillValue, self.L_km]


def _spread(v):
    """Bits of v (< 2^32) into the even positions of a uint64."""
    v = v.astype(np.uint64)
    for s, m in ((16, 0x0000FFFF0000FFFF), (8, 0x00FF00FF00FF00FF), (4, 0x0F0F0F0F0F0F0F0F),
                 (2, 0x3333333333333333), (1, 0x5555555555555555)):
        v = (v | (v << np.uint64(s))) & np.uint64(m)
    return v


class BoxHierarchy(_Levels):
    """Square material boxes over the triangles `tri` (nT,3) of buoys at positions pYX (nP,2) [y,x] km (the
    positions the mesh was built from), `levels` levels of sides L0_km * 2^s.  Host only (numpy), once per run.

    A triangle belongs to the level-1 box holding its centroid ((y0+y1)+y2)/3, ((x0+x1)+x2)/3; the grid origin is
    floor(min centroid / L0) * L0; keys (bj, bi) = floor((c - origin) / L0), and a level-(s+1) key is its children's
    key >> 1.  Triangles are sorted stably by the Morton code of their level-1 key, so every box is a contiguous
    range of `order`.  A box counts when its area >= cover * L_s^2.  `bins`: histogram edges [1/day] (f8, strictly
    increasing; default DEFAULT_BIN_EDGES).

    Attributes: nP, tri (the mesh, caller's order), order (nT,) i8, origin (2,), L_km (levels,), min_area (levels,),
    scale_km (levels+1,) with FillValue for the triangle scale, keys [levels] (nbox,2) i8, tri_off (nbox_1+1,) i8
    ranges of `order`, child_off [levels] (nbox+1,) i8 ranges of the previous level's boxes (None at level 1),
    box_tri_off [levels] ranges of `order` of every level, nbox (levels,) i8, bin_edges."""

    def __init__(self, pYX, tri, L0_km, levels, cover=0.5, bins=None):
        yx = as_c(pYX, np.float64).reshape(-1, 2)
        self.nP = yx.shape[0]
        super().__init__("BoxHierarchy", L0_km, levels, cover, bins)
        self.tri = check_mesh(tri, self.nP).copy()
        nT = self.tri.shape[0]
        if nT == 0:
            raise ValueError("BoxHierarchy: the mesh has no triangle")
        if nT >= 2 ** 31:
            raise ValueError("BoxHierarchy: at most 2^31 - 1 triangles")
        t = self.tri
        c = np.stack([((yx[t[:, 0], k] + yx[t[:, 1], k]) + yx[t[:, 2], k]) / 3.0 for k in (0, 1)], 1)
        if not np.isfinite(c).all():
            raise ValueError("BoxHierarchy: the mesh's positions must be finite")
        self.origin = np.floor(c.min(0) / L0_km) * L0_km
        key = np.floor((c - self.origin) / L0_km)
        if key.max() >= 2 ** 31:
            raise ValueError("BoxHierarchy: L0_km too small for the extent of the mesh (more than 2^31 boxes a side)")
        key = key.astype(np.int64)
        code = (_spread(key[:, 0]) << np.uint64(1)) | _spread(key[:, 1])
        self.order = np.argsort(code, kind="stable")
        cs = code[self.order]
        st = np.flatnonzero(np.r_[True, cs[1:] != cs[:-1]])
        k1 = key[self.order[st]]
        u = cs[st]
        self.tri_off = np.r_[st, nT].astype(np.int64)
        self.keys, self.child_off, self.box_tri_off = [k1], [None], [self.tri_off]
        for s in range(1, self.levels):                           # parents from the previous level's box codes
            u = u >> np.uint64(2)
            b = np.flatnonzero(np.r_[True, u[1:] != u[:-1]])
            u = u[b]
            self.child_off.append(np.r_[b, self.keys[-1].shape[0]].astype(np.int64))
            self.box_tri_off.append(np.r_[self.box_tri_off[-1][b], nT].astype(np.int64))
            self.keys.append(self.keys[-1][b] >> 1)
        self.nbox = np.array([k.shape[0] for k in self.keys], np.int64)

    def matches(self, tri, nP):
        """True when (tri, nP) is the mesh this hierarchy was built on."""
        return nP == self.nP and np.array_equal(np.asarray(tri).reshape(-1, 3), self.tri)


class _DevicePlan:
    """A hierarchy's device buffers for one buoy storage order: the mesh in hierarchy order with vertices `slots`
    ((nT,3) buoy indices as stored on the device, caller's triangle order), box ranges, edges and scratch."""

    def __init__(self, torch, dev, H, slots):
        self.torch, self.H, self.L = torch, H, _lib.lib()
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        self.tri_t = t(np.asarray(slots)[H.order], np.int32)
        self.tri_off_t = t(H.tri_off, np.int64)
        self.child_t = t(np.concatenate(H.child_off[1:]) if H.levels > 1 else np.zeros(1), np.int64)
        self.edges_t = t(H.bin_edges, np.float64)
        self.nbox, self.min_area = as_c(H.nbox, np.int64), as_c(H.min_area, np.float64)
        nb = C.c_int64()
        check(self.L.st_deform_scales_scratch_bytes(int(self.tri_t.shape[0]), H.levels, self.nbox.ctypes.data,
                                                    self.min_area.ctypes.data, H.bin_edges.size, C.byref(nb)), None)
        self.scratch_bytes = nb.value
        self.scratch = torch.empty((nb.value + 7) // 8, dtype=torch.float64, device=dev)
        self.S = H.levels + 1

    def outputs(self, pin=False):
        """(moments (S,4) f8, hist (S,3,len(edges)+1) i8) on the device, or pinned on the host."""
        kw = dict(pin_memory=True) if pin else dict(device=self.scratch.device)
        return (self.torch.empty((self.S, 4), dtype=self.torch.float64, **kw),
                self.torch.empty((self.S, 3, self.H.bin_edges.size + 1), dtype=self.torch.int64, **kw))

    def launch(self, ctx, yx0_t, m0_t, yx1_t, m1_t, dt_days, mom_t, hist_t, boxes_t, stream):
        """st_deform_scales_dev (async on `stream`)."""
        H = self.H
        check(self.L.st_deform_scales_dev(
            ctx, int(self.tri_t.shape[0]), self.tri_t.data_ptr(), yx0_t.data_ptr(), m0_t.data_ptr(), yx1_t.data_ptr(),
            m1_t.data_ptr(), float(dt_days), H.levels, self.nbox.ctypes.data, self.min_area.ctypes.data,
            self.tri_off_t.data_ptr(), self.child_t.data_ptr(), H.bin_edges.size, self.edges_t.data_ptr(),
            self.scratch.data_ptr(), self.scratch_bytes, mom_t.data_ptr(), hist_t.data_ptr(),
            None if boxes_t is None else boxes_t.data_ptr(), C.c_void_p(stream.cuda_stream)), ctx)

    def window(self, ctx, origins, yx1_t, m1_t, dt_days, outs, stream):
        """TrackEngine.track's pass over one window: origins = [(yx0_t, m0_t, 1)]."""
        (yx0_t, m0_t, _), = origins
        self.launch(ctx, yx0_t, m0_t, yx1_t, m1_t, dt_days, *outs, None, stream)

    def results(self, outs):
        """(the statistics of the window,) from its pinned outputs."""
        return (stats_dict(self.H, *(o.numpy() for o in outs)),)


def stats_dict(H, mom, hist):
    """Host moments (S,4) and hist (S,3,nb+2) -> the statistics of one window (see CoarseGrainedRates)."""
    mom, hist = np.array(mom, np.float64), np.array(hist, np.int64)
    return dict(scale_km=H.scale_km.copy(), n=hist[:, 0].sum(1), sum_L_eff=mom[:, 0], sum_eps_tot=mom[:, 1],
                sum_eps_tot2=mom[:, 2], sum_eps_tot3=mom[:, 3], hist_total=hist[:, 0], hist_divergence=hist[:, 1],
                hist_shear=hist[:, 2], bin_edges=H.bin_edges.copy())


def CoarseGrainedRates(pYX0, pYX1, mask0, mask1, H, dt_days, device=None):
    """Deformation of the boxes of the BoxHierarchy H between positions pYX0 and pYX1 ((nP,2) [y,x] km) with masks
    mask0, mask1 (nP,), dt_days apart, and its per-scale statistics.  Host arrays in and out; computed on the GPU.

    -> (boxes, stats).  boxes: per level a dict of (nbox,) f4 BOX_NAMES (divergence, shear, vorticity, total =
    eps_tot [1/day], L_eff [km], y_ctr, x_ctr [km, mid-time centroid]; FillValue where the box does not count) and
    `key` (nbox,2) [bj, bi].  stats: scale_km (S,) (FillValue for the triangles), n (S,) i8 cells that count,
    sum_L_eff, sum_eps_tot, sum_eps_tot2, sum_eps_tot3 (S,) f8, hist_total, hist_divergence (of |div|), hist_shear
    (S, nb+2) i8 with underflow and overflow, bin_edges (nb+1,)."""
    if not isinstance(H, BoxHierarchy):
        raise TypeError("H must be a BoxHierarchy")
    torch, dev, _, rows = _upload_rows(pYX0, pYX1, mask0, mask1, dt_days, device, H.nP)
    with torch.cuda.device(dev):
        plan = _DevicePlan(torch, dev, H, H.tri)
        mom, hist = plan.outputs()
        boxes_t = torch.empty((7, int(H.nbox.sum())), dtype=torch.float32, device=dev)
        plan.launch(None, *rows, dt_days, mom, hist, boxes_t, torch.cuda.current_stream(dev))
        o, mom, hist = boxes_t.cpu().numpy(), mom.cpu().numpy(), hist.cpu().numpy()
    b0 = np.r_[0, np.cumsum(H.nbox)]
    boxes = []
    for s in range(H.levels):
        d = {n: as_c(o[j, b0[s]:b0[s + 1]], np.float32) for j, n in enumerate(BOX_NAMES)}
        d["key"] = H.keys[s].copy()
        boxes.append(d)
    return boxes, stats_dict(H, mom, hist)
