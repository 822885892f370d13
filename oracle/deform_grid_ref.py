"""Reference coarse-graining of buoy-triangle deformation over the cells of a fixed Eulerian grid, rebuilt every
window (test infrastructure only; the product never imports it).

Method -- the contract of csrc/st_deform_grid.cu, sitrack_b200.EulerianGrid and DESIGN.md section 12; everything
not said here is deform_scale_ref's (section 11):

Grid.      origin (oy, ox) km, L0 km, shape (nj, ni) level-1 cells, `levels` levels.  Level-1 cell (bj, bi) covers
           [oy + bj L0, oy + (bj+1) L0) x [ox + bi L0, ox + (bi+1) L0); level s (1-based) has side L0 2^(s-1), key
           (bj, bi) >> (s-1) and nj_s = ((nj-1) >> (s-1)) + 1 rows, ni_s likewise.  Fixed for the whole run.
Binned.    Rebuilt every window [k0, k1]: a triangle valid by k_deform's rule whose mid-time centroid
           Yc = ((Y0+Y1)+Y2)/3 (Y_i = 0.5 (y0_i + y1_i)), Xc likewise, lies in the grid: q = floor((Yc - oy) / L0),
           0 <= q < nj compared in f8 (NaN and inf are never binned; a centroid on a cell edge belongs to the upper
           cell, one on oy + nj L0 is outside), likewise in x.
Order.     Binned triangles sorted stably by the Morton code of their level-1 key (i bits even, j bits odd), ties in
           the caller's triangle order; each level's boxes are the runs of that order.  Then deform_scale_ref's sums,
           box outputs, cover rule and statistics apply unchanged; scale 0 counts the binned triangles only, with their
           own rates.
Fields.    Per level, seven (nj_s, ni_s) f4 planes of BOX_NAMES, FillValue where a cell has no binned triangle or its
           box does not count.
"""
import numpy as np

from . import deform_ref as R
from . import deform_scale_ref as S
from .deform_scale_ref import BOX_NAMES, DEFAULT_EDGES, FillValue


def grid_shape(shape, s):
    """(nj_s, ni_s) of level s (0-based)."""
    return tuple(((int(n) - 1) >> s) + 1 for n in shape)


def eulerian_binning(yx0, yx1, mask0, mask1, tri, origin, L0, shape):
    """-> (binned (nT,) bool, key (nT,2) i8 [bj, bi], meaningful where binned)."""
    yx0, yx1 = np.asarray(yx0, np.float64), np.asarray(yx1, np.float64)
    tri = np.asarray(tri, np.int64).reshape(-1, 3)
    _, valid = R.rates_f8(yx0, yx1, mask0, mask1, tri, 1.0)
    with np.errstate(all="ignore"):
        q = []
        for k in (0, 1):
            P = 0.5 * (yx0[tri, k] + yx1[tri, k])
            c = ((P[:, 0] + P[:, 1]) + P[:, 2]) / 3.0
            q.append(np.floor((c - np.float64(origin[k])) / np.float64(L0)))
        q = np.stack(q, 1)
        inside = (q[:, 0] >= 0) & (q[:, 0] < shape[0]) & (q[:, 1] >= 0) & (q[:, 1] < shape[1])
    binned = valid & inside
    key = np.where(binned[:, None], q, 0).astype(np.int64)
    return binned, key


def eulerian_hierarchy(yx0, yx1, mask0, mask1, tri, origin, L0, shape, levels):
    """deform_scale_ref.hierarchy()'s dict over the cells of a fixed grid for the window (yx0, mask0) -> (yx1, mask1):
    `order` holds the binned triangles only; also `binned` (nT,) bool."""
    binned, key = eulerian_binning(yx0, yx1, mask0, mask1, tri, origin, L0, shape)
    idx = np.flatnonzero(binned)
    code = (S._spread(key[idx, 0]) << np.uint64(1)) | S._spread(key[idx, 1])
    o = np.argsort(code, kind="stable")
    order, cs, ks = idx[o], code[o], key[idx[o]]
    out = []
    prev = None
    for s in range(levels):
        cl = cs >> np.uint64(2 * s)
        st = np.flatnonzero(np.r_[cs.size > 0, cl[1:] != cl[:-1]]) if cs.size else np.zeros(0, np.int64)
        lv = dict(key=ks[st] >> s, off=np.r_[st, cs.size].astype(np.int64), child=None)
        if prev is not None:
            lv["child"] = np.r_[np.searchsorted(prev, st), prev.size].astype(np.int64)
        out.append(lv)
        prev = st
    return dict(order=order, origin=np.asarray(origin, np.float64), levels=out, binned=binned)


def coarse_grain(yx0, yx1, mask0, mask1, tri, dt, E, cover=0.5, edges=DEFAULT_EDGES, L0=None):
    """deform_scale_ref.coarse_grain over an eulerian_hierarchy E, with scale 0 counting E's binned triangles only.
    -> (boxes, stats) in deform_scale_ref's layout."""
    edges = np.asarray(edges, np.float64)
    T, r, valid = S.triangle_terms(yx0, yx1, mask0, mask1, tri, dt)
    valid = valid & E["binned"]
    Ts = T[E["order"]]
    with np.errstate(all="ignore"):
        o0 = S.rates_of(r["ux"], r["uy"], r["vx"], r["vy"])
        o0["L_eff"] = np.sqrt(r["area"])
    st = [S.cell_stats(o0, valid, edges)]
    boxes = []
    Sb = None
    for s, lv in enumerate(E["levels"]):
        Sb = S.level1_sums(Ts, lv["off"]) if s == 0 else S.parent_sums(Sb, lv["child"])
        Ls = L0 * 2.0 ** s
        o, ok = S.box_outputs(Sb, cover * Ls * Ls)
        st.append(S.cell_stats(o, ok, edges))
        b = dict(key=lv["key"], valid=ok, S=Sb)
        with np.errstate(all="ignore"):
            b.update({k: np.where(ok, o[k], FillValue).astype(np.float32) for k in BOX_NAMES})
        boxes.append(b)
    return boxes, dict(n=np.array([x["n"] for x in st], np.int64), sums=np.stack([x["sums"] for x in st]),
                       hist=np.stack([x["hist"] for x in st]))


def grid_fields(boxes, shape):
    """coarse_grain's boxes -> per level dict of (nj_s, ni_s) f4 BOX_NAMES planes, FillValue where no box or the box
    does not count."""
    out = []
    for s, b in enumerate(boxes):
        nj, ni = grid_shape(shape, s)
        d = {}
        for k in BOX_NAMES:
            f = np.full((nj, ni), FillValue, np.float32)
            f[b["key"][:, 0], b["key"][:, 1]] = b[k]
            d[k] = f
        out.append(d)
    return out
