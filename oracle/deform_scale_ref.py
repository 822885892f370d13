"""Reference coarse-graining of buoy-triangle deformation over material boxes, and its per-scale statistics (test
infrastructure only; the product never imports it).

Method -- the contract of csrc/st_deform_scale.cu, sitrack_b200.BoxHierarchy and DESIGN.md section 11:

Boxes.     Built once from the mesh tri (nT,3) and the positions it was built from, pYX (nP,2) [y,x] km.  A triangle
           belongs to the level-1 box holding its build-time centroid ((y0+y1)+y2)/3, ((x0+x1)+x2)/3.  Level-1 boxes
           have side L0; the grid origin is floor(min centroid / L0) * L0 in y and in x; the key is
           (bj, bi) = floor((c - origin) / L0).  Level s+1 has side 2 L_s and key = the children's key >> 1.  Scale
           index 0 is the triangles themselves.  Boxes are material: membership is fixed at build time.
           Triangles are sorted (stably) by the Morton code of their level-1 key (i bits in the even positions, j
           bits in the odd ones), so every box of every level is a contiguous range of that order.
Terms.     Per triangle, f8, with X, Y, U, V, twice_area and edge_sum of deform_ref:
             a2 = 2A, Nux = edge_sum(U,Y), Nuy = -edge_sum(U,X), Nvx = edge_sum(V,Y), Nvy = -edge_sum(V,X),
             NY = a2 * Yc, NX = a2 * Xc    (Yc = ((Y0+Y1)+Y2)/3, mid-time, as k_deform's y_ctr)
           A triangle invalid by k_deform's rule (masked vertex at either end; signed area not positive at k0, k1 or
           mid-time) contributes +0.0 to every sum.  Interior edges cancel, so Sux/Sa2 is the line-integral rate of
           the union (holes allowed).
Order.     Level 1: one warp per box; lane l sums the triangles l, l+32, l+64, ... of the box left to right from
           +0.0, then an xor butterfly with offsets 16, 8, 4, 2, 1: p = p + p[l ^ o].  Level s+1:
           ((c0 + c1) + c2) + c3 over the children that exist, in Morton order, from +0.0.
Outputs.   Per box, f8: ux = Sux/Sa2 (uy, vx, vy likewise), area = 0.5 Sa2, D = ux + vy, d = ux - vy, e = uy + vx,
           shear = sqrt(d*d + e*e), vorticity = vx - uy, eps_tot = sqrt((D*D + d*d) + e*e), L_eff = sqrt(area),
           centroid SY/Sa2, SX/Sa2.  Valid when area >= cover * L_s^2 (the threshold passed per level in f8).
           Scale 0: every valid triangle, with its own k_deform rates and L_eff = sqrt(A).  The f4 box outputs are
           the f8 values rounded once, FillValue where invalid.
Stats.     Per scale: n valid cells; sums of L_eff, eps_tot, eps_tot^2 = eps_tot*eps_tot and eps_tot^3 =
           eps_tot^2*eps_tot (math.fsum here; the device's fixed-order sums agree within 1e-11 relative);
           histograms of eps_tot, |D| and shear on f8 edges, bin = searchsorted(edges, v, side="right"), so
           len(edges) + 1 counts, underflow and overflow included.

Every element-wise operation is spelled in the kernel's order; numpy's f8 operations are correctly rounded and never
contracted, so box sums, box outputs and counts are bit-identical to the kernels'.
"""
import math

import numpy as np

from . import deform_ref as R

FillValue = -9999.0
BOX_NAMES = ("divergence", "shear", "vorticity", "total", "L_eff", "y_ctr", "x_ctr")
DEFAULT_EDGES = np.array([10.0 ** (k / 10.0) for k in range(-50, 11)])   # 1e-5 ... 1e1 day-1, 10 bins per decade


def _spread(v):
    v = v.astype(np.uint64)
    for s, m in ((16, 0x0000FFFF0000FFFF), (8, 0x00FF00FF00FF00FF), (4, 0x0F0F0F0F0F0F0F0F),
                 (2, 0x3333333333333333), (1, 0x5555555555555555)):
        v = (v | (v << np.uint64(s))) & np.uint64(m)
    return v


def hierarchy(yx, tri, L0, levels):
    """-> dict(order (nT,) sorted triangle order, origin (2,), levels=[dict(key (nb,2) [bj,bi], off (nb+1,) ranges of
    the sorted triangles, child (nb+1,) ranges of the previous level's boxes or None)])."""
    yx = np.asarray(yx, np.float64)
    tri = np.asarray(tri, np.int64).reshape(-1, 3)
    c = np.stack([((yx[tri[:, 0], k] + yx[tri[:, 1], k]) + yx[tri[:, 2], k]) / 3.0 for k in (0, 1)], 1)
    origin = np.floor(c.min(0) / L0) * L0
    key = np.floor((c - origin) / L0).astype(np.int64)
    code = (_spread(key[:, 0]) << np.uint64(1)) | _spread(key[:, 1])
    order = np.argsort(code, kind="stable")
    cs, ks = code[order], key[order]
    out = []
    prev = None
    for s in range(levels):
        cl = cs >> np.uint64(2 * s)
        st = np.flatnonzero(np.r_[True, cl[1:] != cl[:-1]])
        lv = dict(key=ks[st] >> s, off=np.r_[st, cs.size], child=None)
        if prev is not None:
            lv["child"] = np.r_[np.searchsorted(prev, st), prev.size]
        out.append(lv)
        prev = st
    return dict(order=order, origin=origin, levels=out)


def triangle_terms(yx0, yx1, mask0, mask1, tri, dt):
    """-> (T (nT,7) f8 [a2, Nux, Nuy, Nvx, Nvy, NY, NX], +0.0 rows for invalid triangles; rates_f8's dict; valid)."""
    yx0, yx1 = np.asarray(yx0, np.float64), np.asarray(yx1, np.float64)
    tri = np.asarray(tri, np.int64).reshape(-1, 3)
    dt = np.float64(dt)
    y0, x0, y1, x1 = yx0[tri, 0], yx0[tri, 1], yx1[tri, 0], yx1[tri, 1]
    with np.errstate(all="ignore"):
        X, Y = 0.5 * (x0 + x1), 0.5 * (y0 + y1)
        U, V = (x1 - x0) / dt, (y1 - y0) / dt
        a2 = R.twice_area(X, Y)
        T = np.stack([a2, R.edge_sum(U, Y), -R.edge_sum(U, X), R.edge_sum(V, Y), -R.edge_sum(V, X),
                      a2 * (((Y[:, 0] + Y[:, 1]) + Y[:, 2]) / 3.0), a2 * (((X[:, 0] + X[:, 1]) + X[:, 2]) / 3.0)], 1)
    r, valid = R.rates_f8(yx0, yx1, mask0, mask1, tri, dt)
    T[~valid] = 0.0
    return T, r, valid


def level1_sums(Ts, off, boxes=None):
    """Warp order: lane partial sums, then the xor butterfly.  Ts (nT,7) in hierarchy order; -> (nb,7)."""
    b = np.arange(off.size - 1) if boxes is None else np.asarray(boxes)
    lo, hi = off[b], off[b + 1]
    lane = np.arange(32)
    P = np.zeros((b.size, 32, Ts.shape[1]))
    for r in range(int(-(-(hi - lo).max() // 32)) if b.size else 0):
        idx = lo[:, None] + 32 * r + lane
        ok = idx < hi[:, None]
        P[ok] = P[ok] + Ts[idx[ok]]
    for o in (16, 8, 4, 2, 1):
        P = P + P[:, lane ^ o]
    return P[:, 0]


def parent_sums(Sc, child):
    S = np.zeros((child.size - 1, Sc.shape[1]))
    for k in range(4):
        idx = child[:-1] + k
        ok = idx < child[1:]
        S[ok] = S[ok] + Sc[idx[ok]]
    return S


def rates_of(ux, uy, vx, vy):
    D, d, e = ux + vy, ux - vy, uy + vx
    return dict(divergence=D, shear=np.sqrt(d * d + e * e), vorticity=vx - uy, total=np.sqrt((D * D + d * d) + e * e))


def box_outputs(S, min_area):
    """S (nb,7) sums -> (dict of f8 BOX_NAMES, valid)."""
    with np.errstate(all="ignore"):
        a = S[:, 0]
        o = rates_of(S[:, 1] / a, S[:, 2] / a, S[:, 3] / a, S[:, 4] / a)
        area = 0.5 * a
        o.update(L_eff=np.sqrt(area), y_ctr=S[:, 5] / a, x_ctr=S[:, 6] / a)
    return o, area >= np.float64(min_area)


def cell_stats(o, valid, edges):
    """-> dict(n, sums [L_eff, eps_tot, eps_tot^2, eps_tot^3] by fsum, hist (3, len(edges)+1)) over the valid cells."""
    t = o["total"][valid]
    t2 = t * t
    hist = np.stack([np.bincount(np.searchsorted(edges, v, side="right"), minlength=edges.size + 1)
                     for v in (t, np.abs(o["divergence"][valid]), o["shear"][valid])]).astype(np.int64)
    return dict(n=int(valid.sum()), sums=np.array([math.fsum(o["L_eff"][valid]), math.fsum(t), math.fsum(t2),
                                                   math.fsum(t2 * t)]), hist=hist)


def coarse_grain(yx0, yx1, mask0, mask1, tri, dt, H, cover=0.5, edges=DEFAULT_EDGES, L0=None):
    """H: hierarchy(...) (L0 given) -> (boxes: per level dict(key, valid, S (nb,7), f4 BOX_NAMES),
    stats: dict(n (S,), sums (S,4), hist (S,3,len(edges)+1)))."""
    edges = np.asarray(edges, np.float64)
    T, r, valid = triangle_terms(yx0, yx1, mask0, mask1, tri, dt)
    Ts = T[H["order"]]
    with np.errstate(all="ignore"):
        o0 = rates_of(r["ux"], r["uy"], r["vx"], r["vy"])
        o0["L_eff"] = np.sqrt(r["area"])
    st = [cell_stats(o0, valid, edges)]
    boxes = []
    S = None
    for s, lv in enumerate(H["levels"]):
        S = level1_sums(Ts, lv["off"]) if s == 0 else parent_sums(S, lv["child"])
        Ls = L0 * 2.0 ** s
        o, ok = box_outputs(S, cover * Ls * Ls)
        st.append(cell_stats(o, ok, edges))
        b = dict(key=lv["key"], valid=ok, S=S)
        with np.errstate(all="ignore"):
            b.update({k: np.where(ok, o[k], FillValue).astype(np.float32) for k in BOX_NAMES})
        boxes.append(b)
    return boxes, dict(n=np.array([x["n"] for x in st], np.int64), sums=np.stack([x["sums"] for x in st]),
                       hist=np.stack([x["hist"] for x in st]))


def coarse_grain_series(posC, mask, tri, every, rdt, H, **kw):
    """The statistics of the windows [w*every, (w+1)*every] of a (nrec+1, nP, 2) series (partial window dropped)."""
    nwin = (posC.shape[0] - 1) // every
    return [coarse_grain(posC[w * every], posC[(w + 1) * every], mask[w * every], mask[(w + 1) * every], tri,
                         every * rdt / 86400.0, H, **kw)[1] for w in range(nwin)]
