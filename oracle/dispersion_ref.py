"""Reference two-particle (pair) dispersion of buoys over time lags, and its per-window statistics (test infrastructure
only; the product never imports it).

Method -- the contract of csrc/st_disperse.cu, sitrack_b200.dispersion and DESIGN.md section 13:

Pairs.     pairs (nQ,2) i4 of buoy indices in the caller's order, a != b, nQ >= 1; kept in that order.
Windows.   As in section 10: with every = n, row (w+1)*n closes window w; row 0 is the state handed to set_buoys,
           masked by the rec_first rule of the engine's _WindowRows.  The rows o*n, o = 0, 1, ..., are origins.
           When window w closes, lags l = 1 .. min(m, w+1) are evaluated between origin row (w+1-l)*n and row
           (w+1)*n, with tau_l = l*n*rdt/86400 days.  Every (origin, lag) combination is evaluated exactly once in a
           run, so the sum of the windows' statistics is the ensemble over all start times at every lag.
Per pair.  For one (origin, lag): valid when both buoys have mask != 0 in both rows.  In f8, in this order:
             dy0 = y_a - y_b, dx0 = x_a - x_b, r0 = sqrt(dy0*dy0 + dx0*dx0); dy1, dx1, r1 likewise at the lag row;
             dr = r1 - r0;  dD2 = (dy1-dy0)*(dy1-dy0) + (dx1-dx0)*(dx1-dx0);  s = |dr| / (r0*tau_l)  [day-1].
Classes.   class = searchsorted(r_edges, r0, side="right"): len(r_edges) + 1 classes with underflow and overflow, NaN
           last.  Stretch bin = searchsorted(bins, s, side="right") (section 11's bin_right).  Defaults: r_edges
           10 ... 1000 km, 4 classes per decade; bins section 11's DEFAULT_BIN_EDGES.  r0 = 0 gives s = inf or NaN:
           the overflow bin.  Ties go to the upper class or bin.
Stats.     Per window, lag and class: hist_stretch (m, C, len(bins)+1) i8 counts (exact), n its row sum, sum_r0,
           sum_dr, sum_dr2 (= dr*dr), sum_dD2 f8.  Lags not reached yet have zero counts and zero sums.  The device
           sums in the fixed order below, so its sums are bit-identical to order_sums; lag_stats' math.fsum is the
           accuracy reference (the fixed order agrees with it within 1e-11 * fsum(|terms|)).
Order.     For one (origin, lag), pair i is in tile i // 256, warp (i % 256) // 32, lane i % 32; nblk =
           min(max(ceil(nQ/256), 1), 1184) blocks, block b taking tiles b, b + nblk, ... in turn.  Per tile, warp and
           class: x = v on the lanes of that class (pairs that do not count have none) and +0.0 on the others, then
           x = x + x[lane ^ sh] for sh = 16, 8, 4, 2, 1; lane 0 is the warp partial (+0.0 for a class absent from the
           warp).  Block partial part[b]: +0.0, then per tile warp partials 0 ... 7 added one after another.  Final:
           slot t of 256 starts at +0.0 and adds part[t], part[t+256], ... in turn; then s[t] += s[t+w] for
           w = 128 ... 1, and the sum is s[0].

Every element-wise operation is spelled in the kernel's order; numpy's f8 operations are correctly rounded and never
contracted, so the per-pair values, the counts and order_sums' sums and block partials are bit-identical to the
kernel's.
"""
import math

import numpy as np

FillValue = -9999.0
DEFAULT_R_EDGES = np.array([10.0 ** (1.0 + k / 4.0) for k in range(9)])          # 10 ... 1000 km, 4 per decade
DEFAULT_BINS = np.array([10.0 ** (k / 10.0) for k in range(-50, 11)])            # section 11's DEFAULT_BIN_EDGES


def per_pair(yx0, yx1, m0, m1, pairs):
    """-> dict(r0, r1, dr, dD2 (nQ,) f8, valid (nQ,) bool); values of invalid pairs are computed all the same."""
    yx0, yx1 = np.asarray(yx0, np.float64), np.asarray(yx1, np.float64)
    m0, m1 = np.asarray(m0), np.asarray(m1)
    a, b = np.asarray(pairs, np.int64)[:, 0], np.asarray(pairs, np.int64)[:, 1]
    with np.errstate(all="ignore"):
        dy0, dx0 = yx0[a, 0] - yx0[b, 0], yx0[a, 1] - yx0[b, 1]
        dy1, dx1 = yx1[a, 0] - yx1[b, 0], yx1[a, 1] - yx1[b, 1]
        r0 = np.sqrt(dy0 * dy0 + dx0 * dx0)
        r1 = np.sqrt(dy1 * dy1 + dx1 * dx1)
        ey, ex = dy1 - dy0, dx1 - dx0
        dD2 = ey * ey + ex * ex
        dr = r1 - r0
    valid = (m0[a] != 0) & (m0[b] != 0) & (m1[a] != 0) & (m1[b] != 0)
    return dict(r0=r0, r1=r1, dr=dr, dD2=dD2, valid=valid)


def per_pair_filled(yx0, yx1, m0, m1, pairs):
    """(4, nQ) f8 r0, r1, dr, dD2 with FillValue for invalid pairs (the kernel's per-pair output)."""
    p = per_pair(yx0, yx1, m0, m1, pairs)
    return np.stack([np.where(p["valid"], p[k], FillValue) for k in ("r0", "r1", "dr", "dD2")])


def pair_class(p, r_edges):
    """(nQ,) class of each pair of per_pair's p by r0: searchsorted(r_edges, r0, side="right"), NaN last; -1 for the
    pairs that do not count."""
    cls = np.searchsorted(r_edges, p["r0"], side="right")
    cls[np.isnan(p["r0"])] = r_edges.size
    return np.where(p["valid"], cls, -1)


def lag_hist(p, tau, r_edges=DEFAULT_R_EDGES, bins=DEFAULT_BINS):
    """(C, len(bins)+1) i8 counts by class of the stretch rate s = |dr| / (r0 tau) of per_pair's p."""
    r_edges, bins = np.asarray(r_edges, np.float64), np.asarray(bins, np.float64)
    cls = pair_class(p, r_edges)
    v = cls >= 0
    with np.errstate(all="ignore"):
        s = np.abs(p["dr"][v]) / (p["r0"][v] * np.float64(tau))
    sb = np.searchsorted(bins, s, side="right")
    sb[np.isnan(s)] = bins.size
    hist = np.zeros((r_edges.size + 1, bins.size + 1), np.int64)
    np.add.at(hist, (cls[v], sb), 1)
    return hist


def lag_stats(yx0, yx1, m0, m1, pairs, tau, r_edges=DEFAULT_R_EDGES, bins=DEFAULT_BINS):
    """One (origin, lag): -> dict(hist (C, len(bins)+1) i8, sums (C, 4) f8 by fsum, absum (C, 4) fsum of |terms|)."""
    r_edges = np.asarray(r_edges, np.float64)
    p = per_pair(yx0, yx1, m0, m1, pairs)
    cls = pair_class(p, r_edges)
    v = cls >= 0
    cls, r0, dr, dD2 = cls[v], p["r0"][v], p["dr"][v], p["dD2"][v]
    terms = (r0, dr, dr * dr, dD2)
    C = r_edges.size + 1
    sums, absum = np.zeros((C, 4)), np.zeros((C, 4))
    for c in np.unique(cls):
        sel = cls == c
        for q, t in enumerate(terms):
            sums[c, q] = math.fsum(t[sel])
            absum[c, q] = math.fsum(np.abs(t[sel]))
    return dict(hist=lag_hist(p, tau, r_edges, bins), sums=sums, absum=absum)


TILE, WARPS, MAX_GRID = 256, 8, 1184          # pairs per tile (one block of the kernel), warps per tile, blocks


def order_sums(yx0, yx1, m0, m1, pairs, r_edges=DEFAULT_R_EDGES):
    """One (origin, closing row) in the device's summation order (Order above): -> (sums (C, 4) f8 of r0, dr, dr*dr,
    dD2, block partials part (nblk, C, 4) f8).  Vectorised over blocks; loops over rounds of tiles, classes and
    butterfly strides."""
    r_edges = np.asarray(r_edges, np.float64)
    p = per_pair(yx0, yx1, m0, m1, pairs)
    cls = pair_class(p, r_edges)
    with np.errstate(all="ignore"):
        v = np.stack([p["r0"], p["dr"], p["dr"] * p["dr"], p["dD2"]], 1)
    nQ, C = cls.size, r_edges.size + 1
    ntile = -(-nQ // TILE)
    nblk = min(max(ntile, 1), MAX_GRID)
    nround = -(-ntile // nblk)
    pad = nround * nblk * TILE - nQ                       # lanes past nQ do not count
    cls = np.r_[cls, np.full(pad, -1)].reshape(nround, nblk, WARPS, 32)
    v = np.concatenate([v, np.zeros((pad, 4))]).reshape(nround, nblk, WARPS, 32, 4)
    lane = np.arange(32)
    part = np.zeros((nblk, C, 4))
    with np.errstate(all="ignore"):
        for r in range(nround):
            runs = (r * nblk + np.arange(nblk) < ntile)[:, None, None]      # the blocks that have a tile this round
            wp = np.zeros((nblk, WARPS, C, 4))
            for c in range(C):
                x = np.where((cls[r] == c)[..., None], v[r], 0.0)            # (nblk, warp, lane, 4)
                for sh in (16, 8, 4, 2, 1):
                    x = x + x[:, :, lane ^ sh]
                wp[:, :, c] = x[:, :, 0]
            for w in range(WARPS):
                part = np.where(runs, part + wp[:, w], part)
        s = np.zeros((TILE, C, 4))
        for b0 in range(0, nblk, TILE):
            k = min(TILE, nblk - b0)
            s[:k] = s[:k] + part[b0:b0 + k]
        w = TILE // 2
        while w:
            s[:w] = s[:w] + s[w:2 * w]
            w //= 2
    return s[0].copy(), part


def window_stats(rows, masks, w, lags, dt_days, r_edges=DEFAULT_R_EDGES, bins=DEFAULT_BINS, pairs=None, every=1):
    """Window w of a series of rows (row k = rows[k]): -> dict(hist (m, C, NB), sums, absum (m, C, 4)) with lags
    1 .. min(m, w+1) between rows (w+1-l)*every and (w+1)*every."""
    C, NB = np.asarray(r_edges).size + 1, np.asarray(bins).size + 1
    out = dict(hist=np.zeros((lags, C, NB), np.int64), sums=np.zeros((lags, C, 4)), absum=np.zeros((lags, C, 4)))
    k1 = (w + 1) * every
    for l in range(1, min(lags, w + 1) + 1):
        k0 = (w + 1 - l) * every
        st = lag_stats(rows[k0], rows[k1], masks[k0], masks[k1], pairs, l * dt_days, r_edges, bins)
        for k in out:
            out[k][l - 1] = st[k]
    return out


def series_stats(posC, mask, pairs, every, lags, rdt, r_edges=DEFAULT_R_EDGES, bins=DEFAULT_BINS):
    """The statistics of every window of a (nrec+1, nP, 2) series (a trailing partial window is dropped)."""
    nwin = (posC.shape[0] - 1) // every
    return [window_stats(posC, mask, w, lags, every * rdt / 86400.0, r_edges, bins, pairs, every) for w in range(nwin)]
