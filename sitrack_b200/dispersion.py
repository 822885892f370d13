"""Two-particle (pair) dispersion of buoys over time lags, and its per-window statistics by initial separation
(Rampal et al. 2008; Girard et al. 2009; Lukovich et al.).

Definitions (DESIGN.md section 13).  For a pair of buoys (a, b) followed from an origin row to a row tau days later,
r0 and r1 are their separations at the two rows, dr = r1 - r0 the change of separation, dD2 the squared change of the
separation vector, and s = |dr| / (r0 tau) the stretch rate [day-1].  A pair counts when both buoys have mask != 0 in
both rows.  Pairs are classed by r0 on `r_edges` (default 10 ... 1000 km, 4 classes per decade) and s is binned on
`bins` (default section 11's edges); both with searchsorted(edges, v, side="right"), underflow and overflow included.
Per lag and class the statistics are the stretch-rate histogram, n and the sums of r0, dr, dr^2 and dD2: sums, so
that windows add up to ensembles.  They are computed on the device (csrc/st_disperse.cu) in a fixed order:
bit-identical run to run and whatever order the buoys are stored in.  No CPU fallback.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_c, check
from .deform_scales import DEFAULT_BIN_EDGES, MAX_EDGES

__all__ = ["MeshPairs", "SeparationPairs", "PairDispersion", "check_pairs", "DEFAULT_R_EDGES", "MAX_LAGS",
           "PAIR_NAMES"]

FillValue = -9999.0
DEFAULT_R_EDGES = np.array([10.0 ** (1.0 + k / 4.0) for k in range(9)])          # 10 ... 1000 km, 4 per decade
MAX_LAGS = 64
MAX_CLASS_EDGES = 63
PAIR_NAMES = ("r0", "r1", "dr", "dD2")


def MeshPairs(tri):
    """-> (nE,2) i4: the unique undirected edges (a < b) of a triangle mesh (TriangulateCloud), sorted; the
    nearest-neighbour pairs."""
    t = as_c(tri, np.int64).reshape(-1, 3)
    e = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
    a, b = e.min(1), e.max(1)
    n = int(b.max()) + 1 if b.size else 1
    key = np.unique(a * n + b)
    return as_c(np.stack(np.divmod(key, n), 1), np.int32)


def SeparationPairs(pYX, r_min_km, r_max_km, n, seed=0):
    """-> (nQ,2) i4 pairs of buoys pYX (nP,2) [y,x] km spread over separations [r_min_km, r_max_km]: for each of n
    draws a random buoy i, a target at a log-uniform distance in [r_min, r_max] in a uniform direction, and the buoy
    j nearest that target (scipy.spatial.cKDTree).  Draws with i == j are dropped; the unique pairs (a < b) are
    returned sorted.  Host only, deterministic for a seed."""
    from scipy.spatial import cKDTree
    yx = as_c(pYX, np.float64).reshape(-1, 2)
    if not (np.isfinite(r_min_km) and r_min_km > 0 and np.isfinite(r_max_km) and r_max_km > r_min_km):
        raise ValueError("SeparationPairs: need 0 < r_min_km < r_max_km, got %r, %r" % (r_min_km, r_max_km))
    if int(n) != n or n < 1:
        raise ValueError("SeparationPairs: n must be a positive integer, got %r" % (n,))
    if yx.shape[0] < 2:
        raise ValueError("SeparationPairs: need at least two buoys")
    rng = np.random.default_rng(seed)
    n = int(n)
    i = rng.integers(0, yx.shape[0], n)
    r = np.exp(rng.uniform(np.log(r_min_km), np.log(r_max_km), n))
    th = rng.uniform(0.0, 2.0 * np.pi, n)
    target = yx[i] + np.stack([r * np.sin(th), r * np.cos(th)], 1)
    j = cKDTree(yx).query(target)[1].astype(np.int64)
    keep = i != j
    a, b = np.minimum(i, j)[keep], np.maximum(i, j)[keep]
    key = np.unique(a * yx.shape[0] + b)
    return as_c(np.stack(np.divmod(key, yx.shape[0]), 1), np.int32)


def check_pairs(pairs, nP):
    """(nQ,2) i4 copy of pairs: nQ >= 1, every index in [0, nP) (the kernel does not range-check), a != b."""
    p = np.asarray(pairs)
    if p.ndim != 2 or p.shape[1] != 2 or p.shape[0] < 1:
        raise ValueError("pairs must have shape (nQ, 2) with nQ >= 1, got %s" % (p.shape,))
    if p.shape[0] >= 2 ** 31:
        raise ValueError("pairs: at most 2^31 - 1 pairs")
    if not np.issubdtype(p.dtype, np.integer):
        raise ValueError("pairs must be integer buoy indices")
    if p.min() < 0 or p.max() >= nP:
        raise ValueError("pair index out of range [0, %d)" % nP)
    if (p[:, 0] == p[:, 1]).any():
        raise ValueError("a pair joins a buoy to itself (a == b)")
    return as_c(p, np.int32)


def check_edges(edges, default, limit, what):
    e = as_c(default if edges is None else edges, np.float64).ravel()
    if not 1 <= e.size <= limit or not np.isfinite(e).all() or (np.diff(e) <= 0).any():
        raise ValueError("%s must be 1..%d finite, strictly increasing edges" % (what, limit))
    return e


def check_lags(lags):
    if int(lags) != lags or not 1 <= lags <= MAX_LAGS:
        raise ValueError("lags must be an integer in 1..%d, got %r" % (MAX_LAGS, lags))
    return int(lags)


class _Plan:
    """Device buffers of one set of pairs (buoy indices as stored on the device, caller's pair order), edges and
    scratch for calls with up to `lags` active origins."""

    def __init__(self, torch, dev, slots, lags, r_edges=None, bins=None):
        self.torch, self.L = torch, _lib.lib()
        self.lags = check_lags(lags)
        self.r_edges = check_edges(r_edges, DEFAULT_R_EDGES, MAX_CLASS_EDGES, "r_edges")
        self.bins = check_edges(bins, DEFAULT_BIN_EDGES, MAX_EDGES, "bins")
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        self.pairs_t = t(slots, np.int32)
        self.nQ = int(self.pairs_t.shape[0])
        self.r_edges_t, self.bins_t = t(self.r_edges, np.float64), t(self.bins, np.float64)
        nb = C.c_int64()
        check(self.L.st_dispersion_scratch_bytes(self.nQ, self.lags, self.r_edges.size, self.bins.size, C.byref(nb)),
              None)
        self.scratch_bytes = nb.value
        self.scratch = torch.empty((nb.value + 7) // 8, dtype=torch.float64, device=dev)
        self.C, self.NB = self.r_edges.size + 1, self.bins.size + 1

    def outputs(self, pin=False):
        """(hist (lags, C, NB) i8, sums (lags, C, 4) f8) on the device, or pinned on the host."""
        kw = dict(pin_memory=True) if pin else dict(device=self.scratch.device)
        return (self.torch.empty((self.lags, self.C, self.NB), dtype=self.torch.int64, **kw),
                self.torch.empty((self.lags, self.C, 4), dtype=self.torch.float64, **kw))

    def launch(self, ctx, yx1_t, m1_t, origins, dt_days, hist_t, sums_t, per_pair_t, stream):
        """st_dispersion_dev (async on `stream`); origins = [(yx0_t, m0_t, lag), ...]."""
        n = len(origins)
        yx0 = (C.c_void_p * max(n, 1))(*[o[0].data_ptr() for o in origins])
        m0 = (C.c_void_p * max(n, 1))(*[o[1].data_ptr() for o in origins])
        lag = (C.c_int * max(n, 1))(*[int(o[2]) for o in origins])
        check(self.L.st_dispersion_dev(
            ctx, self.nQ, self.pairs_t.data_ptr(), yx1_t.data_ptr(), m1_t.data_ptr(), n, C.cast(yx0, C.c_void_p),
            C.cast(m0, C.c_void_p), C.cast(lag, C.c_void_p), float(dt_days), self.lags, self.r_edges.size,
            self.r_edges_t.data_ptr(), self.bins.size, self.bins_t.data_ptr(), self.scratch.data_ptr(),
            self.scratch_bytes, hist_t.data_ptr(), sums_t.data_ptr(),
            None if per_pair_t is None else per_pair_t.data_ptr(), C.c_void_p(stream.cuda_stream)), ctx)


def stats_dict(lag_days, r_edges, bins, hist, sums):
    """Host hist (m, C, NB) and sums (m, C, 4) -> the statistics of one window (see PairDispersion)."""
    hist, sums = np.array(hist, np.int64), np.array(sums, np.float64)
    return dict(lag_days=np.asarray(lag_days, np.float64).copy(), r_edges=r_edges.copy(), bin_edges=bins.copy(),
                n=hist.sum(2), sum_r0=sums[..., 0], sum_dr=sums[..., 1], sum_dr2=sums[..., 2], sum_dD2=sums[..., 3],
                hist_stretch=hist)


def PairDispersion(pYX0, pYX1, mask0, mask1, pairs, dt_days, r_edges=None, bins=None, device=None):
    """Dispersion of the buoy pairs `pairs` (nQ,2) between positions pYX0 and pYX1 ((nP,2) [y,x] km) with masks
    mask0, mask1 (nP,), dt_days apart (one lag).  Host arrays in and out; computed on the GPU.

    -> (per_pair, stats).  per_pair: dict of (nQ,) f8 PAIR_NAMES r0, r1 [km], dr [km], dD2 [km2], FillValue where the
    pair does not count.  stats: lag_days (1,), r_edges, bin_edges, n (1, C) i8, sum_r0, sum_dr, sum_dr2, sum_dD2
    (1, C) f8 and hist_stretch (1, C, len(bins)+1) i8 of s = |dr| / (r0 dt_days), C = len(r_edges) + 1."""
    from .engine import _torch
    from . import config
    torch = _torch()
    yx0, yx1 = as_c(pYX0, np.float64).reshape(-1, 2), as_c(pYX1, np.float64).reshape(-1, 2)
    nP = yx0.shape[0]
    if yx1.shape[0] != nP or np.shape(mask0) != (nP,) or np.shape(mask1) != (nP,):
        raise ValueError("pYX0, pYX1 (nP,2) and mask0, mask1 (nP,) must describe the same buoys")
    if not dt_days > 0:
        raise ValueError("dt_days must be positive")
    pairs = check_pairs(pairs, nP)
    dev = torch.device("cuda", config.device if device is None else int(device))
    with torch.cuda.device(dev):
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        plan = _Plan(torch, dev, pairs, 1, r_edges, bins)
        hist, sums = plan.outputs()
        pp = torch.empty((4, plan.nQ), dtype=torch.float64, device=dev)
        plan.launch(None, t(yx1, np.float64), t(mask1, np.int8), [(t(yx0, np.float64), t(mask0, np.int8), 1)],
                    dt_days, hist, sums, pp, torch.cuda.current_stream(dev))
        pp, hist, sums = pp.cpu().numpy(), hist.cpu().numpy(), sums.cpu().numpy()
    return ({n: pp[j].copy() for j, n in enumerate(PAIR_NAMES)},
            stats_dict([float(dt_days)], plan.r_edges, plan.bins, hist, sums))
