"""Finite-size Lyapunov exponents (FSLE) of buoy pairs: the times pairs take to grow from one separation threshold to
the next, kept as first-passage state on the device during tracking (Aurell et al. 1997; Lacorata et al. 2001;
LaCasce 2008).

Definitions (DESIGN.md section 14).  Every pair carries {level, anchor} across the whole run: the number of thresholds
`deltas` its separation has reached and the sample at which it first reached the current one.  A pair starts at its
first valid sample (both masks != 0, finite separation), ends at its first invalid one after that, and each time it
first reaches a higher threshold the exit time tau_j (in samples) of transition j: delta_j -> delta_{j+1} is recorded
(tau = 0 for thresholds first reached in the same sample interval; the first transition of a pair that starts above
delta_j is not timed).  Per window the statistics are integer: n_start by starting level, the histogram of tau per
transition on `tau_edges`, n, sum_tau, sum_tau2 and the censored transitions.  fsle_lambda gives
lambda_j = ln(delta_{j+1}/delta_j) / <tau_j> [day-1].  Computed on the device (csrc/st_fsle.cu) with integer atomics:
exact, whatever order the buoys are stored in.  No CPU fallback.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_c, check
from .deform_scales import check_edges
from .dispersion import check_pairs

__all__ = ["FiniteSizeLyapunov", "fsle_lambda", "DEFAULT_DELTAS", "DEFAULT_TAU_EDGES", "MAX_THRESHOLDS",
           "MAX_SAMPLES"]

DEFAULT_DELTAS = np.array([2.0 ** (1 + j / 2) for j in range(19)])                 # 2 ... 1024 km, ratio sqrt(2)
DEFAULT_TAU_EDGES = np.array([2.0 ** k for k in range(17)])                        # 1, 2, 4, ... 2^16 samples
MAX_THRESHOLDS = 64
MAX_TAU_EDGES = 512
MAX_SAMPLES = 65535


def check_deltas(deltas):
    """K f8 thresholds [km]: finite, positive, strictly increasing, 2 <= K <= MAX_THRESHOLDS (None: the default)."""
    d = DEFAULT_DELTAS if deltas is None else np.asarray(deltas, np.float64).ravel()
    if not 2 <= d.size <= MAX_THRESHOLDS:
        raise ValueError("deltas: need 2..%d thresholds, got %d" % (MAX_THRESHOLDS, d.size))
    if not (np.isfinite(d).all() and d[0] > 0 and (np.diff(d) > 0).all()):
        raise ValueError("deltas must be finite, positive and strictly increasing")
    return as_c(d.copy(), np.float64)


class _Plan:
    """Device buffers of one set of pairs (buoy indices as stored on the device, caller's pair order), thresholds,
    exit-time edges and the per-pair state; it counts its samples.  As a pass of TrackEngine.track's window driver
    (lags = 1), window 0 evaluates its single origin, row 0, as sample 0 and its closing row as sample 1; later
    windows ignore the origins."""

    def __init__(self, torch, dev, slots, deltas=None, tau_edges=None, sample_days=None):
        self.torch, self.L = torch, _lib.lib()
        self.deltas = check_deltas(deltas)
        self.tau_edges = check_edges(tau_edges, DEFAULT_TAU_EDGES, MAX_TAU_EDGES, "tau_edges")
        self.sample_days = sample_days
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        self.pairs_t = t(slots, np.int32)
        self.nQ = int(self.pairs_t.shape[0])
        self.deltas_t, self.tau_edges_t = t(self.deltas, np.float64), t(self.tau_edges, np.float64)
        nb = C.c_int64()
        check(self.L.st_fsle_state_bytes(self.nQ, self.deltas.size, self.tau_edges.size, C.byref(nb)), None)
        self.state = torch.empty((nb.value // 8, 2), dtype=torch.int32, device=dev)
        K, J = self.deltas.size, self.deltas.size - 1
        self.nstat = K + 1 + J * (self.tau_edges.size + 4)
        self.t = 0

    def outputs(self, pin=False):
        """(stats (nstat,) i8,) on the device, or pinned on the host."""
        kw = dict(pin_memory=True) if pin else dict(device=self.state.device)
        return (self.torch.empty((self.nstat,), dtype=self.torch.int64, **kw),)

    def launch(self, ctx, yx_t, m_t, t, start, stats_t, stream):
        """st_fsle_dev for sample t (async on `stream`); start = (yx0_t, m0_t), row t-1 with a reset, or None."""
        check(self.L.st_fsle_dev(
            ctx, self.nQ, self.pairs_t.data_ptr(), self.state.data_ptr(), yx_t.data_ptr(), m_t.data_ptr(), int(t),
            None if start is None else start[0].data_ptr(), None if start is None else start[1].data_ptr(),
            self.deltas.size, self.deltas_t.data_ptr(), self.tau_edges.size, self.tau_edges_t.data_ptr(),
            stats_t.data_ptr(), C.c_void_p(stream.cuda_stream)), ctx)

    def window(self, ctx, origins, yx1_t, m1_t, dt_days, outs, stream):
        """TrackEngine.track's pass over one window: the next sample."""
        self.t += 1
        if self.t > MAX_SAMPLES:
            raise ValueError("fsle: at most %d samples in a run" % MAX_SAMPLES)
        start = origins[0][:2] if self.t == 1 else None
        self.launch(ctx, yx1_t, m1_t, self.t, start, outs[0], stream)

    def results(self, outs):
        """(the statistics of the window,) from its pinned outputs."""
        return (stats_dict(self.deltas, self.tau_edges, self.sample_days, outs[0].numpy()),)

    def state_dict(self):
        s = self.state.cpu().numpy()
        return dict(level=s[:, 0].copy(), anchor=s[:, 1].copy())


def stats_dict(deltas, tau_edges, sample_days, buf):
    """One window's host stats buffer (layout of st_fsle_dev) -> dict(deltas_km, tau_edges, sample_days, n_start
    (K+1), hist_tau (K-1, NB), n, sum_tau, sum_tau2, n_censored (K-1)), all counts i8."""
    buf = np.array(buf, np.int64)
    K, NB = deltas.size, tau_edges.size + 1
    J = K - 1
    o = K + 1 + J * NB
    hist = buf[K + 1:o].reshape(J, NB)
    return dict(deltas_km=deltas.copy(), tau_edges=tau_edges.copy(),
                sample_days=None if sample_days is None else float(sample_days),
                n_start=buf[:K + 1], hist_tau=hist, n=hist.sum(1), sum_tau=buf[o:o + J], sum_tau2=buf[o + J:o + 2 * J],
                n_censored=buf[o + 2 * J:o + 3 * J])


def fsle_lambda(stats_list):
    """FSLE [day-1] per transition j from the windows' statistics summed: ln(delta_{j+1}/delta_j) / (sample_days *
    sum_tau_j / n_j); NaN where n_j = 0, +inf where sum_tau_j = 0 < n_j."""
    stats_list = [stats_list] if isinstance(stats_list, dict) else list(stats_list)
    if not stats_list:
        raise ValueError("fsle_lambda: no window")
    d, sd = stats_list[0]["deltas_km"], stats_list[0]["sample_days"]
    n = sum(np.asarray(s["n"], np.int64) for s in stats_list)
    tau = sum(np.asarray(s["sum_tau"], np.int64) for s in stats_list)
    with np.errstate(divide="ignore", invalid="ignore"):
        lam = np.log(d[1:] / d[:-1]) / (sd * (tau / n))
    return np.where(n == 0, np.nan, lam)


def FiniteSizeLyapunov(pYX, masks, pairs, sample_days, deltas=None, tau_edges=None, device=None):
    """FSLE statistics of the buoy pairs `pairs` (nQ,2) over the samples pYX (S+1, nP, 2) [y,x] km with masks
    (S+1, nP), sample_days days apart.  Host arrays in and out; computed on the GPU, one launch per sample.

    -> (state, stats).  state: dict of (nQ,) i4 `level` and `anchor` after the last sample.  stats: the list of the S
    windows' dicts (stats_dict; window w holds the events of sample w+1, window 0 also those of sample 0)."""
    from .engine import _torch
    from . import config
    torch = _torch()
    yx = as_c(pYX, np.float64)
    mk = np.asarray(masks)
    if yx.ndim != 3 or yx.shape[2] != 2 or yx.shape[0] < 2 or mk.shape != yx.shape[:2]:
        raise ValueError("pYX must have shape (S+1, nP, 2) with S >= 1 and masks (S+1, nP), got %s and %s"
                         % (yx.shape, mk.shape))
    S = yx.shape[0] - 1
    if S > MAX_SAMPLES:
        raise ValueError("at most %d samples after row 0" % MAX_SAMPLES)
    if not (np.isfinite(sample_days) and sample_days > 0):
        raise ValueError("sample_days must be finite and positive")
    dev = torch.device("cuda", config.device if device is None else int(device))
    with torch.cuda.device(dev):
        plan = _Plan(torch, dev, check_pairs(pairs, yx.shape[1]), deltas, tau_edges, sample_days)
        stream = torch.cuda.current_stream(dev)
        g = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        start = (g(yx[0], np.float64), g(mk[0] != 0, np.int8))
        outs = []
        for s in range(1, S + 1):
            o = plan.outputs()
            plan.window(None, [start], g(yx[s], np.float64), g(mk[s] != 0, np.int8), sample_days, o, stream)
            outs.append(o[0])
        stats = [plan.results((o.cpu(),))[0] for o in outs]
        return plan.state_dict(), stats
