"""Buoy transits between regions: which share of the ice that starts in one region reaches another, how long it takes,
and the region-to-region transitions of every window (DeRepentigny et al. 2016; Newton et al. 2017), counted on the
device from the host cells the engine already holds.

Definitions (DESIGN.md section 16).  A label map (Nj, Ni) on the T-grid names regions 1..R (R <= 31, the largest
label), 0 is "in no region"; a buoy's region is the label of its host cell.  A sample is valid when the row mask is
!= 0 and the cell lies in the grid's interior 1..Nj-2 x 1..Ni-2.  Every buoy carries {status, src, prev, start,
visited} across the whole run: it starts at its first valid sample in region src, ends for good at its first invalid
one after that, and each region r >= 1 it enters for the first time is a first arrival after tau = t - start samples.
Per window the statistics are integer: n_start, n_end by source region, the transitions trans[prev][cur] between
consecutive samples, the first arrivals n_arrive[src][dest], their sum_tau, sum_tau2 and histogram hist_tau on
`tau_edges` (all sums over the window's sample; window 0 also holds the starts of sample 0), and the snapshot
count[src][cur] of the started buoys at the window's closing sample.  Computed on the device (csrc/st_connect.cu) with
integer atomics: exact, whatever order the buoys are stored in and however they are split between processes.  No CPU
fallback.
"""
import ctypes as C

import numpy as np

from . import _lib
from . import fsle
from ._lib import as_c, check
from .deform_scales import check_edges

__all__ = ["RegionConnectivity", "MAX_REGIONS", "CONNECT_STATS"]

MAX_REGIONS = 31
CONNECT_STATS = ("n_start", "n_end", "count", "trans", "n_arrive", "sum_tau", "sum_tau2", "hist_tau")


def check_labels(labels, Nj, Ni):
    """A region map (Nj, Ni) -> (C-contiguous u8 map, R = its largest label).  Masked values become 0; a map of another
    shape, with negative, non-integral or non-finite labels, labels above MAX_REGIONS, or no label >= 1 is refused."""
    if isinstance(labels, np.ma.MaskedArray):
        labels = labels.astype(np.float64).filled(0.0)
    a = np.asarray(labels)
    if a.shape != (Nj, Ni):
        raise ValueError("labels must have shape (%d, %d), got %s" % (Nj, Ni, a.shape))
    if a.dtype.kind not in "biuf":
        raise ValueError("labels must be numbers, got dtype %s" % a.dtype)
    f = a.astype(np.float64)
    if not (np.isfinite(f).all() and (f == np.floor(f)).all()):
        raise ValueError("labels must be finite integers")
    if f.min() < 0 or f.max() > MAX_REGIONS:
        raise ValueError("labels must be in 0..%d, got %g..%g" % (MAX_REGIONS, f.min(), f.max()))
    R = int(f.max())
    if R < 1:
        raise ValueError("labels: no region (every label is 0)")
    return as_c(f.astype(np.uint8), np.uint8), R


def stats_dict(tau_edges, sample_days, nreg, buf):
    """One window's host stats buffer (layout of st_connect_dev) -> dict(tau_edges, sample_days, nreg, n_start, n_end
    (R+1), count, trans (R+1, R+1), n_arrive, sum_tau, sum_tau2 (R+1, R), hist_tau (R+1, R, NB)), all counts i8."""
    buf = np.array(buf, np.int64)
    R1, R, NB = nreg + 1, nreg, tau_edges.size + 1
    shapes = dict(n_start=(R1,), n_end=(R1,), count=(R1, R1), trans=(R1, R1), n_arrive=(R1, R), sum_tau=(R1, R),
                  sum_tau2=(R1, R), hist_tau=(R1, R, NB))
    out = dict(tau_edges=tau_edges.copy(), sample_days=None if sample_days is None else float(sample_days),
               nreg=int(nreg))
    o = 0
    for k in CONNECT_STATS:
        n = int(np.prod(shapes[k]))
        out[k] = buf[o:o + n].reshape(shapes[k])
        o += n
    if o != buf.size:
        raise ValueError("connect: a stats buffer of %d words, expected %d" % (buf.size, o))
    return out


class _Plan:
    """Device buffers of one connectivity setup: the label map, the arrival-time edges and the per-buoy state (in the
    engine's storage order); it counts its samples.  As a pass of TrackEngine.track's window driver (lags = 0: no
    origin ring), start() evaluates row 0 as sample 0 into window 0's outputs before step 0, and window w evaluates
    its closing row as sample w+1 from the context's cells."""

    def __init__(self, torch, dev, labels, nreg, Nj, Ni, nP, tau_edges=None, sample_days=None):
        self.torch, self.L = torch, _lib.lib()
        self.nreg, self.Nj, self.Ni, self.nP = int(nreg), int(Nj), int(Ni), int(nP)
        self.tau_edges = check_edges(tau_edges, fsle.DEFAULT_TAU_EDGES, fsle.MAX_TAU_EDGES, "tau_edges")
        self.sample_days = sample_days
        nb = C.c_int64()
        check(self.L.st_connect_state_bytes(self.nP, self.nreg, self.tau_edges.size, C.byref(nb)), None)
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        self.labels_t, self.tau_edges_t = t(labels, np.uint8), t(self.tau_edges, np.float64)
        self.state = torch.empty((nb.value // 8, 2), dtype=torch.int32, device=dev)
        R1, R = self.nreg + 1, self.nreg
        self.nstat = 2 * R1 + 2 * R1 * R1 + 3 * R1 * R + R1 * R * (self.tau_edges.size + 1)
        self.t = 0

    def outputs(self, pin=False):
        """(stats (nstat,) i8,) on the device, or pinned on the host."""
        kw = dict(pin_memory=True) if pin else dict(device=self.state.device)
        return (self.torch.empty((self.nstat,), dtype=self.torch.int64, **kw),)

    def launch(self, ctx, cell_t, m_t, t, stats_t, stream):
        """st_connect_dev for sample t (async on `stream`): cell_t (nP,2) i4 cell words, or None for the context's."""
        check(self.L.st_connect_dev(
            ctx, self.Nj, self.Ni, self.labels_t.data_ptr(), self.nreg, self.nP,
            None if cell_t is None else cell_t.data_ptr(), m_t.data_ptr(), int(t), self.state.data_ptr(),
            self.tau_edges.size, self.tau_edges_t.data_ptr(), stats_t.data_ptr(), C.c_void_p(stream.cuda_stream)), ctx)

    def start(self, ctx, m0_t, outs, stream, cell_t=None):
        """Sample 0 (row 0, mask m0_t) into window 0's outputs `outs`, which it zeroes first."""
        with self.torch.cuda.stream(stream):
            outs[0].zero_()
        self.t = 0
        self.launch(ctx, cell_t, m0_t, 0, outs[0], stream)

    def window(self, ctx, origins, yx1_t, m1_t, dt_days, outs, stream, cell_t=None):
        """TrackEngine.track's pass over one window: the next sample, added to the outputs start() has begun for
        window 0 and to zeroed outputs for the others."""
        self.t += 1
        if self.t > fsle.MAX_SAMPLES:
            raise ValueError("connect: at most %d samples in a run" % fsle.MAX_SAMPLES)
        if self.t > 1:
            with self.torch.cuda.stream(stream):
                outs[0].zero_()
        self.launch(ctx, cell_t, m1_t, self.t, outs[0], stream)

    def results(self, outs):
        """(the statistics of the window,) from its pinned outputs."""
        return (stats_dict(self.tau_edges, self.sample_days, self.nreg, outs[0].numpy()),)

    def state_dict(self):
        """The per-buoy state decoded: (nP,) status, src, prev, start and visited."""
        s = self.state.cpu().numpy().view(np.uint32).astype(np.int64)
        w = s[:, 1]
        return dict(status=(w >> 26) & 3, src=(w >> 16) & 31, prev=(w >> 21) & 31, start=w & 0xffff, visited=s[:, 0])


def RegionConnectivity(cells, masks, labels, sample_days, tau_edges=None, device=None):
    """Connectivity statistics of the buoys over the samples `cells` (S+1, nP, 2) i4 host cells [jT, iT] (bit 31 of jT,
    the discontinued flag, is ignored) with row masks `masks` (S+1, nP), sample_days days apart, between the regions
    of the label map `labels` (Nj, Ni) of the T-grid the cells index.  Host arrays in and out; computed on the GPU, one
    launch per sample.

    -> (state, stats).  state: dict of (nP,) i8 `status` (0 not started, 1 started, 2 ended), `src`, `prev`, `start`,
    `visited` after the last sample.  stats: the list of the S windows' dicts (stats_dict; window w holds the events
    of sample w+1, window 0 also the starts of sample 0, and the count snapshot of sample w+1)."""
    from .engine import _torch
    from . import config
    cl = np.asarray(cells)
    mk = np.asarray(masks)
    if cl.ndim != 3 or cl.shape[2] != 2 or cl.shape[0] < 2 or cl.shape[1] < 1 or mk.shape != cl.shape[:2]:
        raise ValueError("cells must have shape (S+1, nP, 2) with S >= 1, nP >= 1 and masks (S+1, nP), got %s and %s"
                         % (cl.shape, mk.shape))
    if cl.dtype.kind not in "iu":
        raise ValueError("cells must be integers, got dtype %s" % cl.dtype)
    S = cl.shape[0] - 1
    if S > fsle.MAX_SAMPLES:
        raise ValueError("at most %d samples after row 0" % fsle.MAX_SAMPLES)
    if not (np.isfinite(sample_days) and sample_days > 0):
        raise ValueError("sample_days must be finite and positive")
    lab = np.asarray(labels)
    if lab.ndim != 2:
        raise ValueError("labels must be a (Nj, Ni) map")
    lab, R = check_labels(labels, *lab.shape)
    torch = _torch()
    dev = torch.device("cuda", config.device if device is None else int(device))
    with torch.cuda.device(dev):
        plan = _Plan(torch, dev, lab, R, lab.shape[0], lab.shape[1], cl.shape[1], tau_edges, sample_days)
        stream = torch.cuda.current_stream(dev)
        g = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        c32 = lambda s: g((cl[s].astype(np.int64) & 0xffffffff).astype(np.uint32).view(np.int32), np.int32)
        outs = [plan.outputs() for _ in range(S)]
        plan.start(None, g(mk[0] != 0, np.int8), outs[0], stream, cell_t=c32(0))
        for s in range(1, S + 1):
            plan.window(None, None, None, g(mk[s] != 0, np.int8), sample_days, outs[s - 1], stream, cell_t=c32(s))
        stats = [plan.results((o[0].cpu(),))[0] for o in outs]
        return plan.state_dict(), stats
