"""SI3 T-cell fields sampled along the buoy trajectories: the ice each buoy travels with (concentration, thickness,
snow...) at every sampled row, from the host cells the engine already holds on the device.

Definitions (DESIGN.md section 15).  Row 0 is sampled with the first record of the run, row k+1 with record k (the
record whose velocities moved the buoy there); with every = n the rows 0, n, 2n, ...  A buoy's value is FillValue when
its row mask is 0.  interp "cell": the value of the buoy's host cell, which is the SI3 T-cell (an exact f4 copy).
interp "bilinear": the bilinear interpolation between the four T-points around the buoy, in f8 and without FMA,
land (tmask 0) and non-finite corners dropped and the rest renormalised, the cell value when none is left; rounded
once to f4.  A non-finite result is FillValue.  Computed on the device (csrc/st_sample.cu), bit-identical to
oracle/sample_ref.py.  No CPU fallback.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_c, check

__all__ = ["SampleFields", "MAX_SAMPLE_FIELDS", "SAMPLE_INTERP"]

FillValue = -9999.0
MAX_SAMPLE_FIELDS = 16
SAMPLE_INTERP = {"cell": 0, "bilinear": 1}


def check_interp(interp):
    if interp not in SAMPLE_INTERP:
        raise ValueError("interp must be 'cell' or 'bilinear', got %r" % (interp,))
    return SAMPLE_INTERP[interp]


def tpoints(tyx, Nj, Ni):
    """tyx = (Yt, Xt) (Nj,Ni) km -> (Nj*Ni, 2) f8 [y,x].

    The bilinear quad pick reads "west of S->N" and "south of W->E" from the sign of two orientation tests, which is
    right on a right-handed grid only: cross(T[j,i+1] - T[j,i], T[j+1,i] - T[j,i]) > 0, i eastward and j northward in
    the projected plane, as the step's anticlockwise F-cells are (and NEMO grids in the north polar stereographic
    projection).  A grid on which these crosses are not positive for most of the T-quads is refused; a few that are not
    (a fold, a degenerate land row) are accepted, and buoys in them get the clamped edge values of the opposite quad."""
    if tyx is None or len(tyx) != 2:
        raise ValueError("bilinear sampling needs tyx = (Yt, Xt), the T-points [km]")
    Yt, Xt = (np.asarray(a, np.float64) for a in tyx)
    if Yt.shape != (Nj, Ni) or Xt.shape != (Nj, Ni):
        raise ValueError("tyx: Yt and Xt must have shape (%d, %d)" % (Nj, Ni))
    cross = (Xt[:-1, 1:] - Xt[:-1, :-1]) * (Yt[1:, :-1] - Yt[:-1, :-1]) - \
        (Yt[:-1, 1:] - Yt[:-1, :-1]) * (Xt[1:, :-1] - Xt[:-1, :-1])
    if not np.count_nonzero(cross > 0) > cross.size // 2:
        raise ValueError("tyx: the T-points do not form a right-handed grid (i eastward, j northward in the projected "
                         "plane) on most of their quads; bilinear sampling needs one")
    return as_c(np.stack([Yt, Xt], -1).reshape(-1, 2), np.float64)


class _Plan:
    """Device side of one sampling setup of an engine: the interpolation mode and the T-points."""

    def __init__(self, eng, torch, dev, interp, tyx):
        self.L, self.eng = _lib.lib(), eng
        self.interp = interp
        self.mode = check_interp(interp)
        self.plane = eng.Nj * eng.Ni
        self.tyx_t = None
        if self.mode == 1:
            self.tyx_t = torch.from_numpy(tpoints(tyx, eng.Nj, eng.Ni)).to(dev)

    def launch(self, fields_ptr, nF, stride, yx_t, mask_t, out_ptr, stream):
        """st_sample_dev (async on `stream`): nF planes at fields_ptr, `stride` floats apart, into out_ptr (nF, nP)."""
        check(self.L.st_sample_dev(self.eng.h, int(nF), fields_ptr, int(stride),
                                   None if yx_t is None else yx_t.data_ptr(), mask_t.data_ptr(), self.mode,
                                   None if self.tyx_t is None else self.tyx_t.data_ptr(), out_ptr,
                                   C.c_void_p(stream.cuda_stream)), self.eng.h)


def SampleFields(eng, fields, mask=None, interp="cell", tyx=None, yx=None):
    """Sample the T-cell fields `fields` (nF,Nj,Ni) (or one (Nj,Ni) field) at the buoys of the engine `eng` as they
    stand: their host cells from its state, the row mask `mask` (nP,) (None: every buoy) and, for "bilinear", the
    positions yx (nP,2) f8 [y,x] km (None: the state's) and the T-points tyx = (Yt, Xt).  mask and yx are in the
    caller's buoy order (set_buoys), like the result.  Host arrays in and out; computed on the GPU.

    -> (nF, nP) f4 (or (nP,) for one field), FillValue where the buoy is masked or the value is not finite."""
    from .engine import _torch
    torch = _torch()
    F = np.asarray(fields)
    one = F.ndim == 2
    F = as_c(F[None] if one else F, np.float32)
    if F.ndim != 3 or F.shape[1:] != (eng.Nj, eng.Ni):
        raise ValueError("fields must have shape (nF, %d, %d) or (%d, %d)" % (eng.Nj, eng.Ni, eng.Nj, eng.Ni))
    nF, nP = F.shape[0], eng.nP
    if not 1 <= nF <= MAX_SAMPLE_FIELDS:
        raise ValueError("fields: 1..%d planes, got %d" % (MAX_SAMPLE_FIELDS, nF))
    perm = getattr(eng, "perm", None)
    if perm is None and getattr(eng, "perm_t", None) is not None:
        perm = eng.perm_t.cpu().numpy()
    order = (lambda a: a) if perm is None else (lambda a: a[perm])        # caller's order -> engine slots
    m = np.ones(nP, np.int8) if mask is None else (np.asarray(mask).reshape(-1) != 0).astype(np.int8)
    if m.shape != (nP,):
        raise ValueError("mask must have shape (%d,)" % nP)
    dev = torch.device("cuda", eng.device)
    with torch.cuda.device(dev):
        plan = _Plan(eng, torch, dev, interp, tyx)
        f_t = torch.from_numpy(F).to(dev)
        m_t = torch.from_numpy(np.ascontiguousarray(order(m))).to(dev)
        yx_t = None
        if yx is not None:
            y = as_c(yx, np.float64).reshape(-1, 2)
            if y.shape != (nP, 2):
                raise ValueError("yx must have shape (%d, 2)" % nP)
            yx_t = torch.from_numpy(np.ascontiguousarray(order(y))).to(dev)
        out = torch.empty((nF, nP), dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev)
        if nP:
            plan.launch(f_t.data_ptr(), nF, plan.plane, yx_t, m_t, out.data_ptr(), stream)
        r = out.cpu().numpy()
    if perm is not None:
        back = np.empty_like(r)
        back[:, perm] = r
        r = back
    return r[0] if one else r


class _SampleRun:
    """track(sample=...): the sampled rows of the record loop.

    Rows r = s * every, s = 0 .. nrec // every.  Row 0 is sampled on the compute stream after record 0 has been
    uploaded and before step 0, from the state handed to set_buoys and row 0's mask (_WindowRows.m0); row k+1 right
    after step k, before the step's event is recorded, so the record slot is read before it can be overwritten.
    `siconc` comes straight from plane 2 of the record slot; other names are read with get(k, name) inside the record
    loop's reader, only for sampled records, into a pinned double buffer of their own, and uploaded on the input
    stream.  Outputs (nF, nP) f4 go to the host on the output stream in a ring of 3 (ahead of the row copies of the
    same iteration) and reach the caller in its buoy order: sink(s, {name: (nP,) f4}), or with sink None arrays
    {name: (nsample, nP) f4} under "sample"."""

    NRING = 3

    def __init__(self, eng, torch, dev, spec, rows, nrec):
        names = list(spec.get("names") or [])
        if not names or len(set(names)) != len(names) or not all(isinstance(n, str) for n in names):
            raise ValueError("sample: names must be a non-empty list of distinct variable names")
        if len(names) > MAX_SAMPLE_FIELDS:
            raise ValueError("sample: at most %d fields" % MAX_SAMPLE_FIELDS)
        self.every = int(spec.get("every", 1))
        if nrec < 1:
            raise ValueError("sample: needs at least one record")
        if self.every < 1:
            raise ValueError("sample: every must be >= 1 record")
        self.extra = [n for n in names if n != "siconc"]
        self.get = spec.get("get")
        if self.extra and not callable(self.get):
            raise ValueError("sample: get(k, name) -> (Nj, Ni) is needed for %s" % self.extra)
        self.torch, self.eng, self.rows, self.sink = torch, eng, rows, spec.get("sink")
        self.plan = _Plan(eng, torch, dev, spec.get("interp", "cell"), spec.get("tyx"))
        self.order = (["siconc"] if "siconc" in names else []) + self.extra          # output rows on the device
        self.names = names
        nP, nF, nE, Nj, Ni = eng.nP, len(names), len(self.extra), eng.Nj, eng.Ni
        self.nsample = nrec // self.every + 1
        self.m0 = torch.from_numpy(rows.m0).to(dev)
        self.d_out = [torch.empty((nF, nP), dtype=torch.float32, device=dev) for _ in range(self.NRING)]
        self.h_out = [torch.empty((nF, nP), dtype=torch.float32).pin_memory() for _ in range(self.NRING)]
        self.h_ext = [torch.empty((nE, Nj, Ni), dtype=torch.float32).pin_memory() for _ in range(2)] if nE else None
        self.d_ext = [torch.empty((nE, Nj, Ni), dtype=torch.float32, device=dev) for _ in range(2)] if nE else None
        self.pending = []                                    # (s, iteration whose output event covers it)
        self.collected = {}
        if self.sink is None:
            self.kept = {n: np.empty((self.nsample, nP), np.float32) for n in names}
            self.collected = {"sample": self.kept}

    def wanted(self, k):
        """Record k is read by a sampled row: row 0 (k = 0) or row k+1."""
        return k == 0 or (k + 1) % self.every == 0

    def load(self, k):
        """The reader thread, record k: the extra fields into pinned buffer k % 2 (free once ev_in[k-2] is done)."""
        if not self.extra or not self.wanted(k):
            return
        h = self.h_ext[k % 2].numpy()
        for i, n in enumerate(self.extra):
            a = self.get(k, n)
            if isinstance(a, np.ma.MaskedArray):
                a = a.astype(np.float32).filled(np.nan)          # masked reads count as missing
            h[i] = a
            # a wrong shape raises in the assignment above

    def upload(self, k, s_in):
        if self.extra and self.wanted(k):
            with self.torch.cuda.stream(s_in):
                self.d_ext[k % 2].copy_(self.h_ext[k % 2], non_blocking=True)

    def row(self, r, k, slot, yx_t, mask_t, s_cmp):
        """Sample row r with record k (record slot `slot`) on s_cmp: yx_t the f8 row, or None for the state."""
        s = r // self.every
        out = self.d_out[s % self.NRING]
        off = 0
        if self.order[0] == "siconc":
            ic = self.eng.record_device_ptr(slot) + 2 * self.plan.plane * 4
            self.plan.launch(ic, 1, self.plan.plane, yx_t, mask_t, out.data_ptr(), s_cmp)
            off = 1
        if self.extra:
            d = self.d_ext[k % 2]
            self.plan.launch(d.data_ptr(), len(self.extra), self.plan.plane, yx_t, mask_t,
                             out.data_ptr() + off * out.shape[1] * 4, s_cmp)
        self.pending.append([s, k, False])

    def copy_out(self, k, s_out):
        """On s_out, ahead of iteration k's row copies: the samples queued since the last call."""
        with self.torch.cuda.stream(s_out):
            for p in self.pending:
                if not p[2]:
                    self.h_out[p[0] % self.NRING].copy_(self.d_out[p[0] % self.NRING], non_blocking=True)
                    p[1], p[2] = k, True

    def deliver(self, upto_row, ev_out):
        """Hand over every sample of a row <= upto_row (waits for its output event)."""
        while self.pending and self.pending[0][0] * self.every <= upto_row:
            s, k, _ = self.pending.pop(0)
            ev_out[k].synchronize()
            v = self.h_out[s % self.NRING].numpy()
            inv = self.rows.inv
            v = v.copy() if inv is None else v[:, inv]
            out = {n: v[self.order.index(n)] for n in self.names}
            if self.sink is None:
                for n in self.names:
                    self.kept[n][s] = out[n]
            else:
                self.sink(s, out)
