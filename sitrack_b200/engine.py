"""TrackEngine -- host-side owner of one GPU's share of the tracking run.

Python here is plumbing only (argument marshalling, CUDA streams/events and
pinned buffers through PyTorch); all arithmetic of the path happens in
libsitrack_b200.so.  One engine = one CUDA device = one process (rank).

Reference mapping (paths relative to stephanieleroux/sitrack):
  TrackEngine(...)        static grid + constants   si3_part_tracker.py:192-202, :31, :37
  .seed_locate(...)       SeedInit loop             sitrack/tracking.py:120-160
  .set_buoys(...)         state allocation          si3_part_tracker.py:324-344
  .step(...)              loop body                 si3_part_tracker.py:378-493
  .track(...)             record loop               si3_part_tracker.py:361-496
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_c, check, hptr

FillValue = -9999.0


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise _lib.SitrackCudaError("no CUDA device visible to PyTorch; sitrack_b200 has no CPU fallback")
    return torch


def _dptr(t):
    return None if t is None else t.data_ptr()


def _sptr(stream):
    if stream is None:
        return None
    return stream.cuda_stream


def _rows_f4(*outs):
    """True when the caller's row buffers are float32 (torch tensors or numpy arrays); mixing raises."""
    kinds = {str(o.dtype).replace("torch.", "") for o in outs if o is not None}
    if not kinds:
        return False
    if kinds == {"float32"}:
        return True
    if kinds == {"float64"}:
        return False
    raise TypeError("trajectory row buffers must be all float64 or all float32, got %s" % sorted(kinds))


class _DevMem:
    """__cuda_array_interface__ carrier so torch can view library-owned device memory."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def _tensor_from_ptr(torch, ptr, shape, dtype, itemsize, device):
    ts = {4: "<f4", 8: "<f8"}[itemsize]
    return torch.as_tensor(_DevMem(ptr, shape, ts), device=torch.device("cuda", device))


class TrackEngine:
    def __init__(self, Yf, Xf, Yu=None, Xu=None, Yv=None, Xv=None, tmask=None, uv_strategy=1,
                 rdt=3600.0, rmin_conc=0.1, device=0):
        if tmask is None:
            raise ValueError("tmask is required")
        self.L = _lib.lib()
        self.Nj, self.Ni = tmask.shape
        self.device = int(device)
        self.uv_strategy, self.rdt, self.rmin_conc = int(uv_strategy), float(rdt), float(rmin_conc)
        arrs = [None if a is None else as_c(a, np.float64) for a in (Yf, Xf, Yu, Xu, Yv, Xv)]
        for a in arrs:
            if a is not None and a.shape != (self.Nj, self.Ni):
                raise ValueError("grid arrays must all have shape (Nj,Ni)")
        tm = as_c(tmask, np.int8)
        self._tmask_host = tm
        h = C.c_void_p()
        check(self.L.st_create(C.byref(h), self.device, self.Nj, self.Ni, *[hptr(a) for a in arrs], hptr(tm),
                               self.uv_strategy, self.rdt, self.rmin_conc))
        self.h = h
        self.nP = 0
        self._nslots = 0
        self._has_locate = False

    # -- lifecycle ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self.L.st_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_kernel_variant(self, variant):
        """0 = 2 = k_advect_warp with the orientation filter (default), 3 without it, 1 = k_advect_step_v1
        (straightforward A/B reference), 4 = the certified two-kernel step; see include/sitrack_b200.h."""
        check(self.L.st_set_kernel_variant(self.h, int(variant)), self.h)

    # -- diagnostics of the certified fast path (csrc/st_cert.cuh) ----------------------------
    def cert_stats(self):
        """-> (cells admitted to the certified fast path, cells examined)."""
        a, e = C.c_int64(0), C.c_int64(0)
        check(self.L.st_cert_stats(self.h, C.byref(a), C.byref(e)), self.h)
        return a.value, e.value

    def cert_frames(self):
        """-> frames (Nj,Ni,8) f4 [oy ox a b c d es et], hin (Nj,Ni) f4, msep (Nj,Ni) f4 (hin = -1: never certified)."""
        fr = np.zeros((self.Nj, self.Ni, 8), np.float32)
        mw = np.zeros((self.Nj, self.Ni), np.uint32)
        check(self.L.st_cert_frames(self.h, hptr(fr), hptr(mw)), self.h)
        hin = (mw & np.uint32(0xffff0000)).view(np.float32)
        msep = (mw << np.uint32(16)).view(np.float32)
        return fr, hin, msep

    def selftest_cert(self, yx, cell, vel4):
        """flags (n,) u8 of st_selftest_cert: bit0 pick certified, bit1 stay certified, bit2/3 certified
        llum1/llvm1, bit4/5 the reference's, bit6 the reference's inside test of the reference's new position."""
        yx, cell, vel4 = as_c(yx, np.float64).reshape(-1, 2), as_c(cell, np.int32).reshape(-1, 2), as_c(vel4, np.float32).reshape(-1, 4)
        fl = np.zeros(yx.shape[0], np.uint8)
        check(self.L.st_selftest_cert(self.h, yx.shape[0], hptr(yx), hptr(cell), hptr(vel4), hptr(fl)), self.h)
        return fl

    # -- seeding -----------------------------------------------------------------------
    def set_locate_grid(self, latT, lonT, resKM=None):
        la, lo = as_c(latT, np.float64), as_c(lonT, np.float64)
        rk = None if resKM is None or np.shape(resKM) != (self.Nj, self.Ni) else as_c(resKM, np.float64)
        check(self.L.st_set_locate_grid(self.h, hptr(la), hptr(lo), hptr(rk)), self.h)
        self._has_locate = True
        self._loc = (la, lo, rk)                               # host copies: the near-tie re-check of seed_locate

    def seed_locate(self, SG, SC, ic0, recheck=True, stats=None):
        """-> (cell (nP,2) i4, nearest (nP,2) i4, keep (nP,) i1); SeedInit's loop on the device.

        recheck: seeds whose nearest point or acceptance the device decided by less than 1e-11 relative (CUDA's
        sin/cos/asin differ from numpy's in the last ulp) are re-evaluated here with numpy, i.e. with the reference's
        own arithmetic (locate.py:253-266, util.py:85-103); where that changes the nearest point, Survive and
        FindContainingCell are redone for the seed.  stats (a dict) receives the counts."""
        SG, SC = as_c(SG, np.float64), as_c(SC, np.float64)
        ic0 = as_c(ic0, np.float32)
        nP = SG.shape[0]
        cell = np.zeros((nP, 2), np.int32)
        near = np.zeros((nP, 2), np.int32)
        keep = np.zeros(nP, np.int8)
        if not recheck:
            check(self.L.st_seed_locate(self.h, nP, hptr(SG), hptr(SC), hptr(ic0), hptr(cell), hptr(near), hptr(keep)),
                  self.h)
            return cell, near, keep
        flag = np.zeros(nP, np.int8); first = np.zeros(nP, np.int32); second = np.zeros(nP, np.int32)
        check(self.L.st_seed_locate_ex(self.h, nP, hptr(SG), hptr(SC), hptr(ic0), hptr(cell), hptr(near), hptr(keep),
                                       hptr(flag), hptr(first), hptr(second)), self.h)
        idx = np.flatnonzero(flag)
        changed = 0
        if idx.size:
            from .locate import _recheck_nearest
            la, lo, rk = self._loc
            redo = []
            for p in idx:
                ji = _recheck_nearest(SG[p], int(first[p]), int(second[p]), la, lo, rk)
                if ji != (int(near[p, 0]), int(near[p, 1])):
                    near[p] = ji
                    redo.append(p)
            changed = len(redo)
            if redo:
                redo = np.array(redo)
                ok = near[redo, 0] >= 0
                keep[redo] = 0
                cell[redo] = 0
                r = redo[ok]
                if r.size:
                    from .tracking import SurviveBatch
                    alive = SurviveBatch(near[r], self._tmask_host, ic0.reshape(self.Nj, self.Ni)) == 0
                    c2, found = self.find_containing_cell(SC[r], near[r])
                    cell[r] = c2
                    keep[r] = (alive & found).astype(np.int8)
        if stats is not None:
            stats.update(flagged=int(idx.size), changed=changed)
        return cell, near, keep

    def seed_locate_dev(self, SG_t, SC_t, ic0_t, stream=None):
        """Device tensors in, device tensors out (async on `stream`)."""
        torch = _torch()
        nP = SG_t.shape[0]
        dev = SG_t.device
        cell = torch.empty((nP, 2), dtype=torch.int32, device=dev)
        near = torch.empty((nP, 2), dtype=torch.int32, device=dev)
        keep = torch.empty((nP,), dtype=torch.int8, device=dev)
        stream = stream or torch.cuda.current_stream(dev)
        check(self.L.st_seed_locate_dev(self.h, nP, _dptr(SG_t), _dptr(SC_t), _dptr(ic0_t), _dptr(cell),
                                        _dptr(near), _dptr(keep), _sptr(stream)), self.h)
        return cell, near, keep

    def seed_compact_dev(self, pos_t, cell_t, keep_t, stream=None):
        """(pos, cell) of the kept seeds, order kept (SeedInit's shrink, tracking.py:166-178), on the device."""
        torch = _torch()
        stream = stream or torch.cuda.current_stream(pos_t.device)
        nP = pos_t.shape[0]
        out_pos, out_cell = torch.empty_like(pos_t), torch.empty_like(cell_t)
        n = C.c_int64(0)
        check(self.L.st_seed_compact_dev(self.h, nP, _dptr(pos_t), _dptr(cell_t), _dptr(keep_t), _dptr(out_pos),
                                         _dptr(out_cell), C.byref(n), _sptr(stream)), self.h)
        return out_pos[:n.value], out_cell[:n.value]

    def nearest_point(self, latlon, rd_found_km=2.5, max_itr=10, brute=False):
        ll = as_c(latlon, np.float64).reshape(-1, 2)
        ji = np.zeros((ll.shape[0], 2), np.int32)
        d = np.zeros(ll.shape[0], np.float64)
        check(self.L.st_nearest_point(self.h, ll.shape[0], hptr(ll), rd_found_km, max_itr, int(brute),
                                      hptr(ji), hptr(d)), self.h)
        return ji, d

    def find_containing_cell(self, yx, ji_near):
        yx = as_c(yx, np.float64).reshape(-1, 2)
        jn = as_c(ji_near, np.int32).reshape(-1, 2)
        cell = np.zeros_like(jn)
        found = np.zeros(yx.shape[0], np.int8)
        check(self.L.st_find_containing_cell(self.h, yx.shape[0], hptr(yx), hptr(jn), hptr(cell), hptr(found)),
              self.h)
        return cell, found.astype(bool)

    # -- state -------------------------------------------------------------------------
    def set_buoys(self, pos, cell, rec_first=None, rec_last=None, sort=False):
        """sort=True stores the buoys in cell-major order (stable sort by host cell): a warp's 32 buoys then sit in
        neighbouring cells and its gathers touch a handful of lines instead of 32 (SURVEY section 7 "gather
        locality"; the reference keeps seed order, sitrack/tracking.py:166-178).  The permutation is `self.perm`
        (engine slot -> caller's index); track() in full-series mode and get_state() give results back in the
        caller's order, a `sink` receives rows in engine order."""
        pos, cell = as_c(pos, np.float64), as_c(cell, np.int32)
        rf = None if rec_first is None else as_c(rec_first, np.int32)
        rl = None if rec_last is None else as_c(rec_last, np.int32)
        self.perm = None
        self.perm_t = None
        if sort and pos.shape[0] > 1:
            perm = np.argsort(cell[:, 0].astype(np.int64) * self.Ni + cell[:, 1], kind="stable")
            pos, cell = as_c(pos[perm], np.float64), as_c(cell[perm], np.int32)
            rf = None if rf is None else as_c(rf[perm], np.int32)
            rl = None if rl is None else as_c(rl[perm], np.int32)
            self.perm = perm
        check(self.L.st_set_buoys(self.h, pos.shape[0], hptr(pos), hptr(cell), hptr(rf), hptr(rl)), self.h)
        self.nP = pos.shape[0]

    def set_buoys_dev(self, pos_t, cell_t, rec_first_t=None, rec_last_t=None, stream=None, sort=False):
        """Device tensors in.  sort=True: as set_buoys, the permutation stays on the device as `self.perm_t`."""
        torch = _torch()
        stream = stream or torch.cuda.current_stream(pos_t.device)
        self.perm = None
        self.perm_t = None
        if sort and pos_t.shape[0] > 1:
            with torch.cuda.stream(stream):
                key = cell_t[:, 0].to(torch.int64) * self.Ni + cell_t[:, 1].to(torch.int64)
                perm = torch.argsort(key, stable=True)
                pos_t, cell_t = pos_t[perm].contiguous(), cell_t[perm].contiguous()
                rec_first_t = None if rec_first_t is None else rec_first_t[perm].contiguous()
                rec_last_t = None if rec_last_t is None else rec_last_t[perm].contiguous()
            self.perm_t = perm
            self._sorted_keepalive = (pos_t, cell_t, rec_first_t, rec_last_t)   # until the async copy below has run
        check(self.L.st_set_buoys_dev(self.h, pos_t.shape[0], _dptr(pos_t), _dptr(cell_t), _dptr(rec_first_t),
                                      _dptr(rec_last_t), _sptr(stream)), self.h)
        self.nP = pos_t.shape[0]

    def get_state(self):
        pos = np.zeros((self.nP, 2), np.float64)
        cell = np.zeros((self.nP, 2), np.int32)
        alive = np.zeros(self.nP, np.int8)
        check(self.L.st_get_state(self.h, hptr(pos), hptr(cell), hptr(alive)), self.h)
        perm = getattr(self, "perm", None)
        if perm is not None:                                     # back to the caller's order
            out = [np.empty_like(a) for a in (pos, cell, alive)]
            for o, a in zip(out, (pos, cell, alive)):
                o[perm] = a
            return tuple(out)
        return pos, cell, alive

    def set_row_chain(self, on=True):
        """Row chaining (st_set_row_chain): the f8 yx row of a step is the position input of the next one, as
        xPosC[jt] is in the reference (si3_part_tracker.py:412,459-460); the state's own copy is not rewritten every
        record.  The caller keeps each row intact until the next step has run."""
        check(self.L.st_set_row_chain(self.h, 1 if on else 0), self.h)

    def sync_state(self, stream=None):
        """Bring the position state up to date after chained steps (async on `stream`)."""
        check(self.L.st_sync_state(self.h, _sptr(stream)), self.h)

    # -- records -----------------------------------------------------------------------
    def record_slots(self, n):
        check(self.L.st_record_slots(self.h, int(n)), self.h)
        self._nslots = max(self._nslots, int(n))

    def staging(self, slot):
        """numpy view (3,Nj,Ni) f4 of the slot's pinned host buffer: [u_ice, v_ice, siconc]."""
        p = C.c_void_p()
        check(self.L.st_record_host_buffer(self.h, slot, C.byref(p)), self.h)
        buf = (C.c_float * (3 * self.Nj * self.Ni)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.float32).reshape(3, self.Nj, self.Ni)

    def record_device_ptr(self, slot):
        p = C.c_void_p()
        check(self.L.st_record_device_buffer(self.h, slot, C.byref(p)), self.h)
        return p.value

    def submit_record(self, slot, stream=None):
        check(self.L.st_submit_record(self.h, slot, _sptr(stream)), self.h)

    def upload_record(self, slot, host_rec, stream=None):
        """Async H2D of a whole record from caller-owned host memory: a pinned torch tensor or
        a C-contiguous numpy array (3,Nj,Ni) f4 laid out [u_ice, v_ice, siconc]."""
        if hasattr(host_rec, "data_ptr"):
            if str(host_rec.dtype) != "torch.float32" or not host_rec.is_contiguous():
                raise TypeError("upload_record: the record must be a contiguous float32 tensor (3,Nj,Ni)")
            ptr = host_rec.data_ptr()
        else:
            if host_rec.dtype != np.float32 or not host_rec.flags["C_CONTIGUOUS"]:
                raise TypeError("upload_record: the record must be a C-contiguous float32 array (3,Nj,Ni); "
                                "the reference's f8 work arrays (si3_part_tracker.py:199-202) need .astype('f4')")
            ptr = hptr(host_rec)
        check(self.L.st_upload_record(self.h, slot, ptr, _sptr(stream)), self.h)

    # -- the step ----------------------------------------------------------------------
    def step(self, slot, jrec, out_yx=None, out_latlon=None, out_mask=None, n_alive=None, stream=None):
        """Enqueue one record for all buoys (async).  out_* are CUDA tensors (nP,2) f8 /
        (nP,) i1; n_alive a CUDA int64 scalar tensor that gets incremented.  float32 out_yx /
        out_latlon tensors select the file-dtype rows (st_step_f4; ncio.py:153-159)."""
        fn = self.L.st_step_f4 if _rows_f4(out_yx, out_latlon) else self.L.st_step
        check(fn(self.h, slot, int(jrec), _dptr(out_yx), _dptr(out_latlon), _dptr(out_mask),
                 _dptr(n_alive), _sptr(stream)), self.h)

    def step_ext(self, slot, jrec, scheme=1, interp=0, max_hops=1, out_yx=None, out_latlon=None, out_mask=None,
                 n_alive=None, stream=None):
        """st_step with optional physics beyond the reference: scheme 1|2|4 (Euler, midpoint RK2, RK4),
        interp 0|1 (the reference's face pick, C-grid linear), max_hops cell boundaries per step."""
        check(self.L.st_step_ext(self.h, slot, int(jrec), int(scheme), int(interp), int(max_hops), _dptr(out_yx),
                                 _dptr(out_latlon), _dptr(out_mask), _dptr(n_alive), _sptr(stream)), self.h)

    def step_multi(self, rec_stack, jrec0, out_yx=None, out_latlon=None, out_mask=None, n_alive=None,
                   stream=None):
        """rec_stack: CUDA tensor (nrec,3,Nj,Ni) f4; outputs (nrec,nP,2)/(nrec,nP); one launch."""
        nrec = rec_stack.shape[0]
        assert rec_stack.is_contiguous() and tuple(rec_stack.shape[1:]) == (3, self.Nj, self.Ni)
        fn = self.L.st_step_multi_f4 if _rows_f4(out_yx, out_latlon) else self.L.st_step_multi
        check(fn(self.h, _dptr(rec_stack), 3 * self.Nj * self.Ni, nrec, int(jrec0),
                 _dptr(out_yx), _dptr(out_latlon), _dptr(out_mask), self.nP,
                 _dptr(n_alive), _sptr(stream)), self.h)

    def track_record_host(self, jrec, u, v, ic, out_yx=None, out_latlon=None, out_mask=None, want_alive=True):
        """Synchronous host-buffer form of one loop iteration (H2D + step + D2H).  float32 out_yx /
        out_latlon arrays select the file-dtype rows (ncio.py:153-159)."""
        na = C.c_int64(0)
        fn = self.L.st_track_record_host_f4 if _rows_f4(out_yx, out_latlon) else self.L.st_track_record_host
        # the fields are f4 like the netCDF variables; the reference's f8 work arrays (si3_part_tracker.py:199-202)
        # hold exactly those values, so the cast back is lossless
        u, v, ic = as_c(u, np.float32), as_c(v, np.float32), as_c(ic, np.float32)
        check(fn(self.h, int(jrec), hptr(u), hptr(v), hptr(ic), hptr(out_yx),
                 hptr(out_latlon), hptr(out_mask), C.byref(na) if want_alive else None),
              self.h)
        return na.value

    # -- fused all-gather of positions over peer memory (multi-GPU) ----------------------------------
    def gather_create(self, rank, world, nP_total, offset, f4=False, nbuf=2):
        """Allocate this rank's gathered block; returns its 64-byte CUDA IPC handle (bytes)."""
        h = (C.c_ubyte * 64)()
        check(self.L.st_gather_create(self.h, int(rank), int(world), int(nP_total), int(offset), int(bool(f4)),
                                      int(nbuf), C.cast(h, C.c_void_p)), self.h)
        self._ga = dict(rank=rank, world=world, nP_total=int(nP_total), f4=bool(f4), nbuf=int(nbuf))
        return bytes(h)

    def gather_connect_ipc(self, handles):
        """handles: world x 64 bytes in rank order (other processes' gather_create results)."""
        blob = b"".join(handles) if not isinstance(handles, (bytes, bytearray)) else bytes(handles)
        assert len(blob) == 64 * self._ga["world"]
        buf = C.create_string_buffer(blob, len(blob))
        check(self.L.st_gather_connect_ipc(self.h, C.cast(buf, C.c_void_p)), self.h)

    def gather_block(self):
        p, n = C.c_void_p(), C.c_int64()
        check(self.L.st_gather_block(self.h, C.byref(p), C.byref(n)), self.h)
        return p.value, n.value

    def gather_connect_ptrs(self, blocks):
        """blocks: device pointers of every rank's block (ranks living in this process)."""
        arr = (C.c_void_p * len(blocks))(*blocks)
        check(self.L.st_gather_connect_ptrs(self.h, arr), self.h)

    def gather_buffer(self, buf):
        """The gathered (nP_total,2) array of buffer `buf` as a CUDA tensor view (f8 or f4)."""
        torch = _torch()
        p = C.c_void_p()
        check(self.L.st_gather_buffer(self.h, int(buf), C.byref(p)), self.h)
        g = self._ga
        dt, isz = (torch.float32, 4) if g["f4"] else (torch.float64, 8)
        return _tensor_from_ptr(torch, p.value, (g["nP_total"], 2), dt, isz, self.device)

    def step_gather(self, slot, jrec, buf, seq, out_latlon=None, out_mask=None, n_alive=None, stream=None):
        """st_step whose yx row lands in buffer `buf` of EVERY rank (stores over NVLink from inside the
        step kernel); seq = 1, 2, 3, ... per record."""
        check(self.L.st_step_gather(self.h, int(slot), int(jrec), int(buf), int(seq), _dptr(out_latlon),
                                    _dptr(out_mask), _dptr(n_alive), _sptr(stream)), self.h)

    def gather_wait(self, seq, stream=None):
        check(self.L.st_gather_wait(self.h, int(seq), _sptr(stream)), self.h)

    def gather_ack(self, seq, stream=None):
        check(self.L.st_gather_ack(self.h, int(seq), _sptr(stream)), self.h)

    def gather_timed_out(self):
        v = C.c_int(0)
        check(self.L.st_gather_timed_out(self.h, C.byref(v)), self.h)
        return bool(v.value)

    def gather_set_mode(self, mode):
        """0 per-thread peer stores (default), 1 copy engines, 2 bulk peer stores; see include/sitrack_b200.h."""
        check(self.L.st_gather_set_mode(self.h, int(mode)), self.h)

    def gather_destroy(self):
        check(self.L.st_gather_destroy(self.h), self.h)

    # -- the record loop ---------------------------------------------------------------
    def track(self, records, nrec, kstrt=0, pos0=None, posG0=None, rec_first=None, want_latlon=True,
              sink=None, chunk=None, verbose=None, row_dtype="f8", physics=None, deform=None, dispersion=None,
              fsle=None, sample=None):
        """The record loop (si3_part_tracker.py:361-496), pipelined.

        records: callable k -> (u, v, ic) arrays (Nj,Ni) for record index k (0-based
                 within the run; file record = k + kstrt), or an array (nrec,3,Nj,Ni) /
                 tuple of three (nrec,Nj,Ni) arrays.
        Pipeline per record k: host fills the pinned staging slot k%2 || copy stream H2D ||
        compute stream k_advect_step || output stream D2H of trajectory row k+1 into
        pinned host rows.  With sink=None the full (nrec+1,nP,..) series is returned
        (rows 0 from pos0/posG0); otherwise sink(jt, yx, latlon, mask) is called with
        pinned row views that are only valid during the call.
        physics = dict(scheme=, interp=, max_hops=) switches every record to st_step_ext (f8 rows only).
        row_dtype "f4" moves the rows in the output file's dtype (ncio.py:153-159: 17 B per buoy
        instead of 33 B over PCIe, values = the f8 rows cast to f4); the state stays f8 on the device.
        deform = dict(tri=(nT,3) triangles of buoys in the caller's order (anticlockwise, e.g. TriangulateCloud),
        every=n, sink=callable or None): strain rates of the triangles (sitrack_b200.deform) over the windows of
        rows [w*n, (w+1)*n], computed on the device from the f8 positions as each window closes (a trailing partial
        window is dropped; row 0 is the state handed to set_buoys, masked like the returned series' row 0).
        sink(w, out) receives a dict of (nT,) f4 arrays in the caller's triangle order; with sink None the
        list of them is returned under "deform".  Not with the chunked season path (chunk > 1, sink=None).
        deform may also hold scales=BoxHierarchy (built on the same tri and buoys) and scale_sink=callable or None:
        as each window closes the deformation of its boxes is reduced on the device to per-scale statistics
        (sitrack_b200.deform_scales), and only those reach the host: scale_sink(w, stats), or with scale_sink None
        the list of them under "deform_scales".  They do not depend on the order the buoys are stored in.
        deform may also hold grid=EulerianGrid and grid_sink=callable or None, with or without scales: as each window
        closes its triangles are binned into the grid's fixed cells by their mid-time centroid and coarse-grained on
        the device (sitrack_b200.deform_grid); only the fields and statistics reach the host: grid_sink(w, fields,
        stats), or with grid_sink None the list of (fields, stats) under "deform_grid".  They do not depend on the
        order the buoys are stored in either.
        dispersion = dict(pairs=(nQ,2) buoy pairs in the caller's order (sitrack_b200.dispersion: MeshPairs,
        SeparationPairs), every=n, lags=m (1..MAX_LAGS), r_edges=None, bins=None, sink=callable or None), independent of
        `deform` and combinable with it: the rows w*n are origins, kept on the device in a ring of min(m, windows) f8
        rows and masks (17 B per buoy each); as window w closes, the pairs' dispersion between origin row (w+1-l)*n and
        row (w+1)*n is reduced on the device for lags l = 1 .. min(m, w+1) in one launch, and only the statistics reach
        the host: sink(w, stats), or with sink None the list of them under "dispersion".  They do not depend on the
        order the buoys are stored in.  Not with the chunked season path either.
        fsle = dict(pairs=(nQ,2) buoy pairs in the caller's order, every=n, deltas=None, tau_edges=None, sink=callable or
        None), independent of `deform` and `dispersion` and combinable with both: the rows s*n are the samples of the
        pairs' finite-size Lyapunov exponents (sitrack_b200.fsle); each pair's first-passage state {level, anchor}
        stays on the device for the whole run and is updated at every sample, and only each window's integer
        statistics (the events of sample w+1, window 0 also those of row 0) reach the host: sink(w, stats), or with
        sink None the list of them under "fsle".  They do not depend on the order the buoys are stored in.  At most
        MAX_SAMPLES windows; not with the chunked season path either.
        sample = dict(names=[...], get=callable(k, name) -> (Nj,Ni) or None, every=n, interp="cell"|"bilinear",
        tyx=(Yt, Xt), sink=callable or None), combinable with all of the above: SI3 T-cell fields sampled along the
        trajectories on the device (sitrack_b200.sample, DESIGN.md section 15) at rows 0, n, 2n, ...; row 0 with record
        0, row k+1 with record k.  "siconc" is read from the record itself; every other name with get(k, name), only
        for the records that are sampled.  sink(s, {name: (nP,) f4}) in the caller's buoy order (called before the
        row sink of the same row), or with sink None {name: (nsample, nP) f4} under "sample".  "bilinear" needs tyx,
        the T-points [km].  Not with the chunked season path either.
        """
        torch = _torch()
        dev = torch.device("cuda", self.device)
        nP = self.nP
        get = _record_getter(records)
        perm = getattr(self, "perm", None)
        if perm is not None and chunk and chunk > 1 and sink is None:
            raise ValueError("the chunked season path keeps the caller's order: use set_buoys(sort=False) with it")
        if row_dtype not in ("f8", "f4"):
            raise ValueError("row_dtype must be 'f8' or 'f4'")
        rdt = torch.float32 if row_dtype == "f4" else torch.float64
        if physics:
            if row_dtype != "f8":
                raise ValueError("physics modes write f8 rows")
            chunk = None
        if chunk and chunk > 1 and sink is None:
            if deform is not None or dispersion is not None or fsle is not None or sample is not None:
                raise ValueError("deform, dispersion, fsle and sample run on the streaming record loop: not with chunk > 1 "
                                 "and sink=None")
            return self._track_chunked(get, nrec, kstrt, pos0, posG0, rec_first, want_latlon, int(chunk), rdt)
        specs = ((_deform_run, deform), (_dispersion_run, dispersion), (_fsle_run, fsle))
        wrows = None if all(spec is None for _, spec in specs) and sample is None else \
            _WindowRows(self, torch, rec_first, kstrt, row_f4=rdt == torch.float32)
        runs = [run(self, torch, dev, spec, wrows, nrec) for run, spec in specs if spec is not None]
        smp = None
        if sample is not None:
            from .sample import _SampleRun
            smp = _SampleRun(self, torch, dev, sample, wrows, nrec)
        self.record_slots(2)
        stg = [self.staging(0), self.staging(1)]
        s_in, s_cmp, s_out = (torch.cuda.Stream(dev) for _ in range(3))
        NB = 2
        d_yx = [torch.empty((nP, 2), dtype=rdt, device=dev) for _ in range(NB)]
        d_ll = [torch.empty((nP, 2), dtype=rdt, device=dev) for _ in range(NB)] if want_latlon else [None] * NB
        d_mk = [torch.empty((nP,), dtype=torch.int8, device=dev) for _ in range(NB)]
        d_na = torch.zeros((nrec,), dtype=torch.int64, device=dev)
        s_cmp.wait_stream(torch.cuda.current_stream(dev))      # the zero fill above ran on torch's current stream
        keep = sink is None
        if keep:
            posC = torch.full((nrec + 1, nP, 2), FillValue, dtype=rdt).pin_memory()
            posG = torch.full((nrec + 1, nP, 2), FillValue, dtype=rdt).pin_memory()
            mask = torch.zeros((nrec + 1, nP), dtype=torch.int8).pin_memory()
            rows = lambda k: (posC[k + 1], posG[k + 1] if want_latlon else None, mask[k + 1])
        else:
            h_yx = [torch.empty((nP, 2), dtype=rdt).pin_memory() for _ in range(NB)]
            h_ll = [torch.empty((nP, 2), dtype=rdt).pin_memory() for _ in range(NB)]
            h_mk = [torch.empty((nP,), dtype=torch.int8).pin_memory() for _ in range(NB)]
            rows = lambda k: (h_yx[k % NB], h_ll[k % NB] if want_latlon else None, h_mk[k % NB])
        ev_in = [None] * nrec
        ev_step = [None] * nrec
        ev_out = [None] * nrec

        def drain(k):
            ev_out[k].synchronize()
            if smp is not None:
                smp.deliver(k + 1, ev_out)                 # the samples of rows <= k+1 before the row sink of k
            if not keep:
                y, l, m = rows(k)
                sink(k, y.numpy(), None if l is None else l.numpy(), m.numpy())

        # reader thread (SURVEY 8b "threading"): record k+1 is read and converted into its pinned staging slot while
        # the main thread queues the GPU work of record k (netCDF4 reads and numpy copies release the GIL)
        from concurrent.futures import ThreadPoolExecutor

        def load(k):
            b = k % 2
            if k >= 2:
                ev_in[k - 2].synchronize()                 # staging slot b has left the host
            u, v, ic = get(k)
            stg[b][0], stg[b][1], stg[b][2] = u, v, ic     # f4 copy into pinned memory
            if smp is not None:
                smp.load(k)                                # the extra fields of a sampled record, same reader
        pool = ThreadPoolExecutor(1)
        nxt = pool.submit(load, 0) if nrec > 0 else None
        # f8 rows: the row of record k is the position input of record k+1 (st_set_row_chain); both row buffers
        # live until the chain is closed below
        chain = rdt == torch.float64 and not physics
        if chain:
            self.set_row_chain(True)
        try:
            for k in range(nrec):
                b = k % 2
                nxt.result()
                if k + 1 < nrec:
                    nxt = pool.submit(load, k + 1)             # waits for ev_in[k-1], recorded below before it can matter
                if k >= 2:
                    s_in.wait_event(ev_step[k - 2])            # device slot b no longer read
                self.submit_record(b, s_in)
                if smp is not None:
                    smp.upload(k, s_in)
                ev_in[k] = torch.cuda.Event(); ev_in[k].record(s_in)
                s_cmp.wait_event(ev_in[k])
                if k >= NB:
                    s_cmp.wait_event(ev_out[k - NB])           # device out buffer b drained
                if smp is not None and k == 0:
                    smp.row(0, 0, b, None, smp.m0, s_cmp)     # row 0: the state handed to set_buoys, record 0
                if physics:
                    self.step_ext(b, k + kstrt, physics.get("scheme", 1), physics.get("interp", 0),
                                  physics.get("max_hops", 1), d_yx[b], d_ll[b], d_mk[b], d_na[k:k + 1], s_cmp)
                else:
                    self.step(b, k + kstrt, d_yx[b], d_ll[b], d_mk[b], d_na[k:k + 1], s_cmp)
                if smp is not None and (k + 1) % smp.every == 0:
                    # row k+1 with record k, before ev_step[k]: the slot is not overwritten before this has read it
                    smp.row(k + 1, k, b, d_yx[b] if rdt == torch.float64 else None, d_mk[b], s_cmp)
                ev_step[k] = torch.cuda.Event(); ev_step[k].record(s_cmp)
                s_out.wait_event(ev_step[k])
                if not keep and k >= NB:
                    drain(k - NB)                              # pinned row buffer b is free again
                elif keep and smp is not None and k >= NB:
                    smp.deliver(k - 1, ev_out)                 # as drain(k - NB) would: the sample ring is free again
                if smp is not None:
                    smp.copy_out(k, s_out)
                y, l, m = rows(k)
                with torch.cuda.stream(s_out):
                    y.copy_(d_yx[b], non_blocking=True)
                    if want_latlon:
                        l.copy_(d_ll[b], non_blocking=True)
                    m.copy_(d_mk[b], non_blocking=True)
                ev_out[k] = torch.cuda.Event(); ev_out[k].record(s_out)
                for run in runs:
                    run.after_step(k, d_yx[b], d_mk[b], s_cmp, s_out)
            for k in range(max(0, nrec - NB), nrec):
                if keep:
                    ev_out[k].synchronize()
                else:
                    drain(k)
            for run in runs:
                run.finish()
            if smp is not None:
                smp.deliver(nrec, ev_out)
        finally:
            if chain:
                self.set_row_chain(False)                  # state up to date again (synchronises)
        torch.cuda.synchronize(dev)
        pool.shutdown()
        n_alive = d_na.cpu().numpy()
        extra = {}
        for run in runs:
            extra.update(run.collected)
        if smp is not None:
            extra.update(smp.collected)
        if not keep:
            return dict(n_alive=n_alive, **extra)
        posC, posG, mask = posC.numpy(), posG.numpy(), mask.numpy()
        if perm is not None:                                # engine order -> the caller's order
            inv = np.empty_like(perm); inv[perm] = np.arange(perm.size)
            posC, posG, mask = posC[:, inv], posG[:, inv], mask[:, inv]
        _finish_rows(posC, posG, mask, pos0, posG0, rec_first, kstrt)
        return dict(posC=posC, posG=posG, mask=mask, n_alive=n_alive, **extra)


class _WindowRows:
    """What the per-window passes over the trajectory rows share: the buoy permutation of the engine (set_buoys or
    set_buoys_dev with sort=True), row 0's mask in engine order (the state handed to set_buoys, masked like the returned
    series' row 0: rec_first == kstrt) and the f8 positions of a row.  Positions are f8: with f8 rows the row itself
    (read only, so row chaining is unaffected), with f4 rows the device state (steps with f4 rows do not chain, so it
    is current after every step)."""

    def __init__(self, eng, torch, rec_first, kstrt, row_f4):
        nP = eng.nP
        self.row_f4 = row_f4
        perm = eng.perm
        if perm is None and getattr(eng, "perm_t", None) is not None:      # set_buoys_dev(sort=True)
            perm = eng.perm_t.cpu().numpy()
        m0 = np.ones(nP, np.int8) if rec_first is None else (np.asarray(rec_first) - kstrt == 0).astype(np.int8)
        self.inv = None
        if perm is not None:                                                # caller's order -> engine slots
            if perm.shape != (nP,):
                raise ValueError("the engine's buoy permutation does not match its %d buoys" % nP)
            self.inv = np.empty_like(perm); self.inv[perm] = np.arange(perm.size)
            m0 = m0[perm]
        self.m0 = m0
        p = C.c_void_p()
        check(eng.L.st_state_device_ptrs(eng.h, C.byref(p), None, None), eng.h)
        self.state_pos = _tensor_from_ptr(torch, p.value, (nP, 2), torch.float64, 8, eng.device)

    def slots(self, idx):
        """Buoy indices in the caller's order -> engine slots (same shape, i4)."""
        return idx if self.inv is None else self.inv[idx].astype(np.int32)

    def yx(self, yx_row):
        """The f8 positions of the row a step has just written to yx_row."""
        return self.state_pos if self.row_f4 else yx_row


def _window_every(spec, what):
    """spec["every"]: records per window, >= 1."""
    every = int(spec["every"])
    if every < 1:
        raise ValueError("%s: every must be >= 1 record" % what)
    return every


def _deform_run(eng, torch, dev, spec, rows, nrec):
    """track(deform=...): triangles, then the box hierarchy (`scales`), then the Eulerian grid (`grid`), over the
    window's anchor row and its closing row.

    Triangles are mapped into engine order (set_buoys sort=True) and sorted once by their smallest vertex; the outputs
    go back to the caller's triangle order on the host.  The hierarchy keeps its own triangle order and the grid the
    caller's (both mapped to engine slots only), so neither's sums depend on `perm`."""
    from . import deform as D
    every = _window_every(spec, "deform")
    nP = eng.nP
    tri = rows.slots(D.check_mesh(spec["tri"], nP))
    passes = [("deform", spec.get("sink"), D._Plan(torch, dev, tri))]
    H = spec.get("scales")
    if H is not None:
        from . import deform_scales as DS
        if not isinstance(H, DS.BoxHierarchy) or not H.matches(spec["tri"], nP):
            raise ValueError("deform: scales must be a BoxHierarchy built on the same mesh (tri) and %d buoys" % nP)
        passes.append(("deform_scales", spec.get("scale_sink"), DS._DevicePlan(torch, dev, H, tri)))
    G = spec.get("grid")
    if G is not None:
        from . import deform_grid as DG
        if not isinstance(G, DG.EulerianGrid):
            raise ValueError("deform: grid must be an EulerianGrid")
        passes.append(("deform_grid", spec.get("grid_sink"), DG._GridPlan(torch, dev, G, tri)))
    return _WindowRun(eng, torch, dev, rows, every, nrec, 1, passes)


def _dispersion_run(eng, torch, dev, spec, rows, nrec):
    """track(dispersion=...): every active lag in one pass.  Pairs are mapped to engine slots without reordering
    them, so the sums do not depend on `perm`."""
    from . import dispersion as P
    every = _window_every(spec, "dispersion")
    lags = P.check_lags(spec["lags"])
    pairs = P.check_pairs(spec["pairs"], eng.nP)
    plan = P._Plan(torch, dev, rows.slots(pairs), lags, spec.get("r_edges"), spec.get("bins"),
                   dt_days=every * eng.rdt / 86400.0)
    return _WindowRun(eng, torch, dev, rows, every, nrec, lags, [("dispersion", spec.get("sink"), plan)])


def _fsle_run(eng, torch, dev, spec, rows, nrec):
    """track(fsle=...): one sample per window on the one-slot ring (row 0 is read in window 0 only).  Pairs are mapped
    to engine slots without reordering them, so the state stays in the caller's pair order."""
    from . import fsle as F
    from .dispersion import check_pairs
    every = _window_every(spec, "fsle")
    if nrec // every > F.MAX_SAMPLES:
        raise ValueError("fsle: %d windows, more than the %d samples a run may have" % (nrec // every, F.MAX_SAMPLES))
    pairs = check_pairs(spec["pairs"], eng.nP)
    plan = F._Plan(torch, dev, rows.slots(pairs), spec.get("deltas"), spec.get("tau_edges"),
                   sample_days=every * eng.rdt / 86400.0)
    return _WindowRun(eng, torch, dev, rows, every, nrec, 1, [("fsle", spec.get("sink"), plan)])


class _WindowRun:
    """The windows of one analysis of track(): a ring of origin rows on the device, its passes when a window closes,
    their outputs to the host on the output stream.

    passes: [(result key, sink or None, plan)]; a plan has outputs(pin), window(ctx, origins, yx1, m1, dt_days, outs,
    stream) and results(host outs) -> the sink's arguments after the window index.  Origin row o (= row o*every)
    lives in ring slot o % nslot, nslot = min(lags, windows) (row 0 in slot 0, as _WindowRows gives it).  When window
    w closes every pass reads the origins w+1-l, l = 1 .. min(lags, w+1), on the compute stream; only after them is
    the closing row, origin w+1, copied into slot (w+1) % nslot, the slot of origin w+1-lags that they have just read
    for the last time (no slot index reaches nslot < lags; origins 0 .. windows-1 are the only ones read).  Outputs
    are double-buffered: window w's reach the sinks, or the lists under their keys in `collected`, when window w+2
    closes or at finish()."""

    def __init__(self, eng, torch, dev, rows, every, nrec, lags, passes):
        self.ctx, self.torch, self.rows, self.passes = eng.h, torch, rows, passes
        self.every, self.lags = every, lags
        self.dt = every * eng.rdt / 86400.0
        self.nwin = nrec // every
        nslot = max(1, min(lags, self.nwin))
        nP = eng.nP
        # slot 0: row 0 (on torch's current stream; track's streams wait for it)
        self.r_yx = [rows.state_pos.clone()] + [torch.empty((nP, 2), dtype=torch.float64, device=dev)
                                                 for _ in range(nslot - 1)]
        self.r_mk = [torch.from_numpy(rows.m0).to(dev)] + [torch.empty((nP,), dtype=torch.int8, device=dev)
                                                           for _ in range(nslot - 1)]
        self.d_out = [[plan.outputs() for _, _, plan in passes] for _ in range(2)]
        self.h_out = [[plan.outputs(pin=True) for _, _, plan in passes] for _ in range(2)]
        self.collected = {key: [] for key, sink, _ in passes if sink is None}
        self.ev_out = []
        self.drained = 0

    def after_step(self, k, yx_row, mk_row, s_cmp, s_out):
        """Step k has been queued on s_cmp: row k+1 closes window w when k+1 = (w+1)*every."""
        if (k + 1) % self.every:
            return
        torch, w, n = self.torch, (k + 1) // self.every - 1, len(self.r_yx)
        b = w % 2
        if w >= 2:
            s_cmp.wait_event(self.ev_out[w - 2])                   # d_out[b] has reached the host
        yx = self.rows.yx(yx_row)
        origins = [(self.r_yx[(w + 1 - l) % n], self.r_mk[(w + 1 - l) % n], l)
                   for l in range(1, min(self.lags, w + 1) + 1)]
        for (_, _, plan), outs in zip(self.passes, self.d_out[b]):
            plan.window(self.ctx, origins, yx, mk_row, self.dt, outs, s_cmp)
        if w + 1 < self.nwin:
            with torch.cuda.stream(s_cmp):                          # after the passes that read the slot last
                self.r_yx[(w + 1) % n].copy_(yx)
                self.r_mk[(w + 1) % n].copy_(mk_row)
        ev = torch.cuda.Event(); ev.record(s_cmp)
        if w >= 2:
            self._drain(w - 2)                                      # h_out[b] is free again
        s_out.wait_event(ev)
        with torch.cuda.stream(s_out):
            for hs, ds in zip(self.h_out[b], self.d_out[b]):
                for h, d in zip(hs, ds):
                    h.copy_(d, non_blocking=True)
        self.ev_out.append(torch.cuda.Event()); self.ev_out[w].record(s_out)

    def _drain(self, w):
        self.ev_out[w].synchronize()
        for (key, sink, plan), h in zip(self.passes, self.h_out[w % 2]):
            r = plan.results(h)
            if sink is None:
                self.collected[key].append(r[0] if len(r) == 1 else r)
            else:
                sink(w, *r)
        self.drained = w + 1

    def finish(self):
        for w in range(self.drained, len(self.ev_out)):
            self._drain(w)


def _finish_rows(posC, posG, mask, pos0, posG0, rec_first, kstrt):
    """Row 0 of the series is the seed (si3_part_tracker.py:335-344)."""
    if pos0 is None:
        return
    if rec_first is None:
        posC[0] = pos0; mask[0] = 1
        if posG0 is not None:
            posG[0] = posG0
    else:
        k0 = np.asarray(rec_first) - kstrt
        sel = np.flatnonzero(k0 == 0)
        posC[0, sel] = np.asarray(pos0)[sel]; mask[0, sel] = 1
        if posG0 is not None:
            posG[0, sel] = np.asarray(posG0)[sel]


def _track_chunked(self, get, nrec, kstrt, pos0, posG0, rec_first, want_latlon, chunk, rdt=None):
    """Season path for small clouds: `chunk` records at a time are staged into HBM and advanced by
    ONE launch of k_advect_multi (each thread runs its buoy through the whole chunk), instead of
    one launch per record.  Host fill of chunk c+1 || H2D || compute of chunk c || D2H of its rows."""
    torch = _torch()
    dev = torch.device("cuda", self.device)
    nP, Nj, Ni = self.nP, self.Nj, self.Ni
    s_in, s_cmp, s_out = (torch.cuda.Stream(dev) for _ in range(3))
    rdt = rdt or torch.float64
    h_rec = [torch.empty((chunk, 3, Nj, Ni), dtype=torch.float32).pin_memory() for _ in range(2)]
    d_rec = [torch.empty((chunk, 3, Nj, Ni), dtype=torch.float32, device=dev) for _ in range(2)]
    d_yx = [torch.empty((chunk, nP, 2), dtype=rdt, device=dev) for _ in range(2)]
    d_ll = [torch.empty((chunk, nP, 2), dtype=rdt, device=dev) for _ in range(2)] if want_latlon else [None, None]
    d_mk = [torch.empty((chunk, nP), dtype=torch.int8, device=dev) for _ in range(2)]
    d_na = torch.zeros((nrec,), dtype=torch.int64, device=dev)
    s_cmp.wait_stream(torch.cuda.current_stream(dev))          # the zero fill above ran on torch's current stream
    posC = torch.full((nrec + 1, nP, 2), FillValue, dtype=rdt).pin_memory()
    posG = torch.full((nrec + 1, nP, 2), FillValue, dtype=rdt).pin_memory()
    mask = torch.zeros((nrec + 1, nP), dtype=torch.int8).pin_memory()
    nch = (nrec + chunk - 1) // chunk
    ev_in, ev_cmp, ev_out = [None] * nch, [None] * nch, [None] * nch
    for c in range(nch):
        b = c % 2
        k0, n = c * chunk, min(chunk, nrec - c * chunk)
        if c >= 2:
            ev_in[c - 2].synchronize()                      # pinned stack b has left the host
        hv = h_rec[b].numpy()
        for k in range(n):
            u, v, ic = get(k0 + k)
            hv[k, 0], hv[k, 1], hv[k, 2] = u, v, ic
        if c >= 2:
            s_in.wait_event(ev_cmp[c - 2])                  # device stack b no longer read
        with torch.cuda.stream(s_in):
            d_rec[b][:n].copy_(h_rec[b][:n], non_blocking=True)
        ev_in[c] = torch.cuda.Event(); ev_in[c].record(s_in)
        s_cmp.wait_event(ev_in[c])
        if c >= 2:
            s_cmp.wait_event(ev_out[c - 2])                 # row buffers b drained
        self.step_multi(d_rec[b][:n], k0 + kstrt, d_yx[b], d_ll[b], d_mk[b], d_na[k0:k0 + n], s_cmp)
        ev_cmp[c] = torch.cuda.Event(); ev_cmp[c].record(s_cmp)
        s_out.wait_event(ev_cmp[c])
        with torch.cuda.stream(s_out):
            posC[k0 + 1:k0 + 1 + n].copy_(d_yx[b][:n], non_blocking=True)
            if want_latlon:
                posG[k0 + 1:k0 + 1 + n].copy_(d_ll[b][:n], non_blocking=True)
            mask[k0 + 1:k0 + 1 + n].copy_(d_mk[b][:n], non_blocking=True)
        ev_out[c] = torch.cuda.Event(); ev_out[c].record(s_out)
    torch.cuda.synchronize(dev)
    posC, posG, mask = posC.numpy(), posG.numpy(), mask.numpy()
    _finish_rows(posC, posG, mask, pos0, posG0, rec_first, kstrt)
    return dict(posC=posC, posG=posG, mask=mask, n_alive=d_na.cpu().numpy())


TrackEngine._track_chunked = _track_chunked


def _record_getter(records):
    if callable(records):
        return records
    if isinstance(records, (tuple, list)) and len(records) == 3:
        U, V, IC = records
        return lambda k: (U[k], V[k], IC[k])
    arr = records
    return lambda k: (arr[k, 0], arr[k, 1], arr[k, 2])
