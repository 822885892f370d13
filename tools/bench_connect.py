#!/usr/bin/env python3
"""Time st_connect_dev (k_connect), one connectivity sample of every buoy, against one st_step in the same run, and
print one JSON line.

    python tools/bench_connect.py [--buoys 12500000] [--seconds 1.0] [--out FILE]

Workload: bench.py's cfg5 cloud (synthetic 1/12-degree-class C-grid 1700x1475, 12.5 M dense seeds located on the
device, 12.47 M kept), handed over in random order and stored cell-major (set_buoys_dev(sort=True)), as bench.py
does.  Two label maps: 31 block regions (a 6 x 6 tiling of the grid, tile k labelled 1 + k % 31) and one region
covering the whole grid, where every lane of a warp adds to one bin.  Sample 0 is the state handed to set_buoys (every
buoy starts); the timed call is sample 1 on the cells a first st_step leaves, with 1 % of the buoys masked (they end).
Before each timed call the state after sample 0 is restored and a 256 MB buffer is written, so that neither the state
nor the cells are served from the 126 MB L2; each call is timed alone with CUDA events, over >= --seconds in all.
st_step on the same record is timed back to back (its working set does not fit in L2 either).  Byte model per buoy:
cell word 8 + mask 1 + state 8 read, label 1 gathered (L2-resident map), state 8 written for a buoy whose state
changes (region changed or ended); the rate is also given as a fraction of the data sheet's 7.7 TB/s (HGX B200, one
GPU), labelled so.  Goal: one sample call in <= 0.3 of a step, for both maps.  The state after both samples and the
statistics must equal oracle/connect_ref.py's on the state's cells.
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from bench_deform import card_info, time_loop          # noqa: E402

DATASHEET_TBS = 7.7


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", default="arctic12")
    ap.add_argument("--buoys", type=int, default=12_500_000)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--dead", type=float, default=0.01)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_connect: no CUDA device (there is no CPU fallback to time)")
    import synth
    import sitrack_b200 as sit
    from sitrack_b200 import connect as K
    from oracle import connect_ref as O
    dev = a.device
    torch.cuda.set_device(dev)
    d = torch.device("cuda", dev)
    g = synth.make_grid(**synth.GRID_PRESETS[a.grid], seed=0, with_latlon=True)
    U, V, IC = synth.make_records(g, 1, seed=1)
    _, _, SC = synth.dense_seeds(g, a.buoys, IC[0], seed=3, with_latlon=False)
    Nj, Ni = g["Nj"], g["Ni"]
    eng = sit.TrackEngine(g["Yf"], g["Xf"], g["Yu"], g["Xu"], g["Yv"], g["Xv"], tmask=g["tmask"], device=dev)
    eng.set_locate_grid(g["latT"], g["lonT"], g["ResKM"])
    s = torch.cuda.current_stream(d)
    SC_t = torch.from_numpy(SC).to(d)
    SG_t = torch.empty_like(SC_t)
    sit._lib.check(eng.L.st_xy2latlon_dev(SC_t.shape[0], SC_t.data_ptr(), SG_t.data_ptr(), 70.0, -45.0, s.cuda_stream))
    SG_t[:, 1] = torch.remainder(SG_t[:, 1], 360.0)
    cell_t, _, keep_t = eng.seed_locate_dev(SG_t, SC_t, torch.from_numpy(IC[0]).to(d))
    pos0_t, cell0_t = eng.seed_compact_dev(SC_t, cell_t, keep_t)
    del SG_t, SC_t, cell_t, keep_t
    gen = torch.Generator(device=d); gen.manual_seed(11)
    shuf = torch.randperm(int(pos0_t.shape[0]), device=d, generator=gen)
    eng.set_buoys_dev(pos0_t[shuf].contiguous(), cell0_t[shuf].contiguous(), sort=True)
    torch.cuda.synchronize()
    del pos0_t, cell0_t, shuf
    nP = eng.nP
    # sample 0: the cells handed to set_buoys (engine order; get_state strips bit 31, the device words are copied)
    p = C.c_void_p()
    sit._lib.check(eng.L.st_state_device_ptrs(eng.h, None, C.byref(p), None), eng.h)
    from sitrack_b200.engine import _tensor_from_ptr
    cells0 = _tensor_from_ptr(torch, p.value, (nP, 2), torch.int32, 4, dev).clone().view(torch.int32)
    eng.record_slots(1)
    st = eng.staging(0)
    st[0], st[1], st[2] = U[0], V[0], IC[0]
    eng.submit_record(0)
    yx = torch.empty((nP, 2), dtype=torch.float64, device=d)
    ll = torch.empty((nP, 2), dtype=torch.float64, device=d)
    mk = torch.empty((nP,), dtype=torch.int8, device=d)
    eng.step(0, 0, yx, ll, mk, None, s)
    torch.cuda.synchronize()
    cells1 = _tensor_from_ptr(torch, p.value, (nP, 2), torch.int32, 4, dev).clone().view(torch.int32)
    rng = np.random.default_rng(5)
    m0 = np.ones(nP, np.int8)
    m1 = mk.cpu().numpy().copy()
    m1[rng.random(nP) < a.dead] = 0
    m0_t, m1_t = torch.from_numpy(m0).to(d), torch.from_numpy(m1).to(d)
    us_step, n_step = time_loop(torch, lambda: eng.step(0, 0, yx, ll, mk, None, s), a.seconds)

    jj, ii = np.meshgrid(np.arange(Nj), np.arange(Ni), indexing="ij")
    maps = {"blocks_31": 1 + ((jj * 6 // Nj) * 6 + ii * 6 // Ni) % 31, "one_region": np.ones((Nj, Ni), np.int64)}
    h0, h1 = cells0.cpu().numpy(), cells1.cpu().numpy()
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=d)
    res, ok = {}, True
    for name, lab in maps.items():
        lab, R = K.check_labels(lab, Nj, Ni)
        plan = K._Plan(torch, d, lab, R, Nj, Ni, nP, None, 1.0)
        (o0,) = plan.outputs()
        (o1,) = plan.outputs()
        plan.start(None, m0_t, (o0,), s, cell_t=cells0)
        saved = plan.state.clone()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def one(timed):
            plan.state.copy_(saved)
            flush.fill_(1)
            plan.t = 0
            if timed:
                e0.record(s)
            plan.window(None, None, None, m1_t, 1.0, (o1,), s, cell_t=cells1)
            if timed:
                e1.record(s)
                e1.synchronize()
                return e0.elapsed_time(e1) * 1e3
            return 0.0
        for _ in range(10):
            one(False)
        total, n = 0.0, 0
        while total < a.seconds * 1e6 or n < 50:
            total += one(True)
            n += 1
        us = total / n
        o1.zero_()
        one(False)
        torch.cuda.synchronize()
        got0 = K.stats_dict(plan.tau_edges, 1.0, R, o0.cpu().numpy())
        got1 = plan.results((o1.cpu(),))[0]
        st1 = plan.state_dict()
        s0, r0 = O.sample(O.new_state(nP), lab, R, h0, m0, 0)
        s1, r1 = O.sample(s0, lab, R, h1, m1, 1)
        good = all(np.array_equal(got1[k], r1[k]) for k in O.NAMES) and \
            all(np.array_equal(got0[k], r0[k]) for k in O.NAMES) and \
            all(np.array_equal(st1[k], s1[:, i]) for i, k in enumerate(("status", "src", "prev", "start", "visited")))
        ok &= good
        changed = int((s1 != s0).any(1).sum())
        bpb = 8 + 1 + 8 + 1 + 8 * changed / nP
        rate = bpb * nP / (us * 1e-6) / 1e12
        res[name] = dict(us=round(us, 1), calls_timed=n, over_step=round(us / us_step, 3), regions=R,
                         started=int(r0["n_start"].sum()),
                         state_writes=changed, ended=int(r1["n_end"].sum()), arrivals=int(r1["n_arrive"].sum()),
                         bytes_per_buoy=round(bpb, 3), rate_tbs=round(rate, 3),
                         fraction_of_datasheet_7_7_tbs=round(rate / DATASHEET_TBS, 3), oracle_check_passed=bool(good),
                         goal_at_most_0_3_step=bool(us <= 0.3 * us_step))
        del plan, saved
    r = dict(metric="k_connect: one connectivity sample of every buoy, against one st_step", buoys=int(nP),
             grid="%dx%d" % (Nj, Ni), step_us=round(us_step, 1), step_calls_timed=n_step, connect=res,
             byte_model="per buoy: cell word 8 + mask 1 + state 8 read, label 1 gathered, state 8 written if changed",
             timing="each sample call alone between CUDA events, after restoring the state and writing 256 MB",
             oracle_check_passed=ok,
             workload="bench.py cfg5 cloud (synthetic %s grid, %d dense seeds, cell-major), sample 1 after one step, "
                      "%.0f %% of the buoys ending" % (a.grid, a.buoys, 100 * a.dead),
             card=card_info(torch, dev))
    eng.close()
    line = json.dumps(r)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
