#!/usr/bin/env python3
"""Time st_sample_dev (k_sample), one sampled row of SI3 fields along the trajectories, against one st_step in the
same run, and print one JSON line.

    python tools/bench_sample.py [--buoys 12500000] [--check-buoys 1000000] [--seconds 1.0] [--out FILE]

Workload: bench.py's cfg5 cloud (synthetic 1/12-degree-class C-grid 1700x1475, 12.5 M dense seeds located on the
device, 12.47 M kept), handed over in random order and stored cell-major (set_buoys_dev(sort=True)), as bench.py
does.  One record is resident; the row is the one a first st_step (f8 row, not chained) leaves.  Then, timed with
CUDA events over >= --seconds each after a warm-up: st_step on that record (f8 yx, lat/lon and mask rows, as
bench.py's step), and st_sample_dev in cell and bilinear modes with 1 field (siconc, plane 2 of the record slot) and
with 4 fields (four planes of a separate buffer).  The state and the fields (3 + 4 planes of 10 MB) fit in L2 with
room to spare only in part: the streamed per-buoy inputs (cell, mask, position: 25 B x 12.47 M) do not, so no flush is
needed.  Byte model from shapes, per buoy: cell 8 + mask 1 + 4 nF written; bilinear 16 more for the position; the
rate is also given as a fraction of the data sheet's 7.7 TB/s (HGX B200, one GPU), labelled so.  Goals: one field
in cell mode in <= 0.25 of a step, bilinear in <= 0.5.  The outputs of --check-buoys buoys (seed 1) in all four
configurations must equal oracle/sample_ref.py's on the state's cells.
"""
import argparse
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
    ap.add_argument("--check-buoys", type=int, default=1_000_000)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_sample: no CUDA device (there is no CPU fallback to time)")
    import synth
    import sitrack_b200 as sit
    from sitrack_b200 import sample as S
    from oracle import sample_ref as O
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
    nP = eng.nP
    eng.record_slots(1)
    st = eng.staging(0)
    st[0], st[1], st[2] = U[0], V[0], IC[0]
    eng.submit_record(0)
    yx = torch.empty((nP, 2), dtype=torch.float64, device=d)
    ll = torch.empty((nP, 2), dtype=torch.float64, device=d)
    mk = torch.empty((nP,), dtype=torch.int8, device=d)
    eng.step(0, 0, yx, ll, mk, None, s)
    torch.cuda.synchronize()
    # the sampled row: its cells, positions and mask in engine order (set_buoys_dev keeps its permutation on the
    # device, so get_state hands the state back as stored), kept aside while the step is timed
    cells = eng.get_state()[1]
    yx_s, mk_s = yx.clone(), mk.clone()
    step = lambda: eng.step(0, 0, yx, ll, mk, None, s)
    us_step, n_step = time_loop(torch, step, a.seconds)
    eng.set_buoys_dev(pos0_t[shuf].contiguous(), cell0_t[shuf].contiguous(), sort=True)
    eng.step(0, 0, yx, ll, mk, None, s)                      # back to the sampled row's state (the same first step)
    torch.cuda.synchronize()
    same = torch.equal(yx, yx_s) and torch.equal(mk, mk_s)
    del pos0_t, cell0_t, shuf

    four = np.stack([IC[0], U[0], V[0], np.float32(2.0) * IC[0]])
    f4_t = torch.from_numpy(four).to(d)
    ic_ptr = eng.record_device_ptr(0) + 2 * Nj * Ni * 4
    out = torch.empty((4, nP), dtype=torch.float32, device=d)
    res = {}
    crng = np.random.default_rng(1)
    sel = np.sort(crng.choice(nP, min(a.check_buoys, nP), replace=False))
    hyx, hmk = yx_s.cpu().numpy()[sel], mk_s.cpu().numpy()[sel]
    ok = bool(same)
    for interp in ("cell", "bilinear"):
        plan = S._Plan(eng, torch, d, interp, (g["Yt"], g["Xt"]))
        for nF in (1, 4):
            ptr = ic_ptr if nF == 1 else f4_t.data_ptr()
            fn = lambda: plan.launch(ptr, nF, Nj * Ni, yx_s, mk_s, out.data_ptr(), s)
            us, n = time_loop(torch, fn, a.seconds)
            fn()
            torch.cuda.synchronize()
            got = out[:nF].cpu().numpy()[:, sel]
            ref = O.sample(four[:nF], g["tmask"], cells[sel], hyx, hmk, interp, g["Yt"], g["Xt"])
            good = got.tobytes() == ref.tobytes()
            ok &= good
            bpb = 8 + 1 + 4 * nF + (16 if interp == "bilinear" else 0)
            rate = bpb * nP / (us * 1e-6) / 1e12
            res["%s_%d" % (interp, nF)] = dict(us=round(us, 1), calls_timed=n, over_step=round(us / us_step, 3),
                                               bytes_per_buoy=bpb, rate_tbs=round(rate, 3),
                                               fraction_of_datasheet_7_7_tbs=round(rate / DATASHEET_TBS, 3),
                                               oracle_check_passed=bool(good),
                                               filled=int((got == np.float32(O.FillValue)).sum()))
    r = dict(metric="k_sample: SI3 fields at every buoy of one trajectory row, against one st_step", buoys=int(nP),
             grid="%dx%d" % (Nj, Ni), step_us=round(us_step, 1), step_calls_timed=n_step, sample=res,
             goal_cell_1_at_most_quarter_step=bool(res["cell_1"]["us"] <= 0.25 * us_step),
             goal_bilinear_1_at_most_half_step=bool(res["bilinear_1"]["us"] <= 0.5 * us_step),
             byte_model="per buoy: cell word 8 + row mask 1 + 4 per field written; bilinear +16 (f8 position)",
             check_buoys=int(sel.size), oracle_check_passed=ok,
             workload="bench.py cfg5 cloud (synthetic %s grid, %d dense seeds, cell-major), one record; 1 field = "
                      "siconc from the record slot, 4 fields from a separate buffer" % (a.grid, a.buoys),
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
