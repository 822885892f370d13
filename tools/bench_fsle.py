#!/usr/bin/env python3
"""Time st_fsle_dev (k_fsle), one sample of the finite-size Lyapunov state of every pair, and print one JSON line.

    python tools/bench_fsle.py [--ny 3531 --nx 3531] [--sep-pairs 4000000] [--check-pairs 1000000] [--seconds 1.0]
                               [--out FILE]

Workload: section 10's lattice (tools/bench_deform.py: ~12.47 M buoys on a jittered 3 km lattice stored row by row,
2 triangles per square); the pairs are MeshPairs of its mesh (~37 M nearest-neighbour pairs) plus --sep-pairs
SeparationPairs at 10 to 1000 km (seed 0), in that order, as in tools/bench_dispersion.py.  9 f8 rows with their
masks: row 0 is the lattice, each next row drifts by a smooth field plus noise, and 1 % of the buoys die at each row.
The inputs (~2 GB) are far larger than the 126 MB L2, so no flush is needed.

Timed with CUDA events over >= --seconds after a warm-up: the run of 8 samples as the record loop issues it (sample 1
with row 0 as the start row, which resets every pair, then samples 2 ... 8), repeated, with an event between calls;
the figure is the mean sample call (2 ... 8), the reset call is reported on its own.  In the same run, one
single-origin st_dispersion_dev call (row 7 to row 8) on the same pairs.  Byte model from shapes, per sample call:
8 B of indices and 8 B of state read per pair, 8 B written per pair whose state changes, 17 B (f8 position + mask) per
buoy of the row; the rate is given as a fraction of the data sheet's 7.7 TB/s (HGX B200, one GPU), labelled so.  The
final state and the summed statistics of --check-pairs pairs drawn from the set (seed 1) must equal
oracle/fsle_ref.py's.
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

from bench_deform import card_info, lattice, time_loop          # noqa: E402

DATASHEET_TBS = 7.7
NROW = 9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ny", type=int, default=3531)
    ap.add_argument("--nx", type=int, default=3531)
    ap.add_argument("--sep-pairs", type=int, default=4000000)
    ap.add_argument("--check-pairs", type=int, default=1000000)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_fsle: no CUDA device (there is no CPU fallback to time)")
    import sitrack_b200 as sit
    from sitrack_b200 import dispersion as P
    from sitrack_b200 import fsle as F
    from oracle import fsle_ref as O
    dev = a.device
    torch.cuda.set_device(dev)
    d = torch.device("cuda", dev)
    rng = np.random.default_rng(0)
    yx0, _, m0, _, tri = lattice(a.ny, a.nx, rng)
    nP = yx0.shape[0]
    mesh = sit.MeshPairs(tri)
    pairs = np.concatenate([mesh, sit.SeparationPairs(yx0, 10.0, 1000.0, a.sep_pairs, seed=0)])
    del tri, m0
    nQ = pairs.shape[0]
    g = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(d)
    hrows, hmasks = [yx0], [np.ones(nP, np.int8)]
    for k in range(NROW - 1):
        yx = hrows[-1]
        hrows.append(yx + 1.5 + np.stack([np.sin(yx[:, 1] / 90.0 + k), np.cos(yx[:, 0] / 70.0 - k)], 1) * 0.8 +
                     rng.normal(0.0, 0.05, yx.shape))
        hmasks.append(hmasks[-1] * (rng.random(nP) >= 0.01).astype(np.int8))
    rows, masks = [g(r) for r in hrows], [g(m) for m in hmasks]
    s = torch.cuda.current_stream()
    sd = 6 * 3600.0 / 86400.0
    deltas = F.DEFAULT_DELTAS

    def run_samples(plan, outs, ev=None):
        for t in range(1, NROW):
            plan.launch(None, rows[t], masks[t], t, (rows[0], masks[0]) if t == 1 else None, outs[t - 1], s)
            if ev is not None:
                ev[t].record(s)

    plan = F._Plan(torch, d, pairs, deltas, None, sd)
    outs = [plan.outputs()[0] for _ in range(NROW - 1)]
    # changed pairs per sample (untimed), for the byte model
    changed = []
    for t in range(1, NROW):
        before = plan.state.clone()
        plan.launch(None, rows[t], masks[t], t, (rows[0], masks[0]) if t == 1 else None, outs[t - 1], s)
        changed.append(int((plan.state != before).any(1).sum()))
        del before
    run_samples(plan, outs)
    for _ in range(3):
        run_samples(plan, outs)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(NROW)]
    ev[0].record(s); run_samples(plan, outs, ev); ev[-1].synchronize()
    per_run_ms = ev[0].elapsed_time(ev[-1])
    reps = max(20, int(a.seconds * 1e3 / max(per_run_ms, 1e-3)))
    acc = np.zeros(NROW - 1)
    for _ in range(reps):
        ev[0].record(s)
        run_samples(plan, outs, ev)
        ev[-1].synchronize()
        acc += [ev[t - 1].elapsed_time(ev[t]) for t in range(1, NROW)]
    us = acc * 1e3 / reps
    us_sample = float(us[1:].mean())
    stats = [plan.results((o.cpu(),))[0] for o in outs]

    dplan = P._Plan(torch, d, pairs, 1)
    h, su = dplan.outputs()
    disp = lambda: dplan.launch(None, rows[NROW - 1], masks[NROW - 1], [(rows[NROW - 2], masks[NROW - 2], 1)], sd, h,
                                su, None, s)
    us_disp, n_disp = time_loop(torch, disp, a.seconds)
    del dplan, h, su

    # the oracle on a sample of the pairs, run on the device on its own
    crng = np.random.default_rng(1)
    sel = np.sort(crng.choice(nQ, min(a.check_pairs, nQ), replace=False))
    cp = pairs[sel]
    cplan = F._Plan(torch, d, cp, deltas, None, sd)
    couts = [cplan.outputs()[0] for _ in range(NROW - 1)]
    run_samples(cplan, couts)
    torch.cuda.synchronize()
    got = [cplan.results((o.cpu(),))[0] for o in couts]
    rs, rw = O.run(hrows, hmasks, cp, deltas, F.DEFAULT_TAU_EDGES)
    ok = np.array_equal(cplan.state.cpu().numpy(), rs[-1])
    for k in ("n_start", "hist_tau", "n", "sum_tau", "sum_tau2", "n_censored"):
        ok &= all(np.array_equal(x[k], y[k]) for x, y in zip(got, rw))
    ok = bool(ok)

    nchg = float(np.mean(changed[1:]))
    bytes_sample = 16 * nQ + 8 * nchg + 17 * nP
    rate = bytes_sample / (us_sample * 1e-6) / 1e12
    tot_n = sum(w["n"] for w in stats)
    res = dict(metric="finite-size Lyapunov state of every pair, one sample", buoys=int(nP), pairs=int(nQ),
               mesh_pairs=int(mesh.shape[0]), thresholds=int(deltas.size), samples=NROW - 1,
               fsle_us=round(us_sample, 1), fsle_us_by_sample=[round(float(x), 1) for x in us],
               fsle_reset_call_us=round(float(us[0]), 1), runs_timed=reps,
               dispersion_single_origin_us=round(us_disp, 1), dispersion_calls_timed=n_disp,
               fsle_over_dispersion=round(us_sample / us_disp, 3), goal_at_most_half=bool(us_sample <= 0.5 * us_disp),
               byte_model="16 B per pair (indices + state) + 8 B per changed pair + 17 B per buoy of the row",
               changed_pairs_per_sample=[int(c) for c in changed], sample_bytes=int(bytes_sample),
               fsle_rate_tbs=round(rate, 3), fsle_fraction_of_datasheet_7_7_tbs=round(rate / DATASHEET_TBS, 3),
               exit_times_recorded=int(tot_n.sum()), check_pairs=int(cp.shape[0]), oracle_check_passed=ok,
               workload="jittered 3 km lattice %dx%d, MeshPairs + %d SeparationPairs (10-1000 km), %d f8 rows, 1 %% "
                        "deaths per row, the default 19 thresholds (2-1024 km); inputs larger than L2, no flush"
                        % (a.ny, a.nx, a.sep_pairs, NROW),
               card=card_info(torch, dev))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
