#!/usr/bin/env python3
"""Time st_dispersion_dev (k_disperse) at a window close with 8 active lags and print one JSON line.

    python tools/bench_dispersion.py [--ny 3531 --nx 3531] [--sep-pairs 4000000] [--lags 8] [--seconds 1.0] [--out FILE]

Workload: section 10's lattice (tools/bench_deform.py: ~12.47 M buoys on a jittered 3 km lattice stored row by row,
2 triangles per square); the pairs are MeshPairs of its mesh (~37 M nearest-neighbour pairs) plus --sep-pairs
SeparationPairs at 10 to 1000 km (seed 0), in that order.  lags + 1 f8 rows with their masks: row 0 is the lattice,
each next row drifts by a smooth field plus noise, and 1 % of the buoys die at each row.  The inputs (~2.2 GB) are far
larger than the 126 MB L2, so no flush is needed.

Timed with CUDA events over >= --seconds of back-to-back launches after a warm-up: the fused call (closing row = the
last row, the `lags` rows before it as origins, as the record loop runs it when a window closes once the ring is
full), and in the same run `lags` single-origin calls, one per lag.  Byte model from shapes: 8 B of indices per pair
plus 17 B (f8 position + mask) per buoy for each row read, i.e. lags + 1 rows for the fused call and 2 rows for each
single call; the rate is given as a fraction of the data sheet's 7.7 TB/s (HGX B200, one GPU), labelled so.  The fused
statistics must equal the single calls' bit for bit, and two fused passes too.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ny", type=int, default=3531)
    ap.add_argument("--nx", type=int, default=3531)
    ap.add_argument("--sep-pairs", type=int, default=4000000)
    ap.add_argument("--lags", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_dispersion: no CUDA device (there is no CPU fallback to time)")
    import sitrack_b200 as sit
    from sitrack_b200 import dispersion as P
    dev = a.device
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(0)
    yx0, _, m0, _, tri = lattice(a.ny, a.nx, rng)
    nP = yx0.shape[0]
    mesh = sit.MeshPairs(tri)
    pairs = np.concatenate([mesh, sit.SeparationPairs(yx0, 10.0, 1000.0, a.sep_pairs, seed=0)])
    del tri
    nQ = pairs.shape[0]
    g = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    rows, masks = [g(yx0)], [g(np.ones(nP, np.int8))]
    yx, mk = yx0, np.ones(nP, np.int8)
    for k in range(a.lags):
        yx = yx + 1.5 + np.stack([np.sin(yx[:, 1] / 90.0 + k), np.cos(yx[:, 0] / 70.0 - k)], 1) * 0.8 + \
            rng.normal(0.0, 0.05, yx.shape)
        mk = mk * (rng.random(nP) >= 0.01).astype(np.int8)
        rows.append(g(yx)); masks.append(g(mk))
    del yx, yx0, m0
    dt = 6 * 3600.0 / 86400.0
    s = torch.cuda.current_stream()
    plan = P._Plan(torch, torch.device("cuda", dev), pairs, a.lags)
    origins = [(rows[-1 - l], masks[-1 - l], l) for l in range(1, a.lags + 1)]
    h, su = plan.outputs()
    fused = lambda: plan.launch(None, rows[-1], masks[-1], origins, dt, h, su, None, s)
    us_fused, n_fused = time_loop(torch, fused, a.seconds)
    f_h, f_s = h.cpu().numpy(), su.cpu().numpy()
    fused()
    again = np.array_equal(f_h, h.cpu().numpy()) and np.array_equal(f_s.view(np.int64), su.cpu().numpy().view(np.int64))
    h1, s1 = plan.outputs()

    def singles():
        for o in origins:
            plan.launch(None, rows[-1], masks[-1], [o], dt, h1, s1, None, s)
    us_single, n_single = time_loop(torch, singles, a.seconds, warm=5)
    same = True
    for o in origins:
        plan.launch(None, rows[-1], masks[-1], [o], dt, h1, s1, None, s)
        l = o[2] - 1
        same &= np.array_equal(h1.cpu().numpy()[l], f_h[l]) and \
            np.array_equal(s1.cpu().numpy()[l].view(np.int64), f_s[l].view(np.int64))
    bytes_fused = 8 * nQ + 17 * nP * (a.lags + 1)
    bytes_single = a.lags * (8 * nQ + 17 * nP * 2)
    rate = bytes_fused / (us_fused * 1e-6) / 1e12
    res = dict(metric="pair dispersion at a window close, %d active lags" % a.lags, buoys=int(nP), pairs=int(nQ),
               mesh_pairs=int(mesh.shape[0]), lags=a.lags,
               fused_us=round(us_fused, 1), fused_calls_timed=n_fused,
               single_calls_us=round(us_single, 1), single_calls_timed=n_single,
               fused_over_single=round(us_fused / us_single, 3),
               byte_model="8 B per pair + 17 B per buoy per row read",
               fused_bytes=int(bytes_fused), single_calls_bytes=int(bytes_single),
               fused_rate_tbs=round(rate, 3), fused_fraction_of_datasheet_7_7_tbs=round(rate / DATASHEET_TBS, 3),
               valid_pairs_lag1=int(f_h[0].sum()), fused_equals_single_calls=bool(same), run_to_run_identical=bool(again),
               workload="jittered 3 km lattice %dx%d, MeshPairs + %d SeparationPairs (10-1000 km), %d rows; inputs "
                        "larger than L2, no flush" % (a.ny, a.nx, a.sep_pairs, a.lags + 1),
               card=card_info(torch, dev))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if (same and again) else 1


if __name__ == "__main__":
    sys.exit(main())
