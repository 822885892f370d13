#!/usr/bin/env python3
"""Time st_deform_dev (k_deform) at the cfg5-share size and print one JSON line.

    python tools/bench_deform.py [--ny 3531 --nx 3531] [--seconds 1.0] [--out FILE]

Workload: ~12.5 M buoys (the cfg5-share cloud of bench.py: 1700x1475 grid, ~12.5 M buoys per GPU) on a jittered
lattice stored row by row (the order a cell-major cloud has), 2 triangles per lattice square (~25 M triangles,
anticlockwise, already in the order of their smallest vertex); a random drift between the two rows, 1 % of the
vertices masked.  A Delaunay triangulation of this many points would take minutes on the host, so the mesh is
built in numpy.  Inputs (~740 MB) are far larger than the 126 MB L2.

Timed with CUDA events over >= --seconds of back-to-back launches after a warm-up; the anchor copy the record
loop runs after each window (device-to-device, f8 positions + mask) and the two-f8-row copy to pinned host memory
it replaces are timed the same way.  Byte model from shapes: 12 B of indices + 24 B of outputs per triangle,
2 x (16 + 1) B of positions and masks per buoy.  A random sample of triangles is checked bit for bit against
oracle/deform_ref.py.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def card_info(torch, dev):
    info = dict(name=torch.cuda.get_device_name(dev), power_limit_w=None)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev)
        info["power_limit_w"] = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
    except Exception:                   # noqa: BLE001
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                                 stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
            info["power_limit_w"] = float(out.splitlines()[0])
        except Exception:               # noqa: BLE001
            pass
    return info


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:                   # noqa: BLE001
        return 7700.0, "data sheet (HGX B200, one GPU); not measured"


def lattice(ny, nx, rng):
    jj, ii = np.divmod(np.arange(ny * nx, dtype=np.int64), nx)
    yx0 = np.stack([jj * 3.0, ii * 3.0], 1) + rng.uniform(-0.6, 0.6, (ny * nx, 2))       # 3 km spacing
    yx1 = yx0 + 1.5 + rng.normal(0.0, 0.05, (ny * nx, 2))
    a = (np.arange(ny - 1, dtype=np.int64)[:, None] * nx + np.arange(nx - 1)[None, :]).ravel()
    # square a, a+1, a+nx+1, a+nx in (x, y): two anticlockwise triangles, smallest vertex first
    tri = np.empty((2 * a.size, 3), np.int32)
    tri[0::2, 0], tri[0::2, 1], tri[0::2, 2] = a, a + 1, a + nx + 1
    tri[1::2, 0], tri[1::2, 1], tri[1::2, 2] = a, a + nx + 1, a + nx
    m0 = (rng.random(ny * nx) >= 0.01).astype(np.int8)
    m1 = (rng.random(ny * nx) >= 0.01).astype(np.int8)
    return yx0, yx1, m0, m1, tri


def time_loop(torch, fn, seconds, warm=20):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); [fn() for _ in range(warm)]; e1.record(); e1.synchronize()
    n = max(50, int(seconds * 1e3 / max(e0.elapsed_time(e1) / warm, 1e-3)))
    e0.record()
    for _ in range(n):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n, n                          # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ny", type=int, default=3531)
    ap.add_argument("--nx", type=int, default=3531)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_deform: no CUDA device (there is no CPU fallback to time)")
    from sitrack_b200 import _lib, deform as D
    from oracle import deform_ref as R
    dev = a.device
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(0)
    yx0, yx1, m0, m1, tri = lattice(a.ny, a.nx, rng)
    nP, nT = yx0.shape[0], tri.shape[0]
    g = lambda x: torch.from_numpy(x).cuda()
    tri_t, yx0_t, yx1_t, m0_t, m1_t = g(tri), g(yx0), g(yx1), g(m0), g(m1)
    out_t = torch.empty((6, nT), dtype=torch.float32, device="cuda")
    L, s = _lib.lib(), torch.cuda.current_stream()
    dt = 6 * 3600.0 / 86400.0
    run = lambda: D.launch(L, None, nT, tri_t, yx0_t, m0_t, yx1_t, m1_t, dt, out_t, s)
    us, n = time_loop(torch, run, a.seconds)
    # correctness on a random sample (the oracle is numpy: a sample, not all 25 M)
    out = out_t.cpu().numpy()
    pick = np.sort(rng.choice(nT, 200000, replace=False))
    ref = R.deform(yx0, yx1, m0, m1, tri[pick], dt)
    exact = all(np.array_equal(out[j, pick], ref[k]) for j, k in enumerate(R.NAMES))
    # the anchor copy after each window, and what moving two f8 rows to the host costs instead
    a_yx, a_mk = torch.empty_like(yx1_t), torch.empty_like(m1_t)

    def anchor():
        a_yx.copy_(yx1_t); a_mk.copy_(m1_t)
    us_anchor, n_anchor = time_loop(torch, anchor, a.seconds / 2, warm=5)
    h0, h1 = torch.empty_like(yx0_t, device="cpu").pin_memory(), torch.empty_like(yx1_t, device="cpu").pin_memory()

    def d2h():
        h0.copy_(yx0_t, non_blocking=True); h1.copy_(yx1_t, non_blocking=True)
    us_d2h, n_d2h = time_loop(torch, d2h, a.seconds / 2, warm=3)
    bytes_model = nT * (12 + 24) + nP * 2 * (16 + 1)
    peak, peak_src = hbm_peak()
    gbs = bytes_model / (us * 1e-6) / 1e9
    res = dict(metric="deform_us_per_window", value=round(us, 2), unit="us", higher_is_better=False,
               triangles=nT, buoys=nP, triangles_per_s=nT / (us * 1e-6), launches_timed=n,
               bytes_model=dict(per_triangle=36, per_buoy=34, total=bytes_model, achieved_gbs=round(gbs, 1),
                                hbm_peak_gbs=peak, peak_source=peak_src, frac_of_peak=round(gbs / peak, 4)),
               anchor_copy_us=round(us_anchor, 2), anchor_copies_timed=n_anchor,
               d2h_two_f8_rows_us=round(us_d2h, 1), d2h_copies_timed=n_d2h,
               bit_identical_to_oracle_on_sample=bool(exact), sample=int(pick.size),
               valid_fraction=float((out[0] != -9999.0).mean()),
               workload="jittered 3 km lattice %dx%d, 2 triangles per square, sorted by smallest vertex; "
                        "inputs larger than L2, no flush" % (a.ny, a.nx),
               card=card_info(torch, dev))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if exact else 1


if __name__ == "__main__":
    sys.exit(main())
