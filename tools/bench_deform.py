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

The coarse-graining pass (st_deform_scales_dev: level-1 box sums with the triangles' statistics, one parent pass per
level, box statistics, final reduction) is timed the same way on the same rows, for --L0 km boxes and --levels
levels, with statistics only (no box planes), as the record loop runs it.  Byte model: 12 B of indices per
triangle, 2 x 17 B per buoy, 8 B of level-1 ranges per level-1 box and 64 B box records (written once, read by the
parent and statistics passes).  The level-1 outputs of a random sample of boxes are checked bit for bit against
oracle/deform_scale_ref.py, and two passes must give the same statistics bit for bit.

The Eulerian grid pass (st_deform_grid_dev: cell keys, device radix sort, segmentation, the same box passes, field
scatter) is timed the same way in the same run, on a grid of --L0 km cells and --levels levels covering the lattice
at mid-time, with its statistics and dense fields as the record loop runs it.  The cumulative stages (keys; keys +
sort; keys + sort + segmentation; the whole pass) are timed as well through st_deform_grid_stages_dev, so key, sort
and segmentation times are differences of event timings.  The fields of a random sample of level-1 cells are
checked bit for bit against oracle/deform_grid_ref.py, and two passes must give the same statistics and fields.
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


def scales(torch, a, rng, yx0, yx1, m0, m1, tri, dt, g, us_deform):
    """Time and check the coarse-graining pass on the same rows."""
    import time
    from sitrack_b200 import deform_scales as DS
    from oracle import deform_scale_ref as O
    t0 = time.perf_counter()
    H = DS.BoxHierarchy(yx0, tri, a.L0, a.levels)
    t_build = time.perf_counter() - t0
    nP, nT = yx0.shape[0], tri.shape[0]
    plan = DS._DevicePlan(torch, torch.device("cuda", torch.cuda.current_device()), H, tri)
    mom, hist = plan.outputs()
    yx0_t, yx1_t, m0_t, m1_t = g(yx0), g(yx1), g(m0), g(m1)
    s = torch.cuda.current_stream()
    run = lambda: plan.launch(None, yx0_t, m0_t, yx1_t, m1_t, dt, mom, hist, None, s)
    us, n = time_loop(torch, run, a.seconds)
    m1_, h1_ = mom.cpu().numpy(), hist.cpu().numpy()
    run()
    same = bool(np.array_equal(m1_, mom.cpu().numpy()) and np.array_equal(h1_, hist.cpu().numpy()))
    # level-1 outputs of a sample of boxes against the oracle (the box planes of one more pass)
    boxes_t = torch.empty((7, int(H.nbox.sum())), dtype=torch.float32, device="cuda")
    plan.launch(None, yx0_t, m0_t, yx1_t, m1_t, dt, mom, hist, boxes_t, s)
    planes = boxes_t[:, :int(H.nbox[0])].cpu().numpy()
    pick = np.sort(rng.choice(int(H.nbox[0]), min(20000, int(H.nbox[0])), replace=False))
    lo, hi = H.tri_off[pick], H.tri_off[pick + 1]
    ts = np.concatenate([H.order[i:j] for i, j in zip(lo, hi)])
    off = np.r_[0, np.cumsum(hi - lo)]
    T, _, _ = O.triangle_terms(yx0, yx1, m0, m1, tri[ts], dt)
    o, ok = O.box_outputs(O.level1_sums(T, off), H.min_area[0])
    with np.errstate(all="ignore"):
        exact = all(np.array_equal(planes[j, pick], np.where(ok, o[k], O.FillValue).astype(np.float32))
                    for j, k in enumerate(O.BOX_NAMES))
    nb = H.nbox.astype(np.int64)
    nball = int(nb.sum())
    bytes_model = nT * 12 + nP * 2 * 17 + int(nb[0]) * 8 + 64 * (2 * nball + nball - int(nb[0]))
    peak, _ = hbm_peak()
    gbs = bytes_model / (us * 1e-6) / 1e9
    return dict(us_per_window=round(us, 2), passes_timed=n, vs_k_deform=round(us / us_deform, 3), L0_km=a.L0,
                levels=a.levels, boxes_per_level=nb.tolist(), host_build_s=round(t_build, 2),
                bytes_model=dict(total=bytes_model, achieved_gbs=round(gbs, 1), frac_of_peak=round(gbs / peak, 4)),
                n_per_scale=h1_[:, 0].sum(1).tolist(), sample_boxes=int(pick.size),
                sample_boxes_bit_identical=bool(exact), run_to_run_identical=same)


def grid(torch, a, rng, yx0, yx1, m0, m1, tri, dt, g, us_deform, us_scales):
    """Time and check the Eulerian grid pass on the same rows."""
    import ctypes as C
    import sitrack_b200 as sit
    from sitrack_b200 import deform_grid as DG
    from sitrack_b200._lib import check
    from oracle import deform_scale_ref as O
    from oracle import deform_grid_ref as OG
    L0 = a.L0
    mid = 0.5 * (yx0 + yx1)
    origin = np.floor(mid.min(0) / L0) * L0
    shape = tuple(int(n) for n in np.floor((mid.max(0) - origin) / L0) + 1)
    G = sit.EulerianGrid(origin, L0, shape, a.levels)
    plan = DG._GridPlan(torch, torch.device("cuda", torch.cuda.current_device()), G, tri)
    mom, hist, fields, nbox = plan.outputs()
    yx0_t, yx1_t, m0_t, m1_t = g(yx0), g(yx1), g(m0), g(m1)
    s = torch.cuda.current_stream()
    L = plan.L

    def stages(upto):
        check(L.st_deform_grid_stages_dev(
            None, int(plan.tri_t.shape[0]), plan.tri_t.data_ptr(), yx0_t.data_ptr(), m0_t.data_ptr(), yx1_t.data_ptr(),
            m1_t.data_ptr(), float(dt), G.levels, G.shape[0], G.shape[1], float(G.origin[0]), float(G.origin[1]),
            G.L0_km, plan.min_area.ctypes.data, G.bin_edges.size, plan.edges_t.data_ptr(), plan.scratch.data_ptr(),
            plan.scratch_bytes, mom.data_ptr(), hist.data_ptr(), fields.data_ptr(), nbox.data_ptr(), upto,
            C.c_void_p(s.cuda_stream)))
    run = lambda: plan.launch(None, yx0_t, m0_t, yx1_t, m1_t, dt, mom, hist, fields, nbox, s)
    us, n = time_loop(torch, run, a.seconds)
    cum = [time_loop(torch, lambda u=u: stages(u), a.seconds / 2)[0] for u in (1, 2, 3)]
    run()
    m1_, h1_, f1_, nb = mom.cpu().numpy(), hist.cpu().numpy(), fields.cpu().numpy(), nbox.cpu().numpy()
    run()
    same = bool(np.array_equal(m1_, mom.cpu().numpy()) and np.array_equal(h1_, hist.cpu().numpy()) and
                np.array_equal(f1_.view(np.uint32), fields.cpu().numpy().view(np.uint32)))
    # level-1 cells of a sample of binned triangles' cells against the oracle, bit for bit
    fl = DG.split_fields(G, f1_)
    parts = [OG.eulerian_binning(yx0, yx1, m0, m1, tri[i:i + 2 ** 21], G.origin, L0, G.shape)
             for i in range(0, tri.shape[0], 2 ** 21)]                # in slices: host memory
    binned, key = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
    cell = key[:, 0] * G.shape[1] + key[:, 1]
    cells = np.unique(cell[binned])
    pick = np.sort(rng.choice(cells, min(20000, cells.size), replace=False))
    sel = np.flatnonzero(binned & np.isin(cell, pick))
    sel = sel[np.argsort(cell[sel], kind="stable")]                 # caller's order within each cell
    cs = cell[sel]
    st = np.flatnonzero(np.r_[True, cs[1:] != cs[:-1]])
    off = np.r_[st, cs.size]
    T, _, _ = O.triangle_terms(yx0, yx1, m0, m1, tri[sel], dt)
    o, ok = O.box_outputs(O.level1_sums(T, off), G.min_area[0])
    ucell = cs[st]
    with np.errstate(all="ignore"):
        exact = all(np.array_equal(fl[0][k].ravel()[ucell], np.where(ok, o[k], O.FillValue).astype(np.float32))
                    for k in O.BOX_NAMES)
    stage = dict(key_us=round(cum[0], 2), sort_us=round(cum[1] - cum[0], 2), segmentation_us=round(cum[2] - cum[1], 2),
                 boxes_stats_fields_us=round(us - cum[2], 2))
    return dict(us_per_window=round(us, 2), passes_timed=n, vs_k_deform=round(us / us_deform, 3),
                vs_lagrangian_pass=round(us / us_scales, 3), goal_2x_lagrangian_met=bool(us <= 2.0 * us_scales),
                stages_cumulative_us=[round(c, 2) for c in cum], stages=stage, L0_km=L0, levels=a.levels,
                origin_km=G.origin.tolist(), shape=list(G.shape), boxes_per_level=nb.tolist(),
                n_per_scale=h1_[:, 0].sum(1).tolist(), binned_triangles=int(binned.sum()),
                field_words=G.field_size(), sample_cells=int(pick.size), sample_cells_bit_identical=bool(exact),
                run_to_run_identical=same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ny", type=int, default=3531)
    ap.add_argument("--nx", type=int, default=3531)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    ap.add_argument("--L0", type=float, default=12.0)
    ap.add_argument("--levels", type=int, default=6)
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
    pick = np.sort(rng.choice(nT, min(200000, nT), replace=False))
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
    sc = scales(torch, a, rng, yx0, yx1, m0, m1, tri, dt, g, us)
    gr = grid(torch, a, rng, yx0, yx1, m0, m1, tri, dt, g, us, sc["us_per_window"])
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
               scales=sc, grid=gr, card=card_info(torch, dev))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if (exact and sc["sample_boxes_bit_identical"] and sc["run_to_run_identical"] and
                 gr["sample_cells_bit_identical"] and gr["run_to_run_identical"]) else 1


if __name__ == "__main__":
    sys.exit(main())
