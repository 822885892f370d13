#!/usr/bin/env python3
"""bench.py -- buoy-steps/s of the B200 buoy-advection hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg5|cfg4|cfg3|cfg2]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N > 1)
  python bench.py --impl reference ...        the reference's CPU implementation on host cores
  python bench.py ... --dump-outputs DIR      also write what the last timed step computed, DIR/<name>.npy

A "step" is one hourly record advanced for every buoy of this rank (one launch of
k_advect_step = the body of si3_part_tracker.py:378-493 incl. the lat/lon update).
Workloads (BASELINE.json configs), all synthetic with fixed seeds, weak scaling:
  cfg5 (default)  1/12-degree-class grid 1700x1475, 12.5 M buoys per GPU
                  (= config 5's per-GPU share: 100 M buoys on 8 GPUs)
  cfg4            same grid, 1 M buoys per GPU (config 4)
  cfg3 / cfg2     NANUK4-shaped 566x492 grid, HSS1+scattered (~25 k) / HSS5 (~1 k) buoys
Prints ONE JSON line on rank 0 (see DESIGN.md "Measurement").
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree and writes nothing into it

SEED_BOX = int(os.environ.get("SITRACK_BENCH_SEED_BOX", "0")) or None   # diagnostic only
B_ALG = 83.0          # algorithmic bytes per buoy-step (SURVEY.md §8d): 25 state in + 25 out + 33 row
D2H_PER_BUOY = 33     # y,x f8 + lat,lon f8 + mask i1
# --dump-outputs keeps at most this many buoys (a fixed sample): 44 B each as written (y,x and lat,lon f8, mask f4,
# buoy index f8), 44 MB at most, which leaves room under 64 MB for the per-step alive counts
DUMP_BUOYS = 1_000_000
WORKLOADS = {
    "cfg5": dict(grid="arctic12", buoys=12_500_000, kind="dense", nrec_res=8,
                 label="cfg5-share: synthetic 1/12deg-class C-grid 1700x1475, 12.5M buoys/GPU (100M on 8 GPUs)"),
    "cfg4": dict(grid="arctic12", buoys=1_000_000, kind="dense", nrec_res=8,
                 label="cfg4: synthetic 1/12deg-class C-grid 1700x1475, 1M buoys/GPU"),
    "cfg3": dict(grid="nanuk4", buoys=0, kind="hss1+scattered", nrec_res=48,
                 label="cfg3: NANUK4-shaped 566x492, HSS1 (~25k buoys) + scattered seeding"),
    "cfg2": dict(grid="nanuk4", buoys=0, kind="hss5", nrec_res=48,
                 label="cfg2: NANUK4-shaped 566x492, HSS5 (~1k buoys), -F"),
}


# The contract is ONE JSON line on stdout.  Libraries loaded later write there too (NCCL prints its
# version banner on fd 1 whatever NCCL_DEBUG_FILE says), so the real stdout is kept aside for the result
# and fd 1 is pointed at stderr for everything else.
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(obj):
    os.write(_RESULT_FD, (json.dumps(obj) + "\n").encode())


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------
# clocks during the timed region (NVML; the same counters as the nvidia-smi line of the recipe)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.02):
        self.samples, self.reasons, self.stop_flag, self.period = [], 0, False, period
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:          # noqa: BLE001
            log("clock sampler unavailable:", e)
        self.t = None

    def _once(self):
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            get = getattr(self.nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                self.nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.reasons |= int(get(self.h))
        except Exception:               # noqa: BLE001
            pass

    def _run(self):
        while not self.stop_flag:
            self._once()
            time.sleep(self.period)

    def start(self):
        if self.h is not None:
            self.stop_flag = False
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()

    def stop(self):
        if self.t:
            self.stop_flag = True
            self.t.join()
            self._once()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = [n for b, n in self.REASONS.items() if self.reasons & b and n != "gpu_idle"]
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": float(self.max), "reasons": names,
                "samples": len(self.samples)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:                   # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """dram read+write bytes per launch of k_advect_step from the committed ncu --set full capture."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        return t.get(workload, {}).get("dram_bytes_per_launch")
    except Exception:                   # noqa: BLE001
        return None


# ---------------------------------------------------------------------------------------------
# workload construction (host numpy; not timed)
# ---------------------------------------------------------------------------------------------
def build_workload(name, rank, want_latlon_grid=True, n_dense=None, keep_cells=False):
    import synth
    w = WORKLOADS[name]
    t0 = time.time()
    g = synth.make_grid(**synth.GRID_PRESETS[w["grid"]], seed=0, with_latlon=want_latlon_grid)
    U, V, IC = synth.make_records(g, w["nrec_res"], seed=1)
    if w["kind"] == "dense":
        ids, SG, SC = synth.dense_seeds(g, n_dense or w["buoys"], IC[0], seed=3 + rank, with_latlon=False, box=SEED_BOX,
                                        cells_out=g if keep_cells else None)
    elif w["kind"] == "hss5":
        ids, SG, SC = synth.hss_seeds(g, IC[0], khss=5)
    else:
        i1, G1, C1 = synth.hss_seeds(g, IC[0], khss=1)
        i2, G2, C2 = synth.scattered_seeds(g, 1000, seed=2 + rank)
        ids, SG, SC = np.concatenate([i1, i2 + i1.size]), np.concatenate([G1, G2]), np.concatenate([C1, C2])
    log("[rank %d] workload %s built in %.1fs: grid %dx%d, %d seeds, %d resident records"
        % (rank, name, time.time() - t0, g["Nj"], g["Ni"], SC.shape[0], w["nrec_res"]))
    return g, (U, V, IC), SG, SC


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import sitrack_b200 as sit

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log("WARNING: --gpus %d but WORLD_SIZE=%d; using WORLD_SIZE" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (sitrack_b200 has no CPU path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # stdout carries the one JSON line only
        dist.init_process_group("nccl", device_id=dev)
    from sitrack_b200.dist import bind_host_to_gpu
    cores = bind_host_to_gpu(_physical_index(local))
    log("[rank %d] host threads bound to %s" % (rank, "%d cores near the GPU" % len(cores) if cores else "all cores (no NVML affinity)"))

    K, W = args.steps, args.warmup
    wl = WORKLOADS[args.workload]
    strong = args.scaling == "strong"
    n_dense = None
    if strong:
        if wl["kind"] != "dense":
            raise SystemExit("--scaling strong needs a dense workload (cfg4, cfg5)")
        n_dense = wl["buoys"] // world                    # the workload's buoys are the TOTAL, sharded over the ranks
    g, (U, V, IC), SG, SC = build_workload(args.workload, rank, n_dense=n_dense)
    Nj, Ni = g["Nj"], g["Ni"]
    R = U.shape[0]
    eng = sit.TrackEngine(g["Yf"], g["Xf"], g["Yu"], g["Xu"], g["Yv"], g["Xv"], tmask=g["tmask"], device=local)
    launches = {"n": 0}
    eng.set_kernel_variant({"tuned": 0, "v1": 1}.get(args.kernel, None) if args.kernel in ("tuned", "v1") else int(args.kernel))

    # -- seeding on the device (k_seed_locate), timed separately ------------------------------
    eng.set_locate_grid(g["latT"], g["lonT"], g["ResKM"])
    SC_t = torch.from_numpy(SC).to(dev)
    if SG is None:                                   # dense clouds: lat/lon from our own inverse projection
        SG_t = torch.empty_like(SC_t)
        sit._lib.check(eng.L.st_xy2latlon_dev(SC_t.shape[0], SC_t.data_ptr(), SG_t.data_ptr(), 70.0, -45.0,
                                              torch.cuda.current_stream().cuda_stream))
        SG_t[:, 1] = torch.remainder(SG_t[:, 1], 360.0)
    else:
        SG_t = torch.from_numpy(SG).to(dev)
    ic0_t = torch.from_numpy(IC[0]).to(dev)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    cell_t, near_t, keep_t = eng.seed_locate_dev(SG_t, SC_t, ic0_t)
    e1.record(); torch.cuda.synchronize()
    seed_ms = e0.elapsed_time(e1)
    pos0_t, cell0_t = eng.seed_compact_dev(SC_t, cell_t, keep_t)     # SeedInit's shrink to the kept seeds, on the device
    pos0_t, cell0_t = pos0_t.contiguous(), cell0_t.contiguous()
    nP = int(pos0_t.shape[0])
    if not args.no_shuffle:
        # the synthetic generator emits the cloud cell by cell; hand it to the product in RANDOM order, so that the
        # gather locality of the step comes from the product (set_buoys(sort=True): cell-major storage) and not from
        # the way the input happened to be generated
        gen = torch.Generator(device=dev); gen.manual_seed(11 + rank)
        shuf = torch.randperm(nP, device=dev, generator=gen)
        pos0_t, cell0_t = pos0_t[shuf].contiguous(), cell0_t[shuf].contiguous()
        del shuf
    log("[rank %d] seeding: %d of %d seeds kept, k_seed_locate %.2f ms (%.3g buoys/s)"
        % (rank, nP, SC_t.shape[0], seed_ms, SC_t.shape[0] / (seed_ms * 1e-3)))
    del SG_t, near_t, keep_t, cell_t

    # -- records resident in HBM --------------------------------------------------------------
    eng.record_slots(R)
    for r in range(R):
        st = eng.staging(r)
        st[0], st[1], st[2] = U[r], V[r], IC[r]
        eng.submit_record(r)
    torch.cuda.synchronize()

    # the f8 row of record k is the position input of record k+1, as xPosC[jt] is in the reference: the two row buffers
    # below alternate, so the previous row is intact while the next one is written (st_set_row_chain)
    eng.set_row_chain(not args.no_chain)
    NB = 2
    NBV = max(1, min(NB, args.row_buffers))          # row buffers of the value loop (1: the rows are stepped in place)
    o_yx = [torch.empty((nP, 2), dtype=torch.float64, device=dev) for _ in range(NB)]
    o_ll = [torch.empty((nP, 2), dtype=torch.float64, device=dev) for _ in range(NB)]
    o_mk = [torch.empty((nP,), dtype=torch.int8, device=dev) for _ in range(NB)]
    stream = torch.cuda.Stream(dev)

    def reset(sort=True):
        eng.set_buoys_dev(pos0_t, cell0_t, stream=stream, sort=sort and not args.no_shuffle)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def ll_of(b):                    # --no-latlon: diagnostic run without the lat/lon row (not a bench value)
        return None if args.no_latlon else o_ll[b]

    def timed_steps(nsteps, nwarm, after_step=None, sort=True):
        """-> (ms, alive buoy-steps in the timed part).  after_step(k, buf) may enqueue extra work."""
        reset(sort)
        na = torch.zeros((nwarm + nsteps,), dtype=torch.int64, device=dev)
        for k in range(nwarm):
            b = k % NBV
            eng.step(k % R, k, o_yx[b], ll_of(b), o_mk[b], na[k:k + 1], stream)
            if after_step:
                after_step(k, b)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for k in range(nwarm, nwarm + nsteps):
            b = k % NBV
            eng.step(k % R, k, o_yx[b], ll_of(b), o_mk[b], na[k:k + 1], stream)
            if after_step:
                after_step(k, b)
        t1.record(stream)
        barrier()
        launches["n"] = nsteps
        launches["n_alive"] = na[nwarm:]
        return t0.elapsed_time(t1), int(na[nwarm:].sum().item())

    # -- value: K steps, records and state resident in HBM --------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    ms, bsteps = timed_steps(K, W)
    gpu_launches = launches["n"]                      # k_advect_step launches inside the timed region
    sampler.stop()
    clocks = sampler.summary()
    if args.dump_outputs and rank == 0:
        b = (W + K - 1) % NBV                         # the row buffers of the last timed step
        dump_outputs(args.dump_outputs, o_yx[b], ll_of(b), o_mk[b], launches["n_alive"], eng.perm_t)

    def reduce_max_sum(ms_, bs_):
        if world == 1:
            return ms_, bs_
        t = torch.tensor([ms_], dtype=torch.float64, device=dev)
        s = torch.tensor([bs_], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        return float(t.item()), int(s.item())

    ms_max, bsteps_all = reduce_max_sum(ms, bsteps)
    value = bsteps_all / (ms_max * 1e-3)
    peak, peak_src = measured_peak()
    # roofline of the dominant kernel on THIS rank: algorithmic bytes / its mean launch duration.
    # The K launches run back to back on one stream, so the event span / K is the launch duration.
    achieved = (bsteps / K) * B_ALG / (ms / K * 1e-3) / 1e9
    MOVED = 58.0 if (not args.no_chain and args.kernel in ("tuned", "0", "2", "3", "5")) else 74.0
    roof = {"bound": "hbm", "kernel": "k_advect_step_v1<1,false>" if args.kernel == "v1" else (("k_advect_warp<1,false,0,1,32,32>" if args.no_chain else "k_advect_warp<1,false,2,1,32,32>") if args.kernel == "tuned" else "step variant %s" % args.kernel), "achieved": round(achieved, 1), "peak": peak,
            "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": ncu_traffic(args.workload),
            "peak_source": peak_src, "alg_bytes_per_buoy_step": B_ALG,
            # what this build moves per buoy-step: 24 B of state in (position, cell; the alive flag is bit 31 of the cell
            # word), the 33 B row, ~1 B of cell rewrites (13 % of the buoys change cell) and, without row chaining, the
            # 16 B position write-back of the state; `frac` stays on SURVEY 8(d)'s 83 B
            "moved_bytes_per_buoy_step": MOVED,
            "frac_of_moved_bytes": round(achieved / B_ALG * MOVED / peak, 4),
            "buoy_steps_per_launch": bsteps / K, "us_per_launch": round(ms / K * 1e3, 2)}

    extra = {}
    # -- what the product's cell-major storage buys: the same shuffled input stored as it came ----------------
    if not args.no_shuffle and nP > 100_000:
        Ku = max(3, min(K, 20))
        ms_u, bs_u = timed_steps(Ku, 3, sort=False)
        ms_u, bs_u = reduce_max_sum(ms_u, bs_u)
        extra["input_order"] = {"what": "the seeds reach the product in random order; value/roofline: stored cell-major by "
                                        "set_buoys(sort=True) (stable sort by host cell, once per run); here: the same input "
                                        "stored in the order it came (sort=False)",
                                "us_per_launch_sorted_by_product": round(ms_max / K * 1e3, 2),
                                "us_per_launch_unsorted": round(ms_u / Ku * 1e3, 2), "steps_unsorted": Ku}
    # -- small clouds: the season path, R resident records per launch of k_advect_multi -----------
    if wl["grid"] == "nanuk4" or args.multi or (strong and nP < 2_000_000):
        Rm = args.multi or R
        rec_t = torch.from_numpy(np.stack([U, V, IC], axis=1).astype(np.float32)).to(dev).contiguous()[:Rm]
        m_yx = torch.empty((Rm, nP, 2), dtype=torch.float64, device=dev)
        m_ll = torch.empty((Rm, nP, 2), dtype=torch.float64, device=dev)
        m_mk = torch.empty((Rm, nP), dtype=torch.int8, device=dev)
        nl = max(3, min(50, K // Rm))
        m_na = torch.zeros((nl + 3, Rm), dtype=torch.int64, device=dev)
        reset()
        for i in range(3):
            eng.step_multi(rec_t, i * Rm, m_yx, m_ll, m_mk, m_na[i], stream)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for i in range(3, 3 + nl):
            eng.step_multi(rec_t, i * Rm, m_yx, m_ll, m_mk, m_na[i], stream)
        t1.record(stream)
        barrier()
        ms_m, bs_m = reduce_max_sum(t0.elapsed_time(t1), int(m_na[3:].sum().item()))
        extra["season_path"] = {"value": bs_m / (ms_m * 1e-3), "unit": "buoy-steps/s", "records_per_launch": Rm,
                                "launches": nl, "us_per_record": round(ms_m * 1e3 / (nl * Rm), 3),
                                "what": "k_advect_multi: each thread runs its buoy through %d resident records "
                                        "per launch, trajectory rows written every record" % Rm}
        del rec_t, m_yx, m_ll, m_mk
    # -- optional: the same loop with the per-record NCCL all-gather of positions ----------------
    if world > 1 and not args.no_allgather:
        comm = torch.cuda.Stream(dev)
        gathered = torch.empty((world * nP_max(nP, dist, dev), 2), dtype=torch.float64, device=dev)
        npad = gathered.shape[0] // world
        send = [torch.zeros((npad, 2), dtype=torch.float64, device=dev) for _ in range(NB)]
        evs = [None] * NB

        def ag(k, b):
            ev = torch.cuda.Event(); ev.record(stream)
            comm.wait_event(ev)
            with torch.cuda.stream(comm):
                send[b][:nP].copy_(o_yx[b], non_blocking=True)
                dist.all_gather_into_tensor(gathered, send[b])
                evs[b] = torch.cuda.Event(); evs[b].record(comm)
            nb = (k + 1) % NB
            if evs[nb] is not None:
                stream.wait_event(evs[nb])          # the buffer the next step overwrites has been sent
        Ka = max(4, min(K, 200))
        ms_a, bs_a = timed_steps(Ka, min(W, 5), after_step=ag)
        torch.cuda.synchronize()
        ms_a, bs_a = reduce_max_sum(ms_a, bs_a)
        extra["allgather"] = {"value": bs_a / (ms_a * 1e-3), "unit": "buoy-steps/s", "steps": Ka,
                              "bytes_per_rank_per_step": int(npad * 16), "what": "k_advect_step + NCCL "
                              "all_gather_into_tensor of (y,x) f8 per record on a side stream"}

    # -- the same loop with the all-gather FUSED into the step kernel (stores into every rank's gathered
    #    array over NVLink peer memory; st_step_gather) ---------------------------------------------
    if world > 1 and not args.no_allgather:
        cnt = torch.zeros((world,), dtype=torch.int64, device=dev)
        cnt[rank] = nP
        dist.all_reduce(cnt)
        cnts = cnt.cpu().numpy()
        offs = np.concatenate([[0], np.cumsum(cnts)])
        # every rank's block starts on a tile boundary of the gathered array (the bulk form needs 16-byte aligned tiles)
        offs = np.concatenate([[0], np.cumsum((cnts + 31) // 32 * 32)])
        checks = {}
        forms = (("allgather_fused", False, 0), ("allgather_fused_f4", True, 0), ("allgather_bulk_f4", True, 2),
                 ("allgather_dma_f4", True, 1), ("allgather_bulk", False, 2))
        for tag, f4, mode in forms:
            reset(); torch.cuda.synchronize()
            hnd = eng.gather_create(rank, world, int(offs[-1]), int(offs[rank]), f4=f4, nbuf=NB)
            mine = torch.tensor(list(hnd), dtype=torch.uint8, device=dev)
            allh = torch.empty((world * 64,), dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allh, mine)
            eng.gather_connect_ipc(bytes(allh.cpu().numpy().tobytes()))
            eng.gather_set_mode(mode)
            barrier()
            cons = torch.cuda.Stream(dev)
            Ka = max(4, min(K, 200)); Wa = min(W, 5)
            na_g = torch.zeros((Wa + Ka + 1,), dtype=torch.int64, device=dev)

            def gsteps(k0, n):
                for k in range(k0, k0 + n):
                    b = k % NB
                    eng.step_gather(k % R, k, b, k + 1, ll_of(b), o_mk[b], na_g[k:k + 1], stream)
                    eng.gather_wait(k + 1, cons)        # the consumer stream sees the whole gathered row ...
                    eng.gather_ack(k + 1, cons)         # ... and frees the buffer for sequence k + 1 + NB
            # parity of the exchange (driver-visible on real peers): the first gathered row against every rank's own
            # row of the same record from the plain step, collected with NCCL
            eng.step_gather(0, 0, 0, 1, ll_of(0), o_mk[0], na_g[Wa + Ka:], stream)
            eng.gather_wait(1, cons)
            cons.synchronize()
            got = eng.gather_buffer(0).clone()
            eng.gather_ack(1, cons)
            barrier()
            reset()
            eng.step(0, 0, o_yx[0], ll_of(0), o_mk[0], na_g[Wa + Ka:], stream)
            stream.synchronize()
            sendc = torch.zeros((npad, 2), dtype=torch.float64, device=dev)
            sendc[:nP] = o_yx[0]
            allc = torch.empty((world * npad, 2), dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(allc, sendc)
            ok = True
            for r in range(world):
                ref_r = allc[r * npad: r * npad + int(cnts[r])]
                ref_r = ref_r.to(torch.float32) if f4 else ref_r
                ok = ok and bool(torch.equal(got[int(offs[r]): int(offs[r]) + int(cnts[r])], ref_r))
            okt = torch.tensor([int(ok)], device=dev); dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            checks[tag] = "bit-identical on all %d ranks" % world if int(okt.item()) else "MISMATCH"
            if not int(okt.item()):
                log("[rank %d] gather check FAILED for %s" % (rank, tag))
            del got, sendc, allc
            # the gather protocol restarts from sequence 1 with fresh flags
            eng.gather_destroy(); barrier()
            reset(); torch.cuda.synchronize()
            hnd = eng.gather_create(rank, world, int(offs[-1]), int(offs[rank]), f4=f4, nbuf=NB)
            mine = torch.tensor(list(hnd), dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allh, mine)
            eng.gather_connect_ipc(bytes(allh.cpu().numpy().tobytes()))
            eng.gather_set_mode(mode)
            barrier()
            gsteps(0, Wa)
            barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(stream)
            gsteps(Wa, Ka)
            t1.record(stream)
            ec = torch.cuda.Event(enable_timing=True); ec.record(cons)
            barrier()
            ms_g = max(t0.elapsed_time(t1), t0.elapsed_time(ec))     # until the last row has LANDED here too
            bad = eng.gather_timed_out()
            ms_g, bs_g = reduce_max_sum(ms_g, int(na_g[Wa:Wa + Ka].sum().item()))
            into = int((offs[-1] - cnts[rank]) * (8 if f4 else 16))
            how = {0: "k_advect_warp stores every new (y,x) %s into the gathered array of all %d ranks itself "
                      "(one NVLink peer store per thread per peer, ready/ack flags, no NCCL call)",
                   1: "k_advect_warp writes its own block of (y,x) %s; one peer-to-peer copy per peer on the copy engines "
                      "pushes it into the gathered arrays of all %d ranks (ready/ack flags, no NCCL call)",
                   2: "k_advect_warp stages each tile of 32 (y,x) %s in shared memory and sends it to each of the %d ranks "
                      "with one cp.async.bulk (peer order rotating per tile; ready/ack flags, no NCCL call)"}[mode]
            extra[tag] = {"value": bs_g / (ms_g * 1e-3), "unit": "buoy-steps/s", "steps": Ka,
                          "ms_per_step": round(ms_g / Ka, 4),
                          "bytes_into_each_rank_per_step": into,
                          "ingress_gb_s": round(into / (ms_g / Ka * 1e-3) / 1e9, 1),
                          "timed_out": bool(bad), "check": checks[tag],
                          "what": how % ("f4" if f4 else "f8", world)}
            barrier()
            eng.gather_destroy()
            barrier()
        # config 5 as BASELINE.json states it: every position on every GPU after every record
        forms_done = [t for t in ("allgather", "allgather_fused", "allgather_bulk", "allgather_fused_f4",
                                  "allgather_bulk_f4", "allgather_dma_f4") if t in extra and not extra[t].get("timed_out")]
        if forms_done:
            best = max(forms_done, key=lambda t: extra[t]["value"])
            best8 = max([t for t in forms_done if not t.endswith("_f4")], key=lambda t: extra[t]["value"])
            extra["with_allgather"] = {
                "what": "BASELINE config 5 as stated: the per-record all-gather of positions inside the timed loop. "
                        "`value` (above) is the same loop without the exchange.",
                "best_form": best, "value": extra[best]["value"], "value_f8_positions": extra[best8]["value"],
                "best_form_f8": best8, "unit": "buoy-steps/s",
                "fraction_of_no_exchange_value": round(extra[best]["value"] / value, 4)}

    # -- e2e: host buffers in, host rows out, every step (pinned memory, 3 streams) ---------------
    Ke = args.e2e_steps if args.e2e_steps > 0 else max(4, min(K, 40 if nP > 2_000_000 else 200))
    h_rec = torch.from_numpy(np.stack([U, V, IC], axis=1).astype(np.float32)).pin_memory()   # (R,3,Nj,Ni)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    checksum = [0.0]
    na_e = [None]

    def e2e_run(rdt):
        """-> (seconds, alive buoy-steps) of Ke timed steps with rows of dtype rdt through host buffers."""
        h_yx = [torch.empty((nP, 2), dtype=rdt).pin_memory() for _ in range(NB)]
        h_ll = [torch.empty((nP, 2), dtype=rdt).pin_memory() for _ in range(NB)]
        h_mk = [torch.empty((nP,), dtype=torch.int8).pin_memory() for _ in range(NB)]
        d_yx = o_yx if rdt == torch.float64 else [torch.empty((nP, 2), dtype=rdt, device=dev) for _ in range(NB)]
        d_ll = o_ll if rdt == torch.float64 else [torch.empty((nP, 2), dtype=rdt, device=dev) for _ in range(NB)]

        def e2e_loop(n, k0):
            ev_in, ev_st, ev_out = {}, {}, {}
            for k in range(k0, k0 + n):
                b = k % 2
                if k - 2 in ev_st:
                    s_in.wait_event(ev_st[k - 2])                       # device slot b free again
                eng.upload_record(b, h_rec[k % R], s_in)                # H2D of this step's inputs
                ev_in[k] = torch.cuda.Event(); ev_in[k].record(s_in)
                stream.wait_event(ev_in[k])
                if k - NB in ev_out:
                    stream.wait_event(ev_out[k - NB])                   # device out buffer b drained
                eng.step(b, k, d_yx[b], d_ll[b], o_mk[b], na_e[0][k:k + 1], stream)
                ev_st[k] = torch.cuda.Event(); ev_st[k].record(stream)
                s_out.wait_event(ev_st[k])
                if k - NB in ev_out:
                    ev_out[k - NB].synchronize()                        # host row buffer b consumed
                    checksum[0] += float(h_yx[b][0, 0])                 # the host reads the result
                with torch.cuda.stream(s_out):
                    h_yx[b].copy_(d_yx[b], non_blocking=True)           # D2H of the trajectory row
                    h_ll[b].copy_(d_ll[b], non_blocking=True)
                    h_mk[b].copy_(o_mk[b], non_blocking=True)
                ev_out[k] = torch.cuda.Event(); ev_out[k].record(s_out)
            torch.cuda.synchronize()

        reset(); eng.record_slots(max(R, 2))
        na_e[0] = torch.zeros((Ke + 3,), dtype=torch.int64, device=dev)
        e2e_loop(min(3, Ke), 0)
        barrier()
        t0 = time.perf_counter()
        e2e_loop(Ke, 3)
        barrier()
        sec = time.perf_counter() - t0
        bs = float(na_e[0][3:].sum().item())                            # alive buoys advanced in the timed steps
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev); s_ = torch.tensor([bs], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(s_, op=dist.ReduceOp.SUM)
            sec, bs = float(t.item()), float(s_.item())
        return sec, bs

    # the end-to-end figure is what the command line does: rows leave the GPU in the dtype the reference's output
    # files store (st_step_f4; ncio.py:153-159: every trajectory variable is f4), 17 B per buoy
    f4_s, f4_bs = e2e_run(torch.float32)
    e2e = {"value": f4_bs / f4_s, "unit": "buoy-steps/s", "h2d_bytes_per_step": int(3 * Nj * Ni * 4),
           "d2h_bytes_per_step": int(17 * nP), "steps": Ke, "ms_per_step": round(f4_s / Ke * 1e3, 3),
           "what": "per record: pinned host u/v/siconc -> st_upload_record -> st_step_f4 -> trajectory row "
                   "(y,x,lat,lon f4 + mask i1: the output file's dtypes) copied to pinned host memory and read"}
    e2e_s, e2e_bs = e2e_run(torch.float64)
    extra["e2e_f8_rows"] = {"value": e2e_bs / e2e_s, "unit": "buoy-steps/s", "h2d_bytes_per_step": int(3 * Nj * Ni * 4),
                            "d2h_bytes_per_step": int(D2H_PER_BUOY * nP), "steps": Ke, "ms_per_step": round(e2e_s / Ke * 1e3, 3),
                            "what": "as e2e with the rows as (y,x,lat,lon) f8 + mask, the reference's in-memory arrays"}

    # -- CPU baseline on this box's host cores (rank 0, N=1 only) ---------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        pos0 = pos0_t.cpu().numpy(); cell0 = cell0_t.cpu().numpy()
        cpu = cpu_baseline(g, (U, V, IC), pos0, cell0, args)

    if rank == 0:
        out = {"metric": "buoy-steps/sec", "value": value, "unit": "buoy-steps/s", "n_gpus": world, "steps": K,
               "warmup": W, "ms_per_step": round(ms_max / K, 5), "higher_is_better": True,
               "scaling": "strong" if strong else "weak",
               "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": {"workload": wl["label"], "buoys_per_gpu": nP, "grid": [Nj, Ni],
                          "records_resident": R, "uv_strategy": 1, "rdt_s": 3600,
                          "l2": "inputs larger than L2: per step %.0f MB of buoy state + trajectory rows stream "
                                "through, %d resident records (%.0f MB) are cycled; no flush"
                                % (nP * B_ALG / 1e6, R, R * 3 * Nj * Ni * 4 / 1e6),
                          "input_order": "as generated (cell-major)" if args.no_shuffle else
                                         "random (shuffled); stored cell-major by the product (set_buoys sort)",
                          "state": "separate position state, rewritten every record" if args.no_chain else
                                   "positions chained through the f8 trajectory rows (st_set_row_chain)",
                          "parallelism": "buoys sharded over %d GPU(s), record replicated" % world},
               "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": gpu_launches,
               "clocks": clocks, "seed_locate": {"buoys_per_s": SC_t.shape[0] / (seed_ms * 1e-3), "ms": round(seed_ms, 3)}}
        out.update(extra)
        emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _physical_index(local):
    """NVML counts physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain index list."""
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except (ValueError, IndexError):
            return local
    return local


def nP_max(nP, dist, dev):
    import torch
    t = torch.tensor([nP], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return int(t.item())


def dump_outputs(out_dir, yx, latlon, mask, n_alive, perm=None):
    """What a caller of st_step receives from the last timed step, for comparing two builds output for output:
    the trajectory row (y,x km and lat,lon degrees, f8; the mask as f4) of a fixed sample of at most DUMP_BUOYS
    buoys, that sample's indices in the order the buoys were handed to the product, and the alive count of
    every timed step (f8).  perm: the engine's storage order (set_buoys_dev(sort=True) keeps the rows cell-major,
    row r is buoy perm[r]); the sample is read back in the caller's order, so that it does not depend on how the
    product lays the buoys out."""
    import torch
    nP = yx.shape[0]
    if nP > DUMP_BUOYS:
        idx = np.sort(np.random.default_rng(0).choice(nP, DUMP_BUOYS, replace=False))
    else:
        idx = np.arange(nP)
    rows = torch.from_numpy(idx).to(yx.device)
    if perm is not None:                                # the caller's buoy i is stored in row inv[i]
        inv = torch.empty_like(perm)
        inv[perm] = torch.arange(nP, device=perm.device, dtype=perm.dtype)
        rows = inv.index_select(0, rows)
    out = {"buoy": idx.astype(np.float64),
           "yx": yx.index_select(0, rows).cpu().numpy(),
           "mask": mask.index_select(0, rows).cpu().numpy().astype(np.float32),
           "n_alive": n_alive.cpu().numpy().astype(np.float64)}
    if latlon is not None:
        out["latlon"] = latlon.index_select(0, rows).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log("outputs of the last timed step: %s in %s (%.1f MB)"
        % (", ".join(sorted(out)), out_dir, sum(a.nbytes for a in out.values()) / 1e6))


# ---------------------------------------------------------------------------------------------
# CPU baselines (oracle/ is only ever the thing timed here, never on the product path)
# ---------------------------------------------------------------------------------------------
class _PyShard:
    """One shard of buoys advanced by the reference's interpreted loop (oracle/pyport.py), one record per call,
    followed like upstream by the conversion of the whole new row to lat/lon (si3_part_tracker.py:493; the
    reference calls PROJ, compiled C, through cartopy -- here the oracle's C restatement of it)."""

    def __init__(self, g, recs64, pos, cell):
        nP = pos.shape[0]
        self.g, self.recs64 = g, recs64
        self.cur = pos.copy(); self.nxt = np.empty_like(self.cur); self.m = np.zeros(nP, 'i1')
        self.jiT = cell.astype(int).copy(); self.alive = np.ones(nP, 'i1')
        self.first = np.zeros(nP, int); self.last = np.zeros(nP, int) + 10 ** 9
        self.vM = np.zeros((nP, 4, 2)); self.sin_ = np.zeros(nP, bool)

    def record(self, k):
        from oracle import pyport, corc
        xU, xV, xIC = self.recs64[k % len(self.recs64)]
        self.nxt[:] = pyport.FILL                                   # :327, rows of discontinued buoys stay at the fill value
        n = pyport.advance(self.g, xU, xV, xIC, k, self.cur, self.nxt, self.m, self.jiT, self.alive, self.first,
                           self.last, self.vM, self.sin_)
        corc.inv_stere(self.nxt)                                    # :493, every row, dead ones included
        self.cur, self.nxt = self.nxt, self.cur
        return n


def _py_sample_run(g, recs64, pos, cell, nrec):
    sh = _PyShard(g, recs64, pos, cell)
    n = 0
    t0 = time.perf_counter()
    for k in range(nrec):
        n += sh.record(k)
    return n, time.perf_counter() - t0


def cpu_baseline(g, recs, pos0, cell0, args):
    """Pure-Python port (the reference's execution model) on 1 core + the C oracle on all cores,
    both on a bounded random sub-sample of the same workload."""
    from oracle import corc
    U, V, IC = recs
    rng = np.random.default_rng(7)
    nP = pos0.shape[0]
    npy = min(nP, args.cpu_sample)
    sel = np.sort(rng.choice(nP, npy, replace=False))
    recs64 = [(U[k].astype(np.float64), V[k].astype(np.float64), IC[k].astype(np.float64)) for k in range(U.shape[0])]
    n, dt = _py_sample_run(g, recs64, pos0[sel], cell0[sel], args.cpu_records)
    out = {"value": n / dt, "unit": "buoy-steps/s", "cores": 1, "kind": "port",
           "sample": "oracle/pyport.py (interpreted Python like the reference, lat/lon conversion of every row included) "
                     "on %d random buoys of the workload x %d records, %.1f s" % (npy, args.cpu_records, dt)}
    nc = min(nP, 200_000)
    selc = np.sort(rng.choice(nP, nc, replace=False))
    nrc = 24
    Uc = np.concatenate([U] * (nrc // U.shape[0] + 1))[:nrc]; Vc = np.concatenate([V] * (nrc // U.shape[0] + 1))[:nrc]
    Ic = np.concatenate([IC] * (nrc // U.shape[0] + 1))[:nrc]
    t0 = time.perf_counter()
    r = corc.track(g, Uc, Vc, Ic, pos0[selc], cell0[selc].astype(np.int64), history=False)
    dtc = time.perf_counter() - t0
    out["c_oracle"] = {"value": float(r["mask"][1:].sum()) / dtc, "unit": "buoy-steps/s", "cores": os.cpu_count(),
                       "sample": "oracle/st_oracle.c (OpenMP over buoys) on %d buoys x %d records incl. lat/lon, %.2f s"
                                 % (nc, nrc, dtc)}
    return out


def _ref_worker(conn, barrier, g, recs64, pos, cell, W, K):
    """W warm-up records, a barrier, then K timed records without talking to the parent; reports once."""
    sh = _PyShard(g, recs64, pos, cell)
    for k in range(W):
        sh.record(k)
    barrier.wait()
    t0 = time.perf_counter()                                       # CLOCK_MONOTONIC: comparable across processes
    n = 0
    for k in range(W, W + K):
        n += sh.record(k)
    conn.send((n, t0, time.perf_counter()))


def run_reference(args):
    """The reference's CPU implementation of the path (interpreted Python; oracle/pyport.py is its
    pinned port because /root/reference cannot travel to the GPU box) on all host cores: buoys are
    independent, so each worker process owns a shard of a bounded sample of the same workload and runs the
    whole W + K record loop on its own (one message back at the end).  The sample is sized for at least
    ~2 s of timed work per worker: max(--ref-buoys-per-core, 140000 / K) buoys each."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    wl = WORKLOADS[args.workload]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per = max(args.ref_buoys_per_core, -(-140000 // max(K, 1)))
    dense = wl["kind"] == "dense"
    g, (U, V, IC), SG, SC = build_workload(args.workload, 0, want_latlon_grid=not dense,
                                           n_dense=cores * per if dense else None, keep_cells=True)
    g.pop("warp", None)
    from oracle import corc
    rng = np.random.default_rng(7)
    if dense:
        # the synthetic cloud is generated cell by cell: the cell of origin is the host cell; the oracle's
        # inside test confirms it buoy by buoy
        pos, cell = SC, g.pop("seed_cells").astype(np.int64)
    else:
        n = SC.shape[0]
        cell = np.zeros((n, 2), np.int64)
        for b in range(n):
            cell[b] = _guess_cell(g, SC[b])
        pos = SC
    n = pos.shape[0]
    ok = np.zeros(n, bool)
    for b in range(n):
        j, i = int(cell[b, 0]), int(cell[b, 1])
        if 2 <= j <= g["Nj"] - 3 and 2 <= i <= g["Ni"] - 3:
            ok[b], cell[b, 0], cell[b, 1] = corc.find_containing_cell(pos[b, 0], pos[b, 1], j, i, g["Yf"], g["Xf"])
    pos, cell = pos[ok], cell[ok]
    n = pos.shape[0]
    recs64 = [(U[k].astype(np.float64), V[k].astype(np.float64), IC[k].astype(np.float64)) for k in range(U.shape[0])]
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(cores)
    perm = rng.permutation(n)                                     # every worker gets a spatially mixed shard
    shards = np.array_split(perm, cores)
    procs, conns = [], []
    for sh in shards:
        a, b = ctx.Pipe()
        p = ctx.Process(target=_ref_worker, args=(b, barrier, g, recs64, pos[sh], cell[sh], W, K), daemon=True)
        p.start(); procs.append(p); conns.append(a)
    res = [c.recv() for c in conns]
    for p in procs:
        p.join(timeout=10)
    done = sum(r[0] for r in res)
    dt = max(r[2] for r in res) - min(r[1] for r in res)
    value = done / dt
    per_core = [r[0] / (r[2] - r[1]) for r in res]
    sample = ("oracle/pyport.py (pinned port of the reference's interpreted loop, lat/lon conversion of every row "
              "included) on %d host processes, %d buoys of the workload (bounded sample, %d per process), %d records "
              "in %.1f s; %.0f buoy-steps/s per process (min %.0f, max %.0f)"
              % (cores, n, n // cores, K, dt, value / cores, min(per_core), max(per_core)))
    out = {"impl": "reference", "metric": "buoy-steps/sec", "value": value, "unit": "buoy-steps/s",
           "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": round(dt / K * 1e3, 4),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": wl["label"], "grid": [g["Nj"], g["Ni"]], "sample_buoys": n},
           "cpu_baseline": {"value": value, "unit": "buoy-steps/s", "cores": cores, "kind": "port", "sample": sample,
                            "per_core": value / cores},
           "e2e": {"value": value, "unit": "buoy-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


def _guess_cell(g, p):
    """Coarse-to-fine nearest T-point in the km plane (input preparation for the CPU arm only)."""
    Yt, Xt = g["Yt"], g["Xt"]
    st = 16
    sub = (Yt[::st, ::st] - p[0]) ** 2 + (Xt[::st, ::st] - p[1]) ** 2
    j0, i0 = np.unravel_index(np.argmin(sub), sub.shape)
    j0, i0 = j0 * st, i0 * st
    ja, jb = max(j0 - 2 * st, 0), min(j0 + 2 * st + 1, Yt.shape[0])
    ia, ib = max(i0 - 2 * st, 0), min(i0 + 2 * st + 1, Yt.shape[1])
    d2 = (Yt[ja:jb, ia:ib] - p[0]) ** 2 + (Xt[ja:jb, ia:ib] - p[1]) ** 2
    j, i = np.unravel_index(np.argmin(d2), d2.shape)
    return j + ja, i + ia


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=list(WORKLOADS))
    ap.add_argument("--kernel", default="tuned", help="k_advect_step variant: tuned, v1, or an integer launch-bound experiment")
    ap.add_argument("--e2e-steps", type=int, default=0)
    ap.add_argument("--no-latlon", action="store_true", help="diagnostic: skip the lat/lon row in the value loop")
    ap.add_argument("--multi", type=int, default=0, help="also time k_advect_multi with this many records per launch")
    ap.add_argument("--no-allgather", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: the workload's buoy count is the TOTAL, sharded over the ranks (config 4: --workload cfg4)")
    ap.add_argument("--row-buffers", type=int, default=2, help="device row buffers the value loop cycles through (1: rows stepped in place)")
    ap.add_argument("--no-chain", action="store_true", help="A/B: keep a separate position state (st_set_row_chain off)")
    ap.add_argument("--no-shuffle", action="store_true", help="diagnostic: feed the seeds in generator (cell-major) order, no sort")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=2000, help="buoys in the Python cpu_baseline sample")
    ap.add_argument("--cpu-records", type=int, default=100)
    ap.add_argument("--ref-buoys-per-core", type=int, default=2000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's trajectory row (a fixed sample of at most "
                         "%d buoys, rank 0's shard) and the alive count of every timed step as DIR/<name>.npy"
                         % DUMP_BUOYS)
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        args.steps = 100 if args.steps is None else args.steps
        args.warmup = 3 if args.warmup is None else max(args.warmup, 1)
        run_reference(args)
    else:
        args.steps = 2000 if args.steps is None else args.steps
        args.warmup = 20 if args.warmup is None else max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
