#!/usr/bin/env python
"""bench.py — benchmark of the LM-CMA trajectory-optimisation hot path (BASELINE.json metric: trajectory-cost evals/s +
LM-CMA generations/s at 1/2/4/8 B200).

Headline (`value`, `e2e`, `roofline`): the C2 workload — one 2-D query on a 4096x4096 synthetic occupancy grid, 200
waypoints (n = 400), lambda = 1024, m = 2*sqrt(n) = 40.  A "step" is ONE LM-CMA generation = k_cost (lambda trajectory
evaluations) -> k_rank -> k_update -> k_sample, replayed from a CUDA graph.  The optimiser is first advanced m + 5
generations untimed so that all m direction pairs are live (steady state of the sampler and of the update), then K
generations are timed with L2 flushed (256 MiB write) before every one.  N > 1: every rank optimises its own independent
C2 query (weak scaling, no data-path collective: SURVEY.md section 8e).

The same line also carries the two multi-GPU modes BASELINE.json names:
  c3_sharded : 4096 independent queries x lambda 64 on the C2 map, sharded contiguously over the ranks
               (parallel.shard_range), no collective — strong scaling; at N > 1 rank 0 also runs all 4096 alone so that
               the efficiency is printed from one run.
  c4_split   : ONE population lambda = 8192, n = 1500, m = 77 on a 512^3 u8 voxel map, offspring split over the ranks,
               two small NCCL all-gathers per generation (lambda fitness scalars, then (n + 4) floats per rank), the
               generation captured in one CUDA graph; with the 1-GPU whole-population time beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--skip c3,c4,cpu] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = {"workload": "C2: 2-D 4096x4096 synthetic occupancy grid (seed 42, 2048 rectangles), one query "
                        "(64,64)->(4032,4032), 200 waypoints (n=400), lambda=1024, m=40, sigma0=32, longsafe weights",
            "map": "4096x4096 f32 sign-tagged reciprocal clearance (64 MiB)", "n": 400, "lambda": 1024, "m": 40,
            "waypoints": 200}
W, LAM, M, SIGMA0 = 200, 1024, 40, 32.0
FILL = M + 5                       # untimed generations in front of the timed region: every direction pair live
FP32_FMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # SURVEY 8d: 148 SMs x 128 lanes x 2 flop x 1.965 GHz = 74.4
# dram__bytes_read.sum + dram__bytes_write.sum of one k_cost launch of this workload, from the committed
# `ncu --set full` capture (the map stays L2-resident between generations, so DRAM traffic is far BELOW the
# algorithmic bytes: the kernel is bound by the L1 line rate of the gather, not by HBM)
NCU_DRAM_BYTES_PER_LAUNCH = 2.393e6
NCU_SOURCE = "profiles/r2n_full.md (k_cost<2,0,0,7>: dram_read 2.393 MB, dram_write 0)"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_problem():
    from lmcma_path_planner_b200 import maps
    dist, start, goal = maps.config2_map()
    lo, hi = maps.box_bounds((4096, 4096), W)
    x0 = maps.straight_line(start, goal, W)
    return dist, start, goal, lo, hi, x0


def sampler_roofline(n, lam, live, ms, peak_gbs):
    """SURVEY 8d: the sampler against BOTH rooflines.  flops = 4 lambda m n + 2 lambda n; bytes = 4 n (lambda + 2 m) +
    4 (2 n + m) (device RNG: no Z read; V and P once, X written once)."""
    flops = 4.0 * lam * live * n + 2.0 * lam * n
    nbytes = 4.0 * n * (lam + 2 * live) + 4.0 * (2 * n + live)
    t = ms * 1e-3
    return {"kernel": "k_sample", "launch_ms": ms, "live_pairs": live,
            "fma": {"achieved": flops / t / 1e12, "peak": FP32_FMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": flops / t / 1e12 / FP32_FMA_PEAK_TFLOPS,
                    "flops_per_launch": flops},
            "hbm": {"achieved": nbytes / t / 1e9, "peak": peak_gbs, "unit": "GB/s", "frac": nbytes / t / 1e9 / peak_gbs,
                    "algorithmic_bytes_per_launch": nbytes}}


def dump_outputs(path, opt):
    """What a caller of the timed generation holds after its last step (1.7 MB in all): the best path and cost so far,
    the population that generation sampled for the next one, the fitness and collision counts of the population it
    evaluated, and the mean and step size it updated.  The inputs are seeded, so two builds can be compared file by file."""
    os.makedirs(path, exist_ok=True)
    best_x, best_f = opt.best()
    arrays = {"best_x": best_x, "best_f": best_f, "X": opt.get("X"), "fit": opt.get("fit"),
              "ncoll": opt.get("ncoll").astype(np.float32), "xmean": opt.get("xmean"), "sigma": opt.get("sigma")}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_b200(args):
    import torch
    import lmcma_path_planner_b200 as L
    from lmcma_path_planner_b200 import _capi as K

    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(local)
    dist_pg = None
    if world > 1:
        import torch.distributed as dist_pg
        dist_pg.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist_pg is not None:
            dist_pg.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        if dist_pg is None:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist_pg.all_reduce(t, op=dist_pg.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]

    skip = set(args.skip.split(",")) if args.skip else set()
    dist, start, goal, lo, hi, x0 = build_problem()
    cmap = L.CostMap(dist, "f32", device=local)
    opt = L.Optimizer(2 * W, x0=x0, lam=LAM, m=M, lo=lo, hi=hi, sigma0=SIGMA0, seed=1000 + rank, rng="philox", device=local)
    opt.attach_cost(cmap, [start], [goal], W, L.LONGSAFE, 1e4)
    stream = torch.cuda.Stream()                     # a real (non-null) stream: the library enqueues on it
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    opt.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def one_step(timed):
        flush.fill_(1)                               # evict L2 (not timed)
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record(stream)
        opt.run(1, sync=False)
        e1.record(stream)
        return (e0, e1) if timed else None

    warm = max(args.warmup, 3)
    for _ in range(warm):
        one_step(False)
    opt.run(max(0, FILL - warm))                     # fill-up, untimed: all m pairs live from here on
    live0, sigma0 = int(opt.get("live")[0]), float(opt.get("sigma")[0])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = K.lib().lmcma_b200_launch_count()
    t_wall0 = time.perf_counter()
    evs = [one_step(True) for _ in range(args.steps)]
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = K.lib().lmcma_b200_launch_count() - launches0
    ms_total = sum(a.elapsed_time(b) for a, b in evs)
    nsamp_mean = float(opt.get("nsamp").mean())
    live1, sigma1 = int(opt.get("live")[0]), float(opt.get("sigma")[0])
    ncoll_best = int(opt.get("ncoll")[0].min())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, opt)

    # steady state: back-to-back graph replays, L2 warm (the deployment mode: the map stays L2-resident)
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record(stream)
    opt.run(args.steps, sync=False)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_warm = e0.elapsed_time(e1)

    # per-kernel durations (CUDA events around every kernel), same flush policy as the timed region
    per_kernel = {}
    nsamp_k = []
    for _ in range(3):                               # un-graphed launch path: first use loads these kernel variants
        opt.profile_kernels(1)
    for _ in range(args.steps):
        flush.fill_(1)
        pk = opt.profile_kernels(1)
        nsamp_k.append(float(opt.get("nsamp").mean()))
        for k, v in pk.items():
            per_kernel[k] = per_kernel.get(k, 0.0) + v / args.steps
    sigma2 = float(opt.get("sigma")[0])
    clocks = sampler.stop()

    # the whole planning run of SURVEY 8d (200 generations from the straight line, fill-up and convergence included)
    full = L.Optimizer(2 * W, x0=x0, lam=LAM, m=M, lo=lo, hi=hi, sigma0=SIGMA0, seed=3000 + rank, rng="philox", device=local)
    full.attach_cost(cmap, [start], [goal], W, L.LONGSAFE, 1e4)
    full.set_stream(stream.cuda_stream)
    full.run(200)                                    # last_run_ms: device time of the 200 graph replays
    full.sync()
    ms_full = full.last_run_ms()
    full_best = float(full.best()[1][0])
    full_sigma = float(full.get("sigma")[0])
    full.close()

    e2e = run_e2e(args, L, K, torch, cmap, start, goal, lo, hi, x0, rank, local, flush, barrier)
    ms_total, ms_warm, e2e_t, ms_full = max_over_ranks([ms_total, ms_warm, e2e["t"], ms_full])
    if dist_pg is not None:
        lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist_pg.all_reduce(lt)
        launches = int(lt.item())
    # the same C2 population through k_cost on the two map storages (stand-alone launches, CUDA events, L2 flushed): what the
    # bytes per cell do to a kernel whose gather is paced by the 128-byte lines a warp request touches (DESIGN.md 4.1)
    storage_ms = {}
    if "cpu" not in skip or "c3" not in skip:
        Xd = torch.from_numpy(np.ascontiguousarray(opt.get("X")[0])).cuda()
        fd = torch.empty(LAM, dtype=torch.float32, device="cuda")
        for storage in ("f32", "u8"):
            cm2 = cmap if storage == "f32" else L.CostMap(np.minimum(dist, 63.0), "u8", device=local)
            tot = 0.0
            for it in range(3 + min(args.steps, 20)):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
                e0.record(stream)
                cm2.evaluate_dev(Xd.data_ptr(), Xd.shape[1], LAM, fd.data_ptr(), start, goal, W, L.LONGSAFE, 1e4, stream=stream.cuda_stream)
                e1.record(stream)
                torch.cuda.synchronize()
                if it >= 3:
                    tot += e0.elapsed_time(e1)
            storage_ms[storage] = tot / min(args.steps, 20)
            if storage == "u8":
                cm2.close()
        del Xd, fd
    opt.close()

    peak, peak_src = peaks()
    c3 = None if "c3" in skip else run_c3(args, L, torch, dist_pg, dist, cmap, lo, hi, rank, world, local, stream, barrier, max_over_ranks, peak)
    cmap.close()
    c4 = None if "c4" in skip else run_c4(args, L, torch, dist_pg, rank, world, local, stream, barrier, max_over_ranks)

    out = None
    if rank == 0:
        ms_step = ms_total / args.steps
        evals_per_s = world * LAM * args.steps / (ms_total * 1e-3)
        # cost kernel roofline: algorithmic bytes per trajectory = 4n (candidate) + S*b (map samples) + 8 (f, flag)
        S = float(np.mean(nsamp_k)) if nsamp_k else nsamp_mean
        bytes_per_launch = LAM * (4 * 2 * W + S * cmap.bytes_per_cell + 8)
        cost_ms = per_kernel["cost"]
        achieved = bytes_per_launch / (cost_ms * 1e-3) / 1e9
        strict = LAM * (4 * 2 * W + 8) / (cost_ms * 1e-3) / 1e9
        out = {
            "metric": "trajectory-cost evals/s (LM-CMA generations/s = value / lambda)", "value": evals_per_s, "unit": "evals/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(WORKLOAD, parallelism="independent query per GPU (no collective)" if world > 1 else "1 GPU",
                           l2="flushed before every timed step (256 MiB fill)", rng="device Philox4x32-10",
                           untimed_generations_before_the_timed_region=max(warm, FILL),
                           live_pairs_in_timed_region=[live0, live1], sigma_in_timed_region=[sigma0, sigma1],
                           sigma_after_all_measurements=sigma2, mean_samples_per_trajectory=S,
                           min_collisions_in_last_population=ncoll_best),
            "generations_per_s": world * args.steps / (ms_total * 1e-3),
            "steady_state_l2_warm": {"value": world * LAM * args.steps / (ms_warm * 1e-3), "unit": "evals/s",
                                     "ms_per_step": ms_warm / args.steps,
                                     "note": "back-to-back graph replays, map L2-resident (deployment mode)"},
            "c2_full_planning_run": {"generations": 200, "ms_total": ms_full, "ms_per_generation": ms_full / 200,
                                     "value": world * LAM * 200 / (ms_full * 1e-3), "unit": "evals/s", "best_f_rank0": full_best,
                                     "sigma_end_rank0": full_sigma,
                                     "note": "SURVEY 8d C2 run: 200 fused generations from the straight line (fill-up 0..40 pairs and "
                                             "convergence included), L2 warm, one enqueue, CUDA events"},
            "kernel_ms": per_kernel,
            "roofline": {"kernel": "k_cost", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": NCU_DRAM_BYTES_PER_LAUNCH, "traffic_source": NCU_SOURCE,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bytes_per_launch, "launch_ms": cost_ms,
                         "strict_hbm": {"achieved": strict, "frac": strict / peak, "unit": "GB/s",
                                        "note": "map assumed L2-resident: (4n + 8) B per evaluation only (SURVEY 8d)"},
                         "note": "bytes = lambda*(4n + S*4 + 8), S = mean map samples per trajectory; duration = CUDA events "
                                 "around k_cost on the launching stream, L2 flushed before each generation"},
            "roofline_sample": sampler_roofline(2 * W, LAM, live1, per_kernel["sample"], peak),
            "e2e": {"value": world * LAM * args.steps / e2e_t, "unit": "evals/s", "h2d_bytes_per_step": e2e["h2d"],
                    "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": e2e_t / args.steps * 1e3,
                    "calls_ms_rank0": e2e["calls"], "path": e2e["path"], "variants_rank0": e2e["variants"]},
            "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": t_wall,
        }
        if c3 is not None:
            out["c3_sharded"] = c3
        if c4 is not None:
            out["c4_split"] = c4
        out["cost_kernel"] = {"evals_per_s": LAM / (cost_ms * 1e-3), "note": "k_cost alone (CUDA events, L2 flushed): the numerator of the "
                              "north star's '>= 100x the CPU trajectory-evaluation throughput' target"}
        if storage_ms:
            out["cost_kernel"]["launch_ms_by_map_storage"] = dict(storage_ms, note="stand-alone k_cost launches on the last C2 population, "
                                                                  "f32 bricks (8x4 cells per 128-byte line) vs u8 bricks (16x8, distance "
                                                                  "quantised to 1/4 cell and clamped at 63 cells: a different map, not the C2 workload)")
        if world == 1 and "cpu" not in skip:
            out["cpu_baseline"] = cpu_baseline_all(dist, start, goal, lo, hi, x0)
            try:
                out["cost_kernel"]["speedup_vs_cpu_cost_all_cores"] = out["cost_kernel"]["evals_per_s"] / out["cpu_baseline"]["parts"]["cost_only_all_cores"]["value"]
            except Exception:
                pass
        elif "cpu" not in skip:
            out["cpu_baseline"] = {"note": "timed at N = 1 only (rank 0); see the N = 1 line and --impl reference"}
        print(json.dumps(out))
    if dist_pg is not None:
        dist_pg.barrier()
        dist_pg.destroy_process_group()
    return out


def run_e2e(args, L, K, torch, cmap, start, goal, lo, hi, x0, rank, local, flush, barrier):
    """End to end through the reference-facing protocol with HOST buffers, wall clock around synchronous calls, L2
    flushed before every step.  Headline variant = the library's page-locked candidate mirror when the build has it
    (lmcma_b200_ask_all_view: the sampler's D2H of X overlaps the sampling, ask is a pointer hand-out, cost_evaluate
    recognises the mirror and evaluates the device copy); `caller_buffers` = ask_all into the caller's pinned array,
    k_cost reading it back across PCIe."""
    import ctypes as C
    from lmcma_path_planner_b200.optimizer import _endpoints, _objective
    obj, ends = _objective(W, L.LONGSAFE, 1e4), _endpoints(start, goal)
    lib = K.lib()
    fh = torch.empty(LAM, dtype=torch.float32).pin_memory().numpy()
    nch = torch.empty(LAM, dtype=torch.int32).pin_memory().numpy()
    nsh = torch.empty(LAM, dtype=torch.int32).pin_memory().numpy()
    Xh = torch.empty((LAM, 2 * W), dtype=torch.float32).pin_memory().numpy()
    have_view = hasattr(lib, "lmcma_b200_ask_all_view")
    variants = {}

    def measure(use_view):
        o = L.Optimizer(2 * W, x0=x0, lam=LAM, m=M, lo=lo, hi=hi, sigma0=SIGMA0, seed=2000 + rank, rng="philox", device=local)
        parts = [0.0, 0.0, 0.0]

        def step():
            t0 = time.perf_counter()
            if use_view:
                xp, ld = C.POINTER(C.c_float)(), C.c_int64(0)
                K.check(lib.lmcma_b200_ask_all_view(o._h, C.byref(xp), C.byref(ld)))
                xarg = xp
            else:
                K.check(lib.lmcma_b200_ask_all(o._h, K.fptr(Xh)))
                xarg = K.fptr(Xh)
            t1 = time.perf_counter()
            K.check(lib.lmcma_b200_cost_evaluate(cmap._h, C.byref(obj), C.byref(ends), xarg, LAM, K.fptr(fh), K.iptr(nch), K.iptr(nsh)))
            t2 = time.perf_counter()
            K.check(lib.lmcma_b200_tell_all(o._h, K.fptr(fh)))
            t3 = time.perf_counter()
            parts[0] += t1 - t0; parts[1] += t2 - t1; parts[2] += t3 - t2
            return float(fh[0])

        for _ in range(max(args.warmup, 3) + max(0, FILL - max(args.warmup, 3))):
            step()
        barrier()
        parts[:] = [0.0, 0.0, 0.0]
        tt = 0.0
        for _ in range(args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step()
            tt += time.perf_counter() - t0
        o.close()
        calls = {k: v / args.steps * 1e3 for k, v in zip(("ask", "cost_evaluate", "tell_all"), parts)}
        return tt, calls

    def measure_device_candidates():
        # not the headline: the candidates never leave the device (no host view of X at all); only the fitness crosses PCIe, as
        # the result of the evaluation (k_cost stores it into the caller's pinned array) and as the input of tell_all
        o = L.Optimizer(2 * W, x0=x0, lam=LAM, m=M, lo=lo, hi=hi, sigma0=SIGMA0, seed=2000 + rank, rng="philox", device=local)
        o.attach_cost(cmap, [start], [goal], W, L.LONGSAFE, 1e4)
        parts = [0.0, 0.0]

        def step():
            t0 = time.perf_counter()
            o.mg_evaluate(fh.ctypes.data)                        # page-locked host memory: the same address on the device (UVA)
            o.sync()
            t1 = time.perf_counter()
            K.check(lib.lmcma_b200_tell_all(o._h, K.fptr(fh)))
            t2 = time.perf_counter()
            parts[0] += t1 - t0; parts[1] += t2 - t1

        for _ in range(max(args.warmup, 3) + max(0, FILL - max(args.warmup, 3))):
            step()
        barrier()
        parts[:] = [0.0, 0.0]
        tt = 0.0
        for _ in range(args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step()
            tt += time.perf_counter() - t0
        o.close()
        return tt, {k: v / args.steps * 1e3 for k, v in zip(("evaluate", "tell_all"), parts)}

    t_cb, calls_cb = measure(False)
    try:
        t_dc, calls_dc = measure_device_candidates()
        variants["device_candidates"] = {"ms_per_step": t_dc / args.steps * 1e3, "calls_ms": calls_dc,
                                         "h2d_bytes_per_step": LAM * 4, "d2h_bytes_per_step": LAM * 4,
                                         "path": "NOT the headline (no host copy of the candidates exists): lmcma_b200_mg_evaluate on the "
                                                 "optimiser's own device population into the caller's pinned fitness array -> "
                                                 "lmcma_b200_sync -> lmcma_b200_tell_all (H2D f; update + sample)"}
    except Exception as e:                                       # informational variant: never fails the bench
        variants["device_candidates"] = {"error": str(e)[:200]}
    variants["caller_buffers"] = {"ms_per_step": t_cb / args.steps * 1e3, "calls_ms": calls_cb,
                                  "h2d_bytes_per_step": LAM * 2 * W * 4 + LAM * 4, "d2h_bytes_per_step": LAM * 2 * W * 4 + LAM * 12,
                                  "path": "lmcma_b200_ask_all (D2H X into the caller's pinned array) -> lmcma_b200_cost_evaluate (k_cost reads the "
                                          "caller's page-locked rows across PCIe, stores f / flags into the caller's arrays) -> lmcma_b200_tell_all"}
    if have_view:
        t_v, calls_v = measure(True)
        variants["library_mirror"] = {"ms_per_step": t_v / args.steps * 1e3, "calls_ms": calls_v,
                                      "h2d_bytes_per_step": LAM * 4, "d2h_bytes_per_step": LAM * 2 * W * 4 + LAM * 12,
                                      "path": "lmcma_b200_ask_all_view (the candidates are already in the library's page-locked mirror: the "
                                              "sampler wrote them across PCIe while it ran) -> lmcma_b200_cost_evaluate on that pointer "
                                              "(recognised: evaluates the device copy, f / flags stored into the caller's pinned arrays) -> "
                                              "lmcma_b200_tell_all (H2D f; update + sample + mirror)"}
        best = "library_mirror" if t_v <= t_cb else "caller_buffers"
    else:
        best = "caller_buffers"
    v = variants[best]
    t = t_v if best == "library_mirror" else t_cb
    return {"t": t, "h2d": v["h2d_bytes_per_step"], "d2h": v["d2h_bytes_per_step"], "calls": v["calls_ms"], "path": v["path"],
            "variants": variants}


def run_c3(args, L, torch, dist_pg, dist, cmap, lo, hi, rank, world, local, stream, barrier, max_over_ranks, peak,
           queries=4096, lam=64, gens=20):
    """BASELINE.json configs[2]: 4096 independent start/goal queries (SURVEY 8d: U(free cells), seed 7, |goal - start| >=
    1024) x lambda 64, n = 400, m = 40 on the C2 map, sharded contiguously over the ranks; no data-path collective.
    Strong scaling: the job is fixed, the time is the max over ranks (CUDA events around `gens` fused generations)."""
    from lmcma_path_planner_b200 import maps, parallel
    starts, goals = maps.random_queries(dist, queries, seed=7, min_sep=1024)

    def timed(off, cnt, seed):
        x0b = np.stack([maps.straight_line(starts[q], goals[q], W) for q in range(off, off + cnt)])
        o = L.Optimizer(2 * W, x0=x0b, lam=lam, m=M, batch=cnt, lo=lo, hi=hi, sigma0=SIGMA0, seed=seed, device=local)
        o.attach_cost(cmap, starts[off:off + cnt], goals[off:off + cnt], W, L.LONGSAFE, 1e4)
        o.set_stream(stream.cuda_stream)
        o.run(FILL)                                  # untimed: all m pairs live
        return o

    off, cnt = parallel.shard_range(queries, world, rank)
    o = timed(off, cnt, 7 + rank)
    barrier()
    o.run(gens)
    o.sync()
    ms = o.last_run_ms()
    pk = o.profile_kernels(3)
    nsamp = float(o.get("nsamp").mean())
    live = int(o.get("live")[0])
    o.close()
    (ms_max,) = max_over_ranks([ms])
    res = None
    ms_one = None
    if world > 1:                                    # the whole job on ONE GPU, same run, for the efficiency
        barrier()
        if rank == 0:
            o1 = timed(0, queries, 7)
            o1.run(gens)
            o1.sync()
            ms_one = o1.last_run_ms()
            o1.close()
        barrier()
    if rank == 0:
        cost_bytes = cnt * lam * (4 * 2 * W + nsamp * cmap.bytes_per_cell + 8)
        cost_gbs = cost_bytes / (pk["cost"] * 1e-3) / 1e9
        res = {"workload": "C3: %d queries x lambda %d (n=400, m=40) on the C2 map, sharded contiguously over %d GPU(s), no collective" % (queries, lam, world),
               "scaling": "strong", "generations_timed": gens, "untimed_generations": FILL, "live_pairs": live,
               "ms_per_generation": ms_max / gens, "value": queries * lam * gens / (ms_max * 1e-3), "unit": "evals/s",
               "query_generations_per_s": queries * gens / (ms_max * 1e-3), "queries_per_rank": cnt,
               "kernel_ms_rank0": pk, "mean_samples_per_trajectory": nsamp,
               "roofline_k_cost_rank0": {"bound": "hbm", "achieved": cost_gbs, "peak": peak, "unit": "GB/s", "frac": cost_gbs / peak,
                                         "algorithmic_bytes_per_launch": cost_bytes, "launch_ms": pk["cost"],
                                         "note": "many waves of CTAs: the per-trajectory phases overlap across CTAs, L2 warm"},
               "roofline_sample_rank0": sampler_roofline(2 * W, lam * cnt, live, pk["sample"], peak)}
        if ms_one is not None:
            res["one_gpu_same_run"] = {"ms_per_generation": ms_one / gens, "value": queries * lam * gens / (ms_one * 1e-3)}
            res["efficiency_vs_one_gpu"] = ms_one / (world * ms_max)
    return res


def run_c4(args, L, torch, dist_pg, rank, world, local, stream, barrier, max_over_ranks, size=512, waypoints=500, lam=8192,
           gens=20):
    """BASELINE.json configs[3]: ONE population lambda = 8192, n = 1500, m = 77 on a 512^3 u8 voxel cost map (SURVEY 8d: 4096
    boxes, seed 43, EDT clamped at 64 — built on the device from the occupancy grid), sigma0 = 8.  world > 1: the offspring
    rows are split over the ranks; per generation two NCCL all-gathers (lambda fitness scalars; one (n + 4)-float payload per
    rank), state replicated.  The generation (3 stages + 2 exchanges) is captured in ONE CUDA graph when the capture
    succeeds.  Rank 0 also times the unsplit population on one GPU, so the line carries the efficiency and names the limiter."""
    from lmcma_path_planner_b200 import maps, parallel
    n = 3 * waypoints
    m = int(2 * np.sqrt(n))
    start, goal = (16.0, 16.0, 16.0), (size - 16.0, size - 16.0, size - 16.0)
    occ = maps.random_boxes_occupancy((size, size, size), 4096, 4, 48, 43, border=0, clear=[(start, 12.0), (goal, 12.0)])
    cmap = L.CostMap.from_occupancy(occ, 64.0, "u8", u8_scale=0.25, device=local)
    del occ
    lo, hi = maps.box_bounds((size, size, size), waypoints)
    x0 = maps.straight_line(start, goal, waypoints)
    kw = dict(x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=8.0, seed=43, device=local)
    fill = m + 3
    res = {"workload": "C4: 512^3 u8 voxel map, 500 waypoints (n=1500), lambda=8192, m=77, sigma0=8; offspring split over %d GPU(s)" % world,
           "generations_timed": gens, "untimed_generations": fill}

    ms_whole = None
    if rank == 0:                                    # the unsplit population on one GPU
        whole = L.Optimizer(n, **kw)
        whole.attach_cost(cmap, [start], [goal], waypoints, L.LONGSAFE, 1e4)
        whole.set_stream(stream.cuda_stream)
        whole.run(fill)
        whole.run(gens)
        whole.sync()
        ms_whole = whole.last_run_ms()
        res["one_gpu_whole_population"] = {"ms_per_generation": ms_whole / gens, "value": lam * gens / (ms_whole * 1e-3), "unit": "evals/s",
                                           "kernel_ms": whole.profile_kernels(3), "live_pairs": int(whole.get("live")[0]),
                                           "sigma": float(whole.get("sigma")[0])}
        whole.close()
    if world > 1:
        barrier()
        part = L.Optimizer(n, pop_offset=rank * lam // world, pop_count=lam // world, **kw)
        part.attach_cost(cmap, [start], [goal], waypoints, L.LONGSAFE, 1e4)
        part.set_stream(stream.cuda_stream)
        sp = parallel.SplitPopulation(parallel.DeviceBackend(part, stream.cuda_stream), dist_pg, torch.device("cuda", local))
        sp.run(fill)                                 # eager, untimed: all m pairs live
        torch.cuda.synchronize()
        # the eager generation stage by stage (events between the enqueue calls: host latency included)
        stage_names = ("evaluate", "allgather_fitness", "rank", "allgather_payload", "update_and_sample")
        stage_ms = sp.profile_stages(5)
        graphed = sp.capture()                       # one CUDA graph per generation (falls back to eager enqueue)
        sp.run(3)
        barrier()
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record(stream)
        sp.run(gens)
        e1.record(stream)
        torch.cuda.synchronize()
        (ms,) = max_over_ranks([e0.elapsed_time(e1)])
        (stage_max) = max_over_ranks(stage_ms)
        pk = part.profile_kernels(3)                 # per-kernel device time of THIS rank's shapes (after the timed region: it
        #                                              advances the local replica on its own rows only)
        if rank == 0:
            res["split"] = {"ms_per_generation": ms / gens, "value": lam * gens / (ms * 1e-3), "unit": "evals/s",
                            "rows_per_gpu": lam // world, "exchange": "2 x NCCL all_gather per generation (%d B + %d B per rank)" % (4 * lam // world, 4 * (n + 4)),
                            "generation_enqueue": "one CUDA graph replay" if graphed else "eager (5 enqueue calls)",
                            "kernel_ms_rank0": pk,
                            "stage_ms_eager_with_host_latency_max_over_ranks": dict(zip(stage_names, stage_max)),
                            "live_pairs": int(part.get("live")[0]), "sigma": float(part.get("sigma")[0])}
            res["efficiency_vs_one_gpu"] = ms_whole / (world * ms)
            shard = pk["cost"] + pk["sample"]
            res["limiter"] = ("of the %.3f ms split generation only k_cost + k_sample (%.3f ms on this rank's %d rows) shrink with the GPU count; "
                              "the update (%.3f ms: k_update + k_gram + k_coef + k_combine, the coefficient recurrence k_coef on ONE SM) is "
                              "replicated on every rank (Amdahl), the ranking (%.3f ms) compares the local rows with all lambda values, and "
                              "the two latency-bound all-gathers plus launch gaps take the remaining %.3f ms" %
                              (ms / gens, shard, lam // world, pk["update"], pk["rank"], max(0.0, ms / gens - sum(pk.values()))))
        part.close()
    cmap.close()
    return res if rank == 0 else None


def _cpu_timed(step, budget_s, min_steps=1):
    t0 = time.perf_counter()
    k = 0
    while k < min_steps or time.perf_counter() - t0 < budget_s:
        step()
        k += 1
    return k, time.perf_counter() - t0


def cpu_baseline(dist, start, goal, lo, hi, x0, budget_s, steps=None, warmup=0):
    """The reference's CPU implementation of the path on the host cores: the UNMODIFIED reference LMCMA class
    (oracle/_ref, single serial stream as shipped; m = lambda is its only rule) driven through its ask/tell
    protocol, with the cost restatement (oracle/cost_oracle.c) as the user cost evaluated over the population
    on all host threads.  Bounded sample: generations of the C2 query until `budget_s` (or `steps`)."""
    from oracle import pyoracle as po
    cores = os.cpu_count() or 1
    prob = po.CostProblem(dist, start, goal, W, 1.0, 1000.0, 1e4, threads=cores)
    kind = "reference"
    try:
        opt = po.RefLMCMA(2 * W, x0=x0, lam=LAM, lo=lo, hi=hi, sigma=SIGMA0, seed=1)
        step = lambda: opt.generation(prob)
    except Exception:
        kind = "port"
        opt = po.OracleLMCMA(2 * W, x0=x0, lam=LAM, m=M, lo=lo, hi=hi, sigma=SIGMA0, seed=1)

        def step():
            X = opt.array("X")
            opt.tell_all(prob.evaluate(X)["f"])
    for _ in range(warmup):
        step()
    if steps is not None:
        gens, dt = _cpu_timed(step, 0.0, steps)
    else:
        gens, dt = _cpu_timed(step, budget_s)
    return {"value": LAM * gens / dt, "unit": "evals/s", "cores": cores, "kind": kind,
            "sample": "%d generations of the C2 query (lambda=1024, n=400) in %.1f s: reference LMCMA (oracle/_ref, serial, "
                      "m=lambda, so the live pairs grow 1 per generation up to %d here) + cost restatement on %d threads" % (gens, dt, gens + warmup, cores),
            "ms_per_step": dt / gens * 1e3, "generations": gens}


def cpu_baseline_all(dist, start, goal, lo, hi, x0):
    """BASELINE.md section 3, all four figures, each a bounded sample of the C2 workload on this box's host cores."""
    from oracle import pyoracle as po
    cores = os.cpu_count() or 1
    main = cpu_baseline(dist, start, goal, lo, hi, x0, budget_s=7.0)
    parts = {}
    p1 = po.CostProblem(dist, start, goal, W, 1.0, 1000.0, 1e4, threads=1)
    pall = po.CostProblem(dist, start, goal, W, 1.0, 1000.0, 1e4, threads=cores)
    # (1) the reference as shipped: single thread end to end (-O2, and -O0 because the package ships CMAKE_BUILD_TYPE Debug)
    for label, o0, budget in (("reference_single_thread_O2", False, 5.0), ("reference_single_thread_O0", True, 4.0)):
        try:
            r = po.RefLMCMA(2 * W, x0=x0, lam=LAM, lo=lo, hi=hi, sigma=SIGMA0, seed=1, o0=o0)
            g, dt = _cpu_timed(lambda: r.generation(p1), budget)
            parts[label] = {"value": LAM * g / dt, "unit": "evals/s", "cores": 1, "kind": "reference", "generations": g,
                            "sample": "reference LMCMA (%s) ask/tell + cost restatement, ONE thread, %d generations in %.1f s (live pairs 1..%d)" %
                                      ("-O0 -g" if o0 else "-O2", g, dt, g)}
        except Exception as e:                       # e.g. a prebuilt _ref without the -O0 library
            parts[label] = {"unavailable": str(e)[:120]}
    # (2) cost restatement only, all cores: the denominator of the ">= 100x trajectory-evaluation throughput" target
    rng = np.random.default_rng(0)
    X = np.clip(x0[None] + SIGMA0 * rng.standard_normal((LAM, 2 * W)), lo, hi).astype(np.float32)
    g, dt = _cpu_timed(lambda: pall.evaluate(X), 4.0)
    parts["cost_only_all_cores"] = {"value": LAM * g / dt, "unit": "evals/s", "cores": cores, "kind": "port",
                                    "sample": "oracle/cost_oracle.c over a 1024-row C2 population (sigma 32 around the straight line), "
                                              "%d threads, %d passes in %.1f s" % (cores, g, dt)}
    g, dt = _cpu_timed(lambda: p1.evaluate(X[:128]), 2.0)
    parts["cost_only_single_thread"] = {"value": 128 * g / dt, "unit": "evals/s", "cores": 1, "kind": "port",
                                        "sample": "128 rows per pass, %d passes in %.1f s" % (g, dt)}
    # (3) the equal-algorithm baseline: the restatement with m = 40 (what the device runs), single thread
    o = po.OracleLMCMA(2 * W, x0=x0, lam=LAM, m=M, lo=lo, hi=hi, sigma=SIGMA0, seed=1)

    def step():
        o.tell_all(p1.evaluate(o.array("X"))["f"])
    g, dt = _cpu_timed(step, 5.0)
    parts["restatement_m40_single_thread"] = {"value": LAM * g / dt, "unit": "evals/s", "cores": 1, "kind": "port", "generations": g,
                                              "sample": "oracle/lmcma_oracle.cpp with m = 40 + cost restatement, ONE thread, %d generations in %.1f s" % (g, dt)}
    main["parts"] = parts
    main["note"] = ("`value` = reference LMCMA (m = lambda: its cost per generation grows with the generation count, so a longer sample "
                    "reads lower) + cost restatement on all host threads, the same arm `--impl reference` times; parts = BASELINE.md section 3")
    return main


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    dist, start, goal, lo, hi, x0 = build_problem()
    cb = cpu_baseline(dist, start, goal, lo, hi, x0, budget_s=None, steps=args.steps, warmup=args.warmup)
    world = int(os.environ.get("WORLD_SIZE", 1))
    out = {"impl": "reference", "metric": "trajectory-cost evals/s (LM-CMA generations/s = value / lambda)",
           "value": cb["value"], "unit": "evals/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": dict(WORKLOAD, parallelism="host CPU: ONE process using all host threads whatever N is (at N > 1 a ratio against this "
                                                "line is N GPUs vs one host)",
                          m="lambda (the reference's only rule: live pairs = generation count here)"),
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--skip", default="", help="comma list of c3,c4,cpu (development runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed generation computed as DIR/<name>.npy (rank 0, --impl b200)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
