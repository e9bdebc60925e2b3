"""Queries on several maps served by one handle (attach_cost_maps) against one handle per map, and against C3 on one map.

C3 shape: 4096 queries x lambda 64, n = 400 (200 waypoints), m = 40, sigma0 = 32.  Four 4096^2 maps of the C2 kind
(maps.config2_map, seeds 42..45); 1024 queries per map (maps.random_queries on that map, seed 7 + k, |goal - start| >= 1024).
  (a)      one handle of 4096 over the four maps as u8 (u8_scale 1: 16 MiB each, 64 MiB together, L2-resident), map_of =
           query // 1024; k_cost's multi-map build at seven CTAs per SM (the default) and at six (LMCMA_B200_COST_MINB=6)
  (a_f32)  the same over the four maps as f32 (64 MiB each, 256 MiB together: past the 126 MB L2)
  (b)      the same queries as four single-map handles of 1024 (u8), all on one torch stream, run back to back
  (c)      today's C3: one handle of 4096 queries on map 0 alone (u8), and (c_f32) the same on the f32 map, bench.py's C3
Per generation: device time of `GENS` fused generations after `FILL` warm-up ones (last_run_ms for one handle, CUDA
events on the shared stream for (b)), median of the repetitions; the variants alternate within each repetition.
k_cost: profile_kernels' mean cost-kernel time over 5 un-graphed generations (for (b) the sum over the four handles).

    python tools/multi_map_timing.py [--reps 5] [--out profiles/r3e_multi_map_timing.json]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import maps

W, M, SIGMA0, LAM, FILL, GENS = 200, 40, 32.0, 64, 10, 40
MAPS, PER_MAP = 4, 1024


def card():
    """Name and power limit of GPU 0, read now (the numbers below belong to them)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (s.strip() for s in q.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def stats(v, digits=3):
    return {"median": round(float(np.median(v)), digits), "min": round(float(np.min(v)), digits),
            "max": round(float(np.max(v)), digits), "runs": [round(float(x), digits) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps({"card": info}), flush=True)
    dists = [maps.config2_map(seed=42 + k)[0] for k in range(MAPS)]
    lo, hi = maps.box_bounds(dists[0].shape[::-1], W)
    u8 = [L.CostMap(d, "u8", u8_scale=1.0) for d in dists]
    f32 = [L.CostMap(d, "f32") for d in dists]
    qs = [maps.random_queries(dists[k], PER_MAP, seed=7 + k, min_sep=1024) for k in range(MAPS)]
    starts = np.concatenate([q[0] for q in qs])
    goals = np.concatenate([q[1] for q in qs])
    x0 = np.stack([maps.straight_line(starts[b], goals[b], W) for b in range(len(starts))])
    map_of = np.repeat(np.arange(MAPS, dtype=np.int32), PER_MAP)
    s0, g0 = maps.random_queries(dists[0], MAPS * PER_MAP, seed=7, min_sep=1024)
    x00 = np.stack([maps.straight_line(s0[b], g0[b], W) for b in range(len(s0))])

    def handle(cm, st, gl, x, mo=None, minb=None, seed=1):
        if minb:
            os.environ["LMCMA_B200_COST_MINB"] = str(minb)
        o = L.Optimizer(2 * W, x0=x, lam=LAM, m=M, batch=len(x), lo=lo, hi=hi, sigma0=SIGMA0, seed=seed)
        os.environ.pop("LMCMA_B200_COST_MINB", None)
        o.attach_cost(cm, st, gl, W, L.LONGSAFE, 1e4, map_of=mo)
        return o

    one = {
        "a_u8_minb7": handle(u8, starts, goals, x0, map_of),
        "a_u8_minb6": handle(u8, starts, goals, x0, map_of, minb=6),
        "a_f32": handle(f32, starts, goals, x0, map_of),
        "c_u8_one_map": handle(u8[0], s0, g0, x00),
        "c_f32_one_map": handle(f32[0], s0, g0, x00),
    }
    stream = torch.cuda.Stream()
    four = []
    for k in range(MAPS):
        sl = slice(k * PER_MAP, (k + 1) * PER_MAP)
        h = handle(u8[k], starts[sl], goals[sl], x0[sl], seed=1 + k)
        h.set_stream(stream.cuda_stream)
        four.append(h)

    def run_one(o):
        o.run(FILL)
        o.run(GENS)                                              # sync = True
        return o.last_run_ms() / GENS

    def run_four():
        for h in four:
            h.run(FILL, sync=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(GENS // 10):
            for h in four:
                h.run(10, sync=False)
        e1.record(stream)
        stream.synchronize()
        for h in four:
            h.sync()
        return e0.elapsed_time(e1) / GENS

    variants = dict({k: (lambda o=o: run_one(o)) for k, o in one.items()}, b_u8_four_handles=run_four)
    times = {k: [] for k in variants}
    for r in range(args.reps + 1):
        for name, fn in variants.items():
            ms = fn()
            if r:                                                # repetition 0 warms up every variant
                times[name].append(ms)
        print(json.dumps({k: [round(x, 4) for x in v[-1:]] for k, v in times.items()}), flush=True)

    cost = {k: [] for k in variants}
    for r in range(args.reps):
        for name, o in one.items():
            cost[name].append(o.profile_kernels(5)["cost"])
        cost["b_u8_four_handles"].append(sum(h.profile_kernels(5)["cost"] for h in four))
    doc = {"tool": "tools/multi_map_timing.py", "card": info,
           "workload": "C3 shape: %d queries x lambda %d, n = 400, m = 40; four 4096^2 maps (config2_map seeds 42..45), "
                       "%d queries per map" % (MAPS * PER_MAP, LAM, PER_MAP),
           "clock": "per generation: device events around %d fused generations after %d warm-up ones, L2 warm; "
                    "%d repetitions, variants alternated" % (GENS, FILL, args.reps),
           "ms_per_generation": {k: stats(v) for k, v in times.items()},
           "k_cost_ms": {k: stats(v) for k, v in cost.items()}}
    print(json.dumps(doc), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)
    for o in list(one.values()) + four:
        o.close()
    for m in u8 + f32:
        m.close()


if __name__ == "__main__":
    main()
