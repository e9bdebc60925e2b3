"""Restarting instances of a live batch in place (reset_instances) against rebuilding the handle, and what recording a
device reset into every generation of a captured loop costs when it resets nothing.

C3: bench.py's batch, 4096 queries (maps.random_queries, seed 7, |goal - start| >= 1024) x lambda 64, n = 400 (200
waypoints), m = 40, sigma0 = 32 on the 4096^2 C2 map.  C2: one query, lambda 1024, same n and m.
  (a) host_reset      reset_instances of 1, 64 (every 64th) and all 4096 instances of a C3 handle, each to its query's
                      straight line: host clock around the call, which ends in a device synchronise; median of 20
  (b) rebuild         the route without reset: create + attach_cost + the first run(1) + sync at C3; median of 5
  (c) device loop     per generation [cost -> tell_all_dev] with and without reset_instances_dev(all-zero flags) behind it,
                      captured in torch.cuda.graph (20 generations per graph, replayed 10 times), at C3 and at C2; the
                      variants alternate within each repetition.  Cost at C3: the weighted sphere as a torch expression on
                      X (4096 calls of the map's evaluate_dev per generation would time the host); at C2: the map's
                      evaluate_dev.  Host clock around 200 generations ending in a device synchronise, L2 warm.

    python tools/reset_timing.py [--reps 7] [--out result.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import maps

W, M, SIGMA0, FILL, GENS, CHUNK = 200, 40, 32.0, 45, 200, 20
QUERIES, LAM3, LAM2 = 4096, 64, 1024


def card():
    """Name and power limit of GPU 0, read now (the numbers below belong to them)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (s.strip() for s in q.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def stats(v, digits=1):
    return {"median": round(float(np.median(v)), digits), "min": round(float(np.min(v)), digits),
            "max": round(float(np.max(v)), digits), "runs": [round(float(x), digits) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps({"card": info}), flush=True)
    dist, start, goal = maps.config2_map()
    lo, hi = maps.box_bounds(dist.shape[::-1], W)
    cmap = L.CostMap(dist, "f32")
    starts, goals = maps.random_queries(dist, QUERIES, seed=7, min_sep=1024)
    x0_3 = np.stack([maps.straight_line(starts[q], goals[q], W) for q in range(QUERIES)])

    def c3(seed):
        o = L.Optimizer(2 * W, x0=x0_3, lam=LAM3, m=M, batch=QUERIES, lo=lo, hi=hi, sigma0=SIGMA0, seed=seed)
        o.attach_cost(cmap, starts, goals, W, L.LONGSAFE, 1e4)
        return o

    def c2(seed):
        o = L.Optimizer(2 * W, x0=maps.straight_line(start, goal, W), lam=LAM2, m=M, lo=lo, hi=hi, sigma0=SIGMA0, seed=seed)
        o.attach_cost(cmap, [start], [goal], W, L.LONGSAFE, 1e4)
        return o

    doc = {"tool": "tools/reset_timing.py", "card": info,
           "workload": "C3: %d queries x lambda %d, n = 400, m = 40, 4096^2 f32 map; C2: one query x lambda %d" % (QUERIES, LAM3, LAM2)}

    # (a) host resets of a live C3 handle
    o = c3(7)
    o.run(FILL)
    o.sync()
    host = {}
    for count in (1, 64, QUERIES):
        idx = np.arange(0, QUERIES, QUERIES // count)[:count]
        o.reset_instances(idx, x0_3[idx])                        # untimed: first use allocates the staging descriptor
        t = []
        for _ in range(20):
            o.run(1)
            o.sync()
            t0 = time.perf_counter()
            o.reset_instances(idx, x0_3[idx])
            t.append(1e3 * (time.perf_counter() - t0))
        host["reset_%d" % count] = stats(t, 3)
        print(json.dumps({"host_reset_ms_%d" % count: host["reset_%d" % count]["median"]}), flush=True)
    o.close()
    doc["a_host_reset_ms"] = host

    # (b) the rebuild route
    t = []
    for r in range(6):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h = c3(100 + r)
        h.run(1)
        h.sync()
        ms = 1e3 * (time.perf_counter() - t0)
        h.close()
        if r:                                                    # the first one loads the modules
            t.append(ms)
    doc["b_rebuild_ms"] = stats(t, 3)
    print(json.dumps({"rebuild_ms": doc["b_rebuild_ms"]["median"]}), flush=True)

    # (c) captured device loops with and without an all-zero reset per generation
    def captured(o, shape, reset):
        s = torch.cuda.Stream()
        o.set_stream(s.cuda_stream)
        X, F = o.device_tensors()
        flags = torch.zeros(o.batch, dtype=torch.int32, device="cuda")
        x0 = torch.zeros((o.batch, o.n), dtype=torch.float64, device="cuda")
        w = 1.0 + torch.arange(o.n, device="cuda", dtype=torch.float32)

        def gens(count):
            for _ in range(count):
                if shape == "c3":
                    F.copy_((w * X * X).sum(-1))
                else:
                    cmap.evaluate_dev(X.data_ptr(), o.ld, o.lam, F.data_ptr(), start, goal, W, L.LONGSAFE, 1e4,
                                      stream=s.cuda_stream)
                o.tell_all_dev()
                if reset:
                    o.reset_instances_dev(flags, x0)
        with torch.cuda.stream(s):
            gens(FILL)                                           # every pair live
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            gens(CHUNK)
        torch.cuda.synchronize()

        def replay():
            for _ in range(GENS // CHUNK):
                g.replay()
            torch.cuda.synchronize()
        # the graph reads flags, x0 and w where they are now: they must live as long as it does (the next capture's
        # empty_cache() would hand their memory back to the driver)
        return (g, flags, x0, w), replay

    loops, keep = {}, []
    for shape, make in (("c3", c3), ("c2", c2)):
        for reset in (False, True):
            o = make(21 + len(loops))
            graph_and_inputs, fn = captured(o, shape, reset)
            keep += [o, graph_and_inputs]
            loops["%s_%s" % (shape, "with_reset" if reset else "plain")] = fn
    times = {k: [] for k in loops}
    for r in range(args.reps + 1):
        for name, fn in loops.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            if r:                                                # repetition 0 warms up every variant
                times[name].append(1e6 * (time.perf_counter() - t0) / GENS)
        print(json.dumps({k: [round(x, 2) for x in v[-1:]] for k, v in times.items()}), flush=True)
    doc["c_device_loop_us_per_generation"] = {k: stats(v, 2) for k, v in times.items()}
    doc["c_clock"] = "host perf_counter around %d captured generations ending in a device synchronise, L2 warm, %d repetitions" % (GENS, args.reps)
    print(json.dumps(doc), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)
    loops.clear()
    keep.clear()                                                 # the graphs, then the handles they launch into
    cmap.close()


if __name__ == "__main__":
    main()
