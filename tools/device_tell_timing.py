"""A cost computed on the GPU by the caller: the device protocol (device_tensors -> cost -> tell_all_dev) against the fused
run and the host-buffer protocol, per generation.

C2: the 4096^2 map of bench.py (maps.config2_map), (64, 64) -> (4032, 4032), 200 waypoints (n = 400), lambda = 1024,
m = 40, sigma0 = 32, longsafe weights.  Each variant has an optimiser of its own, warmed up for 60 generations so that all
40 pairs are live in the timed region.  Variants, alternated within each repetition:
  fused          run(200) (the cost attached, one CUDA graph per generation or per 8)
  device         200 x (CostMap.evaluate_dev of X into F on the handle's stream, tell_all_dev): tell_all's forked graph
                 without the fitness copy (the default)
  device_linear  the same with LMCMA_B200_TELL_OVERLAP=0: the stream-ordered generation, launched kernel by kernel
  device_graph   the same loop captured in torch.cuda.graph (20 generations per graph, replayed 10 times), which records
                 the stream-ordered generation
  host           200 x (ask_all_view, CostMap.evaluate of the view, tell_all)
Host clock around 200 generations ending in a device synchronise, L2 warm (nothing is flushed); µs per generation, median
and range of --reps repetitions after one untimed one.

    python tools/device_tell_timing.py [--reps 7] [--out result.json]"""
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

W, LAM, M, SIGMA0, GENS, CHUNK = 200, 1024, 40, 32.0, 200, 20


def card():
    """Name and power limit of GPU 0, read now (the numbers below belong to them)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (s.strip() for s in q.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps({"card": info}), flush=True)
    dist, start, goal = maps.config2_map()
    lo, hi = maps.box_bounds(dist.shape[::-1], W)
    x0 = maps.straight_line(start, goal, W)
    cmap = L.CostMap(dist, "f32")

    def handle(seed, env=None):
        for k, v in (env or {}).items():
            os.environ[k] = v
        o = L.Optimizer(2 * W, x0=x0, lam=LAM, m=M, lo=lo, hi=hi, sigma0=SIGMA0, seed=seed)
        for k in env or {}:
            del os.environ[k]
        o.attach_cost(cmap, [start], [goal], W, L.LONGSAFE, 1e4)
        return o

    variants = {}

    fused = handle(11)
    variants["fused"] = lambda: fused.run(GENS)

    def device_loop(o, stream):
        X, F = o.device_tensors()

        def gens(count):
            for _ in range(count):
                cmap.evaluate_dev(X.data_ptr(), o.ld, LAM, F.data_ptr(), start, goal, W, L.LONGSAFE, 1e4,
                                  stream=stream.cuda_stream)
                o.tell_all_dev()
        return gens

    streams = {}
    launch = {}
    for name, env in (("device", None), ("device_linear", {"LMCMA_B200_TELL_OVERLAP": "0"}), ("device_graph", None)):
        o = handle(12 + len(streams), env)
        s = torch.cuda.Stream()
        o.set_stream(s.cuda_stream)
        streams[name] = (o, s, device_loop(o, s))
        launch[name] = o.launch()
    for name in ("device", "device_linear"):
        o, s, gens = streams[name]
        variants[name] = (lambda gens, s: lambda: (gens(GENS), s.synchronize()))(gens, s)

    o, s, gens = streams["device_graph"]
    gens(60)                                                     # warm-up: every pair live
    s.synchronize()
    o.device_tensors()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        gens(CHUNK)

    def replayed():
        for _ in range(GENS // CHUNK):
            graph.replay()
        torch.cuda.synchronize()
    variants["device_graph"] = replayed

    host = handle(16)

    def host_loop():
        for _ in range(GENS):
            X = host.ask_all_view()[0]
            f = cmap.evaluate(X, start, goal, W, L.LONGSAFE, 1e4)["f"]
            host.tell_all(f)
    variants["host"] = host_loop

    fused.run(60)
    for name in ("device", "device_linear"):
        streams[name][2](60)
        streams[name][1].synchronize()
    for _ in range(60):
        host.tell_all(cmap.evaluate(host.ask_all_view()[0], start, goal, W, L.LONGSAFE, 1e4)["f"])

    times = {k: [] for k in variants}
    for r in range(args.reps + 1):
        for name, fn in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            us = 1e6 * (time.perf_counter() - t0) / GENS
            if r:                                                # repetition 0 warms up every variant
                times[name].append(us)
        print(json.dumps({k: [round(x, 2) for x in v[-1:]] for k, v in times.items()}), flush=True)
    live = {name: int(h.get("live")[0]) for name, h in
            (("fused", fused), ("host", host), *((n, streams[n][0]) for n in streams))}
    res = {k: {"median_us_per_generation": round(float(np.median(v)), 2), "min_us": round(float(np.min(v)), 2),
               "max_us": round(float(np.max(v)), 2), "runs_us": [round(x, 2) for x in v]} for k, v in times.items()}
    doc = {"tool": "tools/device_tell_timing.py", "card": info,
           "workload": "C2: 4096^2 f32 map, n = 400, lambda = 1024, m = 40, sigma0 = 32, one query",
           "clock": "host perf_counter around %d generations ending in a device synchronise, L2 warm" % GENS,
           "repetitions": args.reps, "overlap": {k: v["overlap"] for k, v in launch.items()}, "live_pairs_after": live,
           "results": res}
    print(json.dumps(doc), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)
    del graph
    for h in (fused, host, *(streams[n][0] for n in streams), cmap):
        h.close()


if __name__ == "__main__":
    main()
