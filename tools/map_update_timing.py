"""Replanning on a changing map: an in-place occupancy update (CostMap.update_occupancy) against the rebuild route
(CostMap.from_occupancy of the edited grid + attach_cost + the first run(1), which captures the fused graphs again).

C2: 4096^2 occupancy (seed 42, 2048 rectangles), f32, clamp 256, an attached C2 optimiser (n = 400, lambda = 1024, m = 40);
square boxes of 16, 64 and 256 cells on the straight path.  C4: 512^3 occupancy (seed 43, 4096 boxes), u8 (1/4 cell), clamp
64, an attached C4 optimiser (n = 1500, lambda = 8192, m = 77); cubes of 16 and 64 cells.  Each repetition applies the box
(all obstacle) or restores its original content, alternately, so every update changes the map.

Host clock around synchronous calls; the two routes alternate, each on an optimiser of its own (the in-place one stays
attached, the other is re-attached to every rebuilt map); median and quartiles of --reps repetitions after one untimed
repetition of each.  run(1) right after each route is timed as well: after the update it replays the graphs as they are,
after the rebuild it is the route's first run(1).

    python tools/map_update_timing.py [--reps 20] [--out result.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import maps


def card():
    """Name and power limit of GPU 0, read now (the numbers below belong to them)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (s.strip() for s in q.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def stats(v):
    q = np.percentile(v, [25, 50, 75])
    return {"median_ms": round(float(q[1]), 4), "p25_ms": round(float(q[0]), 4), "p75_ms": round(float(q[2]), 4)}


def measure(label, occ, clamp, storage, start, goal, waypoints, opt_kw, sides, reps):
    dims = occ.ndim
    shape_xyz = occ.shape[::-1]
    n = dims * waypoints
    lo_b, hi_b = maps.box_bounds(shape_xyz, waypoints)
    x0 = maps.straight_line(start, goal, waypoints)
    cmap = L.CostMap.from_occupancy(occ, clamp, storage)
    inplace = L.Optimizer(n, x0=x0, lo=lo_b, hi=hi_b, **opt_kw)
    rebuilt = L.Optimizer(n, x0=x0, lo=lo_b, hi=hi_b, **opt_kw)
    inplace.attach_cost(cmap, [start], [goal], waypoints, L.LONGSAFE, 1e4)
    inplace.run(4)
    rebuilt.attach_cost(cmap, [start], [goal], waypoints, L.LONGSAFE, 1e4)
    rebuilt.run(4)
    out = []
    for s in sides:
        lo = tuple(c // 2 - s // 2 for c in shape_xyz)                     # the middle of the diagonal start -> goal
        sl = tuple(slice(l, l + s) for l in lo[::-1])
        original = occ[sl].copy()
        block = np.ones((s,) * dims, np.uint8)
        rec = {k: [] for k in ("update", "run1_after_update", "from_occupancy", "attach_cost", "run1_after_rebuild")}
        for r in range(reps + 1):
            box = block if r % 2 == 0 else original
            t_up = timed(lambda: cmap.update_occupancy(lo, box))
            t_run = timed(lambda: inplace.run(1))
            grid = occ.copy()
            grid[sl] = box
            fresh = []
            t_build = timed(lambda: fresh.append(L.CostMap.from_occupancy(grid, clamp, storage)))
            del grid
            t_att = timed(lambda: rebuilt.attach_cost(fresh[0], [start], [goal], waypoints, L.LONGSAFE, 1e4))
            t_run_b = timed(lambda: rebuilt.run(1))
            if r:                                                           # repetition 0 warms up both routes
                for k, v in zip(rec, (t_up, t_run, t_build, t_att, t_run_b)):
                    rec[k].append(v)
            rebuilt.attach_cost(cmap, [start], [goal], waypoints, L.LONGSAFE, 1e4)    # untimed: release the rebuilt map
            fresh[0].close()
        route_in = [a + b for a, b in zip(rec["update"], rec["run1_after_update"])]
        route_re = [a + b + c for a, b, c in zip(rec["from_occupancy"], rec["attach_cost"], rec["run1_after_rebuild"])]
        res = {"map": label, "box_cells_per_axis": s, "box_lo_xyz": list(lo), "repetitions": reps,
               "in_place": {"update": stats(rec["update"]), "run1_after": stats(rec["run1_after_update"]),
                            "update_plus_run1": stats(route_in)},
               "rebuild": {"from_occupancy": stats(rec["from_occupancy"]), "attach_cost": stats(rec["attach_cost"]),
                           "first_run1": stats(rec["run1_after_rebuild"]), "total": stats(route_re)},
               "speedup_of_median_route": round(float(np.median(route_re) / np.median(route_in)), 2)}
        print(json.dumps(res), flush=True)
        out.append(res)
    for h in (inplace, rebuilt, cmap):
        h.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps({"card": info}), flush=True)
    results = []
    start, goal = (64.0, 64.0), (4096 - 64.0, 4096 - 64.0)
    occ = maps.random_boxes_occupancy((4096, 4096), 2048, 8, 128, 42, border=2, clear=[(start, 64.0), (goal, 64.0)])
    results += measure("C2: 4096^2, f32, clamp 256", occ, 256.0, "f32", start, goal, 200,
                       dict(lam=1024, m=40, sigma0=16.0, seed=1), (16, 64, 256), args.reps)
    start, goal = (16.0, 16.0, 16.0), (512 - 16.0, 512 - 16.0, 512 - 16.0)
    occ = maps.random_boxes_occupancy((512, 512, 512), 4096, 4, 48, 43, border=0, clear=[(start, 12.0), (goal, 12.0)])
    results += measure("C4: 512^3, u8 (1/4 cell), clamp 64", occ, 64.0, "u8", start, goal, 500,
                       dict(lam=8192, m=77, sigma0=8.0, seed=43), (16, 64), args.reps)
    doc = {"tool": "tools/map_update_timing.py", "card": info, "clock": "host perf_counter around synchronous calls",
           "results": results}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)


if __name__ == "__main__":
    main()
