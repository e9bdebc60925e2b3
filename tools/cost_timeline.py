"""Per-CTA phase timeline of k_cost on the C2 shape (LMCMA_B200_DBG=1) and, optionally, a C3-shaped batch.
  LMCMA_B200_DBG=1 python tools/cost_timeline.py [batch]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("LMCMA_B200_DBG", "1")
import numpy as np
import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import maps

batch = int(sys.argv[1]) if len(sys.argv) > 1 else 1
W, M = 200, 40
dist, start, goal = maps.config2_map()
lo, hi = maps.box_bounds((4096, 4096), W)
cm = L.CostMap(dist, "f32")
if batch == 1:
    opt = L.Optimizer(2 * W, x0=maps.straight_line(start, goal, W), lam=1024, m=M, lo=lo, hi=hi, sigma0=32.0, seed=1)
    opt.attach_cost(cm, [start], [goal], W, L.LONGSAFE, 1e4)
else:
    starts, goals = maps.random_queries(dist, batch, seed=7, min_sep=1024)
    x0 = np.stack([maps.straight_line(starts[q], goals[q], W) for q in range(batch)])
    opt = L.Optimizer(2 * W, x0=x0, lam=64, m=M, batch=batch, lo=lo, hi=hi, sigma0=32.0, seed=7)
    opt.attach_cost(cm, starts, goals, W, L.LONGSAFE, 1e4)
opt.run(45)
for _ in range(3):
    pk = opt.profile_kernels(1)
print("per-kernel ms:", {k: round(v, 4) for k, v in pk.items()}, "sigma", float(opt.get("sigma")[0]), "nsamp", float(opt.get("nsamp").mean()))
