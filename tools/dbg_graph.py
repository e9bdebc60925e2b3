"""Device timeline of the fused C2 generation (k_update / k_rank / k_sample globaltimer stamps, printed by lmcma_b200_sync):
  LMCMA_B200_DBG=1 python tools/dbg_graph.py [flush]     flush: 256 MiB fill before every generation"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, bench
import torch
import lmcma_path_planner_b200 as L
flush = len(sys.argv) > 1 and sys.argv[1] == "flush"
dist, start, goal, lo, hi, x0 = bench.build_problem()
cmap = L.CostMap(dist, "f32")
opt = L.Optimizer(2 * bench.W, x0=x0, lam=bench.LAM, m=bench.M, lo=lo, hi=hi, sigma0=bench.SIGMA0, seed=1000)
opt.attach_cost(cmap, [start], [goal], bench.W, L.LONGSAFE, 1e4)
buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
opt.run(60); opt.sync()
for _ in range(3):
    if flush:
        buf.fill_(1); torch.cuda.synchronize()
    opt.run(1); opt.sync()
    print("last_run_ms", opt.last_run_ms(), file=sys.stderr)
