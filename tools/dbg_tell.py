"""Device timeline of tell_all on the C2 shape (k_update / k_rank / k_sample globaltimer stamps, printed by lmcma_b200_sync):
  LMCMA_B200_DBG=1 python tools/dbg_tell.py [flush]     flush: 256 MiB fill before every generation"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, bench
import torch
import lmcma_path_planner_b200 as L
flush = len(sys.argv) > 1 and sys.argv[1] == "flush"
dist, start, goal, lo, hi, x0 = bench.build_problem()
cmap = L.CostMap(dist, "f32")
opt = L.Optimizer(2 * bench.W, x0=x0, lam=bench.LAM, m=bench.M, lo=lo, hi=hi, sigma0=bench.SIGMA0, seed=1000)
buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for g in range(64):
    X = opt.ask_all()[0]
    r = cmap.evaluate(X, start, goal, bench.W, L.LONGSAFE, 1e4)
    if g >= 60:
        if flush:
            buf.fill_(1); torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt.tell_all(r["f"])
        t1 = time.perf_counter()
        opt.sync()
        print("tell_all wall us", (t1 - t0) * 1e6, file=sys.stderr)
    else:
        opt.tell_all(r["f"])
