import os, sys, time, torch, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'colvars-finder_b200'))
import __graft_entry__ as g; g.build()
import bench
dev = torch.device('cuda', 0)
for wl, n in (('c1', 1000), ('c3', 20000), ('c2', 20000), ('c4', 20000)):
    step, X, w, task = bench.build_workload(wl, n, dev, seed=1)
    for _ in range(20): step(X, w)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    N = 200
    for _ in range(N): step(X, w)
    torch.cuda.synchronize(); t1 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    print(wl, n, 'us/step', round((t1 - t0) / N * 1e6, 1), 'frames/s', round(n * N / (t1 - t0) / 1e6, 2), 'M', flush=True)
