import os, sys, time, torch, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'colvars-finder_b200'))
import __graft_entry__ as g; g.build()
import bench, bench_data as bd
dev = torch.device('cuda', 0)
for wl, n in (('c3', 10_000_000), ('c4', 8_000_000)):
    step, X, w, task = bench.build_workload(wl, n, dev, seed=1)
    torch.cuda.synchronize(); t0 = time.time()
    l1 = step(X, w); torch.cuda.synchronize(); t1 = time.time()
    l2 = step(X, w); torch.cuda.synchronize(); t2 = time.time()
    # additivity of the batch sums at full size
    ctx = task._ctx
    _, s_all = ctx.stats(X, w)
    h = n // 2 + 12345
    _, s1 = ctx.stats(X[:h], w[:h]); _, s2 = ctx.stats(X[h:], w[h:])
    rel = ((s1 + s2 - s_all).abs() / s_all.abs().clamp_min(1e-300)).max().item()
    print(wl, n, 'loss', float(l1), float(l2), 'step s', round(t2 - t1, 4), 'frames/s', round(n / (t2 - t1) / 1e6, 1), 'M  additivity rel', rel,
          'mem GB', round(torch.cuda.max_memory_allocated() / 1e9, 1), flush=True)
    del step, X, w, task, ctx
    torch.cuda.empty_cache()
