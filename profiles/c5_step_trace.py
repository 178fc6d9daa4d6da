import os, sys, time, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'colvars-finder_b200'))
import __graft_entry__ as g; g.build()
import bench, gc
dev = torch.device('cuda', 0)
step, X, w, task = bench.build_workload('c5', 1 << 16, dev, seed=1)
for _ in range(3): step(X, w)
torch.cuda.synchronize()
gc.collect(); gc.disable()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(11)]
t_host = []
ev[0].record()
for i in range(10):
    t0 = time.perf_counter(); step(X, w); t_host.append(time.perf_counter() - t0); ev[i + 1].record()
torch.cuda.synchronize()
print('gpu ms per step', [round(ev[i].elapsed_time(ev[i + 1]), 2) for i in range(10)])
print('host ms per step', [round(1e3 * t, 2) for t in t_host], flush=True)
