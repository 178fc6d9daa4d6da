#!/usr/bin/env python
"""bench.py -- train-step throughput (frames/s) of the colvars-finder step on B200, one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c1|c4] [--impl reference] [--dump-outputs DIR]

A step is the body of the reference's mini-batch loop (core.py:498-522 / 699-712): zero_grad, loss,
backward, optimizer.step -- through the drop-in classes, on one batch of synthetic frames per GPU
(SURVEY.md section 8d).  Default workload C3: alanine-dipeptide-sized frames (22 atoms, Kabsch on all atoms,
position features d_r = 66), EigenFunctions([66,20,20,20,1], k=3), generator loss, Boltzmann weights.
Weak scaling: every rank keeps `--frames` frames (default 2^22, 1.1 GB > L2) resident in its own HBM.

`value`   : frames/s with the batch resident in HBM (CUDA events, max over ranks).
`e2e`     : frames/s with the batch in pinned HOST memory, H2D copy + step + D2H of the loss inside the timed region.
`roofline`: the dominant kernel (most device time per step in the library's own launch accounting, CUDA events around
            every launch on the launching stream, measured in a separate profiled run of K steps): algorithmic bytes
            = SURVEY 8d's per-frame figure x frames, against the measured HBM peak.  `roofline_fp32` puts the kernel and
            the whole step against the fp32 FMA peak measured in the same run (cvf_fma_probe), which is the roofline
            that actually binds this path (SURVEY.md section 8d); `kernels` lists every kernel's share of the step.
`scaling_strong` (N-GPU runs of C1-C4): the same step on SURVEY 8d's fixed global batch of 2^23 frames split over the ranks.
`dp_parity` (N > 1): before the timed region, one common batch is run once on a single rank's worth of code (collectives off)
            and once sharded over the ranks with the NCCL all-reduces; loss, eigenvalues and gradients must agree.
`native`  : source hash stamped into libcvf_sm100.so and whether it equals the hash of the sources next to it.
`cpu_baseline` / `--impl reference`: oracle/ref_torch.py (restatement of the reference's PyTorch path; /root/reference does
            not exist on the GPU box) on the host cores, on a bounded sample of the same workload.  Only these two legs
            import oracle/.
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step computed to DIR/<name>.npy (float32 or
            float64): the step's return values, every parameter gradient and every parameter after the optimizer update
            (see dump_outputs).  The inputs depend on the arguments only, so two builds can be compared output for output.

The library must have been built (__graft_entry__.build()) from the sources next to it; bench.py compiles nothing and writes
nothing into the tree (the tasks' log directory is a temporary directory).
"""
from __future__ import annotations

import argparse
import atexit
import gc
import signal
import ctypes as C
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True      # the tree may be read-only and is left as build() made it
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "colvars-finder_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (description, bytes/frame, flops/frame of one step) -- SURVEY.md section 8d
    "c3": ("alanine-dipeptide EigenFunctionTask, generator loss, k=3, 22-atom Kabsch, position features (d_r=66), "
           "nets [66,20,20,20,1]", 268, 97400),
    "c2": ("alanine-dipeptide AutoEncoderTask step on aligned positions (d_r=66), enc [66,20,20,20,2], dec [2,10,10,66]",
           268, 17640),
    "c1": ("2-d EigenFunctionTask, generator loss, k=1, Identity pre-processing, net [2,20,20,20,1]", 12, 12040),
    "c4": ("166-atom chain EigenFunctionTask, generator loss, k=3, 45 distances + 18 dihedrals (d_r=81), "
           "nets [81,20,20,20,1]", 1996, 128500),
    "c5": ("1000-atom AutoEncoderTask step on position features (d_r=3000), enc [3000,512,512,2], dec [2,512,512,3000]; "
           "layer-wise products on tcgen05 tensor cores (3 x TF32 split, fp32 accumulation in tensor memory)", 12004, 21590016),
    "c2p": ("alanine-dipeptide AutoEncoderTask pre-pass (core.py:635): Kabsch alignment of every frame onto the reference, "
            "22 atoms, aligned positions out (one pass over the trajectory, HBM-bound)", 528, 1500),
}
METRIC = "train-step frames/sec"
# fp32 flops per frame (FMA = 2) of the kernels that can dominate a step; derivation in DESIGN.md ("work per frame")
KERNEL_FLOPS = {
    # fast_pass2 = tangent forward (the primal activations come back from pass 1), reverse sweep of (G, s), every weight-gradient
    # outer product incl. dW_1: the flops the kernel EXECUTES (it is bound by the shared-memory pipe, DESIGN.md 5 (d))
    ("c3", "fast_pass2"): 45240 + 15840 - 12720, ("c3", "fast_pass1"): 25680,
    ("c1", "fast_pass2"): 5240 - 1680, ("c1", "fast_pass1"): 1760,
    ("c4", "fast_pass2"): 48720 + 19440 - 14520, ("c4", "fast_pass1"): 29160,
    ("c2", "ae_fast_main"): 9120, ("c2", "ae_fast_dw"): 6176,   # forward P + delta sweep (P - first layer); weight + bias products
}
def measured_traffic(workload, kernel, frames):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel`, from the `ncu --set full` capture of this very
    command that profiles/ncu_traffic.py condensed into profiles/ncu_traffic.json -- used only when the capture was taken at
    the same workload, frame count and source hash as the running library; None otherwise (no stale constants)."""
    try:
        import __graft_entry__ as entry
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tab = json.load(f)
        if tab.get("source_hash") != entry.library_hash() or tab.get("workload") != workload or tab.get("frames") != frames:
            return None, "no ncu capture of this build (profiles/ncu_traffic.json is of another source hash / size)"
        v = tab["kernels"].get(kernel)
        return (None, "kernel not in the capture") if v is None else (float(v), f"ncu --set full capture {tab.get('capture')}")
    except Exception as exc:
        return None, f"no capture table ({type(exc).__name__})"


# ------------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  The sampler is started before
    the warm-up steps (nvidia-smi needs ~0.1 s to start) and `mark()` / `stop()` bracket the timed region; only samples read
    inside the bracket count.  If the region was too short for one, the samples of the warm-up steps (same load) are used and
    the result says so."""

    # SM clock and the throttle-reason BITMASK only: every extra field is another driver query, and a query can hold up kernel
    # dispatch for milliseconds (visible on steps made of a hundred launches).  Bits: 0x4 sw_power_cap, 0x8 hw_slowdown,
    # 0x20 sw_thermal_slowdown, 0x40 hw_thermal_slowdown (nvml.h nvmlClocksEventReason*).
    Q = "index,clocks.sm,clocks.max.sm,clocks_event_reasons.active"
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t_mark = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def mark(self):
        """Start of the timed region.  The sampler is paused until `resume()`: an NVML query can hold up this process's kernel
        launches for milliseconds, which is invisible once the launch queue is a step deep but not while it is being filled
        from empty right after the barrier."""
        self.t_mark = time.perf_counter()
        if self.proc is not None:
            try:
                self.proc.send_signal(signal.SIGSTOP)
            except Exception:
                pass

    def resume(self):
        if self.proc is not None:
            try:
                self.proc.send_signal(signal.SIGCONT)
            except Exception:
                pass

    def stop(self):
        t_end = time.perf_counter()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.resume()
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0 = self.t_mark if self.t_mark is not None else 0.0
        inside = [r for t, r in self.rows if t0 <= t <= t_end + 0.05]
        window = "timed region"
        if not inside:
            inside, window = [r for _, r in self.rows], "warm-up + timed region (timed region shorter than one sampling period)"
        sm, mx, reasons = [], None, set()
        for r in inside:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                mask = int(r[3], 16) if r[3].lower().startswith("0x") else 0
                for name, bit in self.BITS:
                    if mask & bit:
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def bind_to_gpu_numa_node(index):
    """Pin this process (and, by first touch, the pinned host buffers it allocates next) to the NUMA node of GPU `index`: with one
    process per GPU, eight ranks streaming their batches out of one node's memory share that node's bandwidth (r01: 23 GB/s per
    GPU at N = 8).  Returns a short description for the JSON line; silently does nothing where sysfs does not say."""
    try:
        pr = torch.cuda.get_device_properties(index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return "numa node unknown"
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"numa node {node}: none of its cores is available to this process"
        os.sched_setaffinity(0, cpus)
        return f"bound to numa node {node} ({len(cpus)} cores)"
    except Exception as exc:
        return f"not bound ({type(exc).__name__})"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def build_workload(name, n_frames, dev, seed, lr=1e-3):
    """Returns (step_fn(X, w) -> loss tensor, X, w, task).  step_fn.last holds what the caller of the step's path received in
    the latest call (the return values of loss_func / weighted_MSE_loss / Align), by name."""
    from colvarsfinder import core, nn, utils
    import bench_data as bd
    FakeTrajectory = bd.SyntheticTrajectory
    torch.manual_seed(2026)
    tmp = tempfile.mkdtemp(prefix="cvf_bench_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    last = {}
    if name == "c2p":
        base = bd.DIPEPTIDE_NM * 10.0
        X = bd.frames(base, n_frames, dev, seed)
        w = torch.ones(n_frames, device=dev)
        align = utils.Align(base, list(range(22))).to(dev)

        out = torch.empty_like(X)

        def step(Xb, wb):
            last["aligned"] = align(Xb, out=out)
            return last["aligned"][0, 0, 0]
        step.last = last
        return step, X, w, None
    if name in ("c3", "c2"):
        base = bd.DIPEPTIDE_NM * 10.0
        X = bd.frames(base, n_frames, dev, seed)
        w = bd.boltzmann_weights(n_frames, dev, seed) if name == "c3" else torch.ones(n_frames, device=dev)
        small = FakeTrajectory(X[:1024].cpu().numpy(), np.ones(1024), dt=1.0)
        align = utils.Align(base, list(range(22)))
        if name == "c3":
            model = nn.EigenFunctions([66, 20, 20, 20, 1], 3)
            task = core.EigenFunctionTask(small, align, model, tmp, 20.0, [1.0, 0.6, 0.3], k=3, learning_rate=lr, device=dev,
                                          verbose=False, debug_mode=False)
        else:
            model = nn.AutoEncoder([66, 20, 20, 20, 2], [2, 10, 10, 66])
            task = core.AutoEncoderTask(small, align, model, tmp, learning_rate=lr, device=dev, verbose=False, debug_mode=False)
            X = task.preprocessing_layer(X).reshape(n_frames, 66).contiguous()   # the pre-pass is outside the step (core.py:635)
    elif name == "c5":
        g = torch.Generator(device=dev).manual_seed(seed)
        X = torch.randn(n_frames, 3000, generator=g, device=dev)          # features of the pre-pass (core.py:635) directly
        w = torch.ones(n_frames, device=dev)
        small = FakeTrajectory(X[:256].cpu().numpy(), np.ones(256), dt=1.0)
        model = nn.AutoEncoder([3000, 512, 512, 2], [2, 512, 512, 3000])
        task = core.AutoEncoderTask(small, torch.nn.Identity(), model, tmp, learning_rate=lr, device=dev, verbose=False,
                                    debug_mode=False)
    elif name == "c1":
        X = bd.ring_2d(n_frames, dev, seed)
        w = torch.ones(n_frames, device=dev)
        small = FakeTrajectory(X[:1024].cpu().numpy(), np.ones(1024), dt=0.1)
        model = nn.EigenFunctions([2, 20, 20, 20, 1], 1)
        task = core.EigenFunctionTask(small, torch.nn.Identity(), model, tmp, 20.0, [1.0], k=1, learning_rate=lr, device=dev,
                                      verbose=False, debug_mode=False)
    elif name == "c4":
        base = bd.chain_structure(166, seed=2026)
        X = bd.frames(base, n_frames, dev, seed)
        w = bd.boltzmann_weights(n_frames, dev, seed)
        feats, align_idx = bd.c4_features()
        pp = utils.Preprocessing(utils.Align(base[align_idx], align_idx), utils.FeatureMap(feats))
        small = FakeTrajectory(X[:1024].cpu().numpy(), np.ones(1024), dt=1.0)
        model = nn.EigenFunctions([81, 20, 20, 20, 1], 3)
        task = core.EigenFunctionTask(small, pp, model, tmp, 20.0, [1.0, 0.6, 0.3], k=3, learning_rate=lr, device=dev,
                                      verbose=False, debug_mode=False)
    else:
        raise SystemExit(f"unknown workload {name}")

    if isinstance(task, core.EigenFunctionTask):
        def step(Xb, wb):
            task.optimizer.zero_grad(set_to_none=True)
            out = task.loss_func(Xb, wb, None, None)
            out[0].backward()
            task.optimizer.step()
            last["loss"], last["eig"], last["obj"], last["pen"], last["cvec"] = out
            return out[0]
    else:
        def step(Xb, wb):
            task.optimizer.zero_grad(set_to_none=True)
            loss = task.weighted_MSE_loss(Xb, wb)
            loss.backward()
            task.optimizer.step()
            last["loss"] = loss
            return loss
    step.last = last
    return step, X, w, task


DUMP_MAX_ELEMENTS = 1 << 22     # per array; larger outputs are sampled by rows
DUMP_MAX_BYTES = 64 << 20       # all files together


def dump_outputs(path, step, task):
    """Write what the latest call of `step` computed to path/<name>.npy: the tensors in step.last, then grad.<parameter>
    and param.<parameter> (the gradient of that step and the parameter after its optimizer update) for every parameter of
    the model.  float64 stays float64, everything else is written as float32.  An array of more than DUMP_MAX_ELEMENTS
    elements is replaced by the rows np.random.default_rng(0).choice(rows, m, replace=False), sorted, with m the largest row
    count that fits: the same rows for the same shape in every run."""
    arrays = dict(step.last)
    if task is not None:
        for name, p in task.model.named_parameters():
            if p.grad is not None:
                arrays[f"grad.{name}"] = p.grad
            arrays[f"param.{name}"] = p
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.size > DUMP_MAX_ELEMENTS:
            m = max(1, DUMP_MAX_ELEMENTS // (a.size // a.shape[0]))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], m, replace=False))]
        total += a.nbytes
        if total > DUMP_MAX_BYTES:
            raise SystemExit(f"--dump-outputs: the outputs exceed {DUMP_MAX_BYTES >> 20} MB at {name}")
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_run(name, n_frames, steps, warmup, seed=7, dataloader_steps=0):
    """The reference's PyTorch path (oracle/ref_torch.py restatement: autograd through torch.linalg.svd, double
    backward, Adam) on the host cores.  Returns (frames/s, ms/step, cores)."""
    from oracle import ref_torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(2026)
    if name == "c2p":
        base = ref_torch.DIPEPTIDE_NM * 10.0
        X = torch.as_tensor(ref_torch.synth_frames(base, n_frames, seed=seed))
        pp = ref_torch.Preprocess(ref_torch.Align(base, list(range(22))), None)
        times = []
        with torch.no_grad():
            for it in range(warmup + steps):
                t0 = time.perf_counter()
                pp(X)
                if it >= warmup:
                    times.append(time.perf_counter() - t0)
        return n_frames * steps / sum(times), 1e3 * sum(times) / steps, cores
    if name == "c5":
        X = torch.randn(n_frames, 3000)
        w = torch.ones(n_frames)
        pp = None
    elif name in ("c3", "c2"):
        base = ref_torch.DIPEPTIDE_NM * 10.0
        X = torch.as_tensor(ref_torch.synth_frames(base, n_frames, seed=seed))
        w = torch.as_tensor(ref_torch.boltzmann_weights(n_frames, seed=seed)) if name == "c3" else torch.ones(n_frames)
        pp = ref_torch.Preprocess(ref_torch.Align(base, list(range(22))), None)
    elif name == "c1":
        rng = np.random.default_rng(seed)
        th, r = rng.uniform(-np.pi, np.pi, n_frames), rng.normal(1.0, 0.25, n_frames)
        X = torch.as_tensor(np.stack([r * np.cos(th), r * np.sin(th)], 1).astype(np.float32))
        w = torch.ones(n_frames)
        pp = ref_torch.Preprocess()
    else:
        base = ref_torch.chain_structure(166, seed=2026)
        X = torch.as_tensor(ref_torch.synth_frames(base, n_frames, seed=seed))
        w = torch.as_tensor(ref_torch.boltzmann_weights(n_frames, seed=seed))
        import bench_data as bd
        feats, align_idx = bd.c4_features()
        pp = ref_torch.Preprocess(ref_torch.Align(base[align_idx], align_idx), ref_torch.FeatureMap(feats))
    if name in ("c2", "c5"):
        ed, dd = ([66, 20, 20, 20, 2], [2, 10, 10, 66]) if name == "c2" else ([3000, 512, 512, 2], [2, 512, 512, 3000])
        enc = [p.requires_grad_() for p in ref_torch.init_mlp_params(ed)]
        dec = [p.requires_grad_() for p in ref_torch.init_mlp_params(dd)]
        params = enc + dec
        with torch.no_grad():
            Fx = pp(X.double()).float() if pp is not None else X

        def loss_fn():
            return ref_torch.ae_loss(Fx, w, enc, dec)
    else:
        dims = {"c3": [66, 20, 20, 20, 1], "c1": [2, 20, 20, 20, 1], "c4": [81, 20, 20, 20, 1]}[name]
        k = 1 if name == "c1" else 3
        nets = [[p.requires_grad_() for p in ref_torch.init_mlp_params(dims)] for _ in range(k)]
        params = [p for n in nets for p in n]
        eig_w = [1.0, 0.6, 0.3][:k]

        def loss_fn():
            Xr = X.clone().requires_grad_()
            return ref_torch.eigen_loss(Xr, w, nets, pp, 20.0, eig_w)[0]
    opt = torch.optim.Adam(params, lr=1e-3)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = loss_fn()
        loss.backward()
        opt.step()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    if dataloader_steps > 0 and name in ("c1", "c3", "c4"):
        # (ii) of SURVEY 8d: the same step fed by the reference's loader (core.py:470-475: TensorDataset + default collate,
        # shuffle=False, drop_last=True), batch size = the sample
        ds = torch.utils.data.TensorDataset(X.repeat((dataloader_steps,) + (1,) * (X.dim() - 1)), w.repeat(dataloader_steps),
                                            torch.arange(n_frames * dataloader_steps))
        loader = torch.utils.data.DataLoader(dataset=ds, batch_size=n_frames, drop_last=True, shuffle=False)
        t0 = time.perf_counter()
        for Xb, wb, _ in loader:
            opt.zero_grad(set_to_none=True)
            Xr = Xb.clone().requires_grad_()
            loss = ref_torch.eigen_loss(Xr, wb, nets, pp, 20.0, eig_w)[0]
            loss.backward()
            opt.step()
        cpu_reference_run.dataloader_fps = n_frames * dataloader_steps / (time.perf_counter() - t0)
    return n_frames * steps / total, 1e3 * total / steps, cores


# ------------------------------------------------------------------------------------------------ multi-GPU checks
def _loss_and_grads(task, X, w):
    from colvarsfinder import core
    task.optimizer.zero_grad(set_to_none=True)
    if isinstance(task, core.EigenFunctionTask):
        out = task.loss_func(X, w, None, None)
        loss, eig = out[0], out[1].double()
    else:
        loss, eig = task.weighted_MSE_loss(X, w), torch.zeros(1, dtype=torch.float64, device=X.device)
    loss.backward()
    g = torch.cat([p.grad.reshape(-1) for p in task.model.parameters()]).double()
    task.optimizer.zero_grad(set_to_none=True)
    return loss.detach().double(), eig, g


def dp_parity_check(task, X, w, rank, world, frames=1 << 18):
    """N ranks on shards of ONE common batch (NCCL all-reduce of batch sums and gradient sums) against the same batch on one
    rank (collectives off): loss, eigenvalues, gradients.  Outside the timed region; parameters are not updated."""
    import torch.distributed as dist
    from colvarsfinder import _ops
    n = min(frames, X.shape[0])
    n -= n % (512 * world)
    Xc, wc = X[:n].clone(), w[:n].clone()
    dist.broadcast(Xc, 0)
    dist.broadcast(wc, 0)
    with _ops.no_collectives():
        l1, e1, g1 = _loss_and_grads(task, Xc, wc)
    lo, hi = _ops.shard_range(n, rank, world)
    l2, e2, g2 = _loss_and_grads(task, Xc[lo:hi].contiguous(), wc[lo:hi].contiguous())
    res = {"frames": n, "loss_rel": float((l1 - l2).abs() / l1.abs()),
           "eig_rel_max": float(((e1 - e2).abs() / e1.abs().clamp_min(1e-300)).max()),
           "grad_rel_l2": float((g1 - g2).norm() / g1.norm())}
    worst = torch.tensor([res["loss_rel"], res["eig_rel_max"], res["grad_rel_l2"]], dtype=torch.float64, device=X.device)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    res.update(loss_rel=float(worst[0]), eig_rel_max=float(worst[1]), grad_rel_l2=float(worst[2]))
    # fp32 sums inside a 512-frame tile are identical (shard boundaries are tile boundaries); only the fp64 order differs
    res["ok"] = bool(worst[0] < 1e-6 and worst[1] < 1e-6 and worst[2] < 1e-6)
    if not res["ok"]:
        raise SystemExit(f"data-parallel parity check failed: {res}")
    return res


# ------------------------------------------------------------------------------------------------ main
def _quiet_stdout():
    """Route everything libraries print on file descriptor 1 (e.g. NCCL's version banner) to stderr; returns a writer for
    the one JSON line, so that stdout carries nothing else."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(saved, "w")

    def emit(obj):
        out.write(json.dumps(obj) + "\n")
        out.flush()
    return emit


def main():
    emit = _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))   # c2p: the HBM-bound alignment pre-pass alone
    ap.add_argument("--frames", type=int, default=None, help="frames per GPU per step (default 2^22; 2^16 for c5)")
    ap.add_argument("--cpu-frames", type=int, default=None, help="frames per step of the CPU sample (default 100000; 4096 for c5)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--strong", action="store_true", help="also time the 2^23-frame global batch of SURVEY 8d at N = 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world, local = dist_env()
    if args.frames is None:
        args.frames = 1 << 16 if args.workload == "c5" else 1 << 22
    if args.cpu_frames is None:
        args.cpu_frames = 4096 if args.workload == "c5" else 100000
    desc, bytes_per_frame, flops_per_frame = WORKLOADS[args.workload]
    config = {"workload": f"{args.workload.upper()}: {desc}", "frames_per_gpu_per_step": args.frames,
              "global_batch": args.frames * max(world, 1), "optimizer": "Adam", "parallelism": f"dp{max(world, 1)}",
              "l2_policy": "inputs larger than L2 (no flush needed)"}
    if args.frames * bytes_per_frame < 160e6:
        config["l2_policy"] = "batch smaller than L2: steps are back to back on the same batch (intermediates exceed L2)"

    if args.impl == "reference":
        if rank != 0:
            return
        w_ = max(args.warmup, 1)
        fps, ms, cores = cpu_reference_run(args.workload, args.cpu_frames, args.steps, w_)
        sample = (f"{args.cpu_frames} frames/step x {args.steps} steps (+{w_} warm-up) of the same synthetic workload, "
                  "oracle/ref_torch.py (PyTorch CPU autograd restatement of core.py:387-457,517 + Adam)")
        config["frames_per_gpu_per_step"] = args.cpu_frames
        config["global_batch"] = args.cpu_frames
        emit(({"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": w_, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
                          "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    import __graft_entry__ as entry
    if entry.library_hash() != entry.source_hash():
        raise SystemExit(f"{entry.LIB} is missing or was built from other sources: run __graft_entry__.build() first")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    from colvarsfinder import _lib

    # started early: nvidia-smi takes a while to deliver its first row (CVF_BENCH_CLOCKS=0 switches the sampling off)
    sampler = ClockSampler(local).start() if rank == 0 and os.environ.get("CVF_BENCH_CLOCKS", "1") != "0" else None
    # strong scaling (SURVEY 8d): the global batch of 2^23 frames split over the ranks, next to the weak-scaling headline
    strong_frames = (1 << 23) // world if args.workload in ("c1", "c2", "c3", "c4") and (world > 1 or args.strong) else 0
    step, X_all, w_all, task = build_workload(args.workload, max(args.frames, strong_frames), dev, seed=2026 + rank)
    X, w = X_all[:args.frames], w_all[:args.frames]
    W = max(args.warmup, 3)
    K = args.steps
    dp_parity = None
    if world > 1 and task is not None:
        dp_parity = dp_parity_check(task, X, w, rank, world)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- resident-in-HBM throughput
    for _ in range(W):
        step(X, w)
    barrier()
    _lib.profile_read(reset=True)      # launch counters to zero: the timed region is counted exactly
    if sampler:
        sampler.mark()
    # the launch queue is empty at this point: a pause of the host (a full garbage collection takes tens of milliseconds in a
    # process with torch loaded) would leave the GPU idle for as long, so collect now and keep the collector off while timing
    gc.collect()
    gc.disable()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        loss = step(X, w)
        if sampler and i == min(1, K - 1):
            sampler.resume()      # the queue now holds a step or two of GPU work
    e1.record()
    barrier()
    gc.enable()
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    clocks = sampler.stop() if sampler else None
    if world > 1:
        torch.distributed.all_reduce(ms_total, op=torch.distributed.ReduceOp.MAX)
    ms_total = float(ms_total)
    value = args.frames * world * K / (ms_total * 1e-3)
    final_loss = float(loss.detach())
    launches_timed = sum(v[2] for v in _lib.profile_read(reset=True).values())
    if args.dump_outputs and rank == 0:      # before the steps below change the parameters
        dump_outputs(args.dump_outputs, step, task)

    # ---- end to end: batch in pinned host memory, H2D + step + D2H(loss) per step, copy of step i+1 overlapped
    numa = bind_to_gpu_numa_node(local) if world > 1 else "single process: not bound"
    hosts = [torch.empty(X.shape, dtype=X.dtype).pin_memory() for _ in range(2)]
    hw = [torch.empty(w.shape, dtype=w.dtype).pin_memory() for _ in range(2)]
    for hb, hwb in zip(hosts, hw):
        hb.copy_(X)
        hwb.copy_(w)
    devb = [torch.empty_like(X) for _ in range(2)]
    devw = [torch.empty_like(w) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    h2d = X.numel() * 4 + w.numel() * 4

    def enqueue_copy(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[b])
            devb[b].copy_(hosts[b], non_blocking=True)
            devw[b].copy_(hw[b], non_blocking=True)
            ready[b].record(copy_stream)

    def e2e_loop(n):
        cur = torch.cuda.current_stream()
        for b in range(2):
            freed[b].record(cur)
        enqueue_copy(0)
        for i in range(n):
            b = i % 2
            if i + 1 < n:
                enqueue_copy(i + 1)
            cur.wait_event(ready[b])
            l = step(devb[b], devw[b])
            freed[b].record(cur)
            loss_host.copy_(l.detach(), non_blocking=True)
        torch.cuda.synchronize()

    e2e_loop(2)
    barrier()
    gc.collect()
    gc.disable()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    e2e_loop(K)
    t1.record()
    barrier()
    gc.enable()
    ms_e2e = torch.tensor([t0.elapsed_time(t1)], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(ms_e2e, op=torch.distributed.ReduceOp.MAX)
    e2e_value = args.frames * world * K / (float(ms_e2e) * 1e-3)
    del hosts, hw, devb, devw

    # ---- strong scaling: global batch 2^23 fixed, K_s steps (>= 50: at N > 1 one host hiccup must not dominate)
    strong = None
    if strong_frames:
        Xs, ws_ = X_all[:strong_frames], w_all[:strong_frames]
        K_s = max(K, 50) if world > 1 else K
        for _ in range(3):
            step(Xs, ws_)
        barrier()
        gc.collect()
        gc.disable()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(K_s):
            step(Xs, ws_)
        s1.record()
        barrier()
        gc.enable()
        ms_s = torch.tensor([s0.elapsed_time(s1)], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(ms_s, op=torch.distributed.ReduceOp.MAX)
        strong = {"global_batch": strong_frames * world, "frames_per_gpu_per_step": strong_frames, "steps": K_s,
                  "ms_per_step": float(ms_s) / K_s, "value": strong_frames * world * K_s / (float(ms_s) * 1e-3), "unit": "frames/s"}

    # ---- per-kernel device time: K more steps with a CUDA-event pair around every launch of the library
    L = _lib.lib()
    _lib.check(L.cvf_profile_enable(1), "cvf_profile_enable")
    for _ in range(K):
        step(X, w)
    torch.cuda.synchronize()
    prof = {k_: v for k_, v in _lib.profile_read(reset=True).items() if v[1] > 0}
    _lib.check(L.cvf_profile_enable(0), "cvf_profile_enable")
    dom_name = max(prof, key=lambda k_: prof[k_][0])
    kern_ms = prof[dom_name][0] / prof[dom_name][1]
    step_kernel_ms = sum(v[0] for v in prof.values()) / K
    rank_kernel_ms = None
    if world > 1:      # every rank's own kernel time per step: tells a slow GPU (all ranks wait for it at the all-reduces) from waiting
        t = torch.zeros(world, dtype=torch.float64, device=dev)
        t[rank] = step_kernel_ms
        torch.distributed.all_reduce(t)
        rank_kernel_ms = [round(float(v), 4) for v in t]
    # ---- fp32 FMA peak probe
    sink = torch.zeros(4, device=dev)
    flops = C.c_double(0.0)
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(2):
        _lib.check(L.cvf_fma_probe(sink.data_ptr(), 20000, C.byref(flops), stream), "cvf_fma_probe")
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(3):
        _lib.check(L.cvf_fma_probe(sink.data_ptr(), 20000, C.byref(flops), stream), "cvf_fma_probe")
    p1.record()
    torch.cuda.synchronize()
    fma_peak = 3 * flops.value / (p0.elapsed_time(p1) * 1e-3) / 1e12

    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    hbm_peak, peak_src = measured_peaks()
    traffic, traffic_src = measured_traffic(args.workload, dom_name, args.frames)
    achieved = bytes_per_frame * args.frames / (kern_ms * 1e-3) / 1e9
    step_tflops = value / world * flops_per_frame / 1e12
    dom_flops = KERNEL_FLOPS.get((args.workload, dom_name))
    out = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config, "clocks": clocks, "final_loss": final_loss,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": 4 * world,
                "ms_per_step": float(ms_e2e) / K, "host_memory": numa},
        "gpu_launches": launches_timed * world,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": dom_name, "kernel_ms": kern_ms,
                     "kernel_share_of_step": prof[dom_name][0] / K / step_kernel_ms, "peak_source": peak_src,
                     "note": ("HBM-bound kernel: algorithmic bytes = frame read + aligned frame written" if args.workload == "c2p" else
                              "this path is fp32-FMA bound, not HBM bound (SURVEY 8d): see roofline_fp32")},
        "roofline_fp32": {"bound": "fp32_fma", "peak": fma_peak, "unit": "TFLOP/s",
                          "peak_source": "cvf_fma_probe measured in this run",
                          "step": {"achieved": step_tflops, "frac": step_tflops / fma_peak, "flops_per_frame": flops_per_frame},
                          "kernel": None if dom_flops is None else {
                              "name": dom_name, "flops_per_frame": dom_flops,
                              "achieved": dom_flops * args.frames / (kern_ms * 1e-3) / 1e12,
                              "frac": dom_flops * args.frames / (kern_ms * 1e-3) / 1e12 / fma_peak}},
        "kernels": {k_: {"ms_per_step": v[0] / K, "launches_per_step": v[1] / K} for k_, v in sorted(prof.items())},
        "native": {"so": "colvars-finder_b200/colvarsfinder/libcvf_sm100.so", "source_hash": entry.library_hash(),
                   "matches_sources": entry.library_hash() == entry.source_hash()},
    }
    if rank_kernel_ms is not None:
        out["kernel_ms_per_step_by_rank"] = rank_kernel_ms
    if strong is not None:
        out["scaling_strong"] = strong
    if dp_parity is not None:
        out["dp_parity"] = dp_parity
    if args.workload == "c5":
        # the layer products run on the tensor cores as three TF32 passes: the fp32-equivalent ceiling is the measured dense
        # bf16 rate / 2 (TF32 runs at half the bf16 rate) / 3 (passes)
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                bf16 = float(json.load(f)["bf16_tflops_sustained"])
            src = "MEASURED_PEAKS.json bf16_tflops_sustained / 2 (TF32) / 3 (split passes)"
        except Exception:
            bf16, src = 1379.4, "fallback 1379.4 TF/s bf16 / 2 / 3"
        peak = bf16 / 6.0
        out["roofline"] = {"bound": "tensor", "achieved": step_tflops, "peak": peak, "unit": "TFLOP/s", "frac": step_tflops / peak,
                           "traffic": None, "kernel": "ae_step (tcgen05 3xTF32 products + transposes, whole step)",
                           "kernel_ms": kern_ms, "kernel_share_of_step": prof[dom_name][0] / K / step_kernel_ms,
                           "peak_source": src,
                           "note": "achieved = algorithmic fp32 flops of the step (6P per frame) per second; tensor-pipe active "
                                   "cycles per product kernel are in profiles/"}
    if not args.no_cpu_baseline:
        fps, ms, cores = cpu_reference_run(args.workload, args.cpu_frames, 5, 1, dataloader_steps=2)
        out["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                               "sample": f"{args.cpu_frames} frames/step x 5 steps (+1 warm-up), oracle/ref_torch.py on the host"}
        dl = getattr(cpu_reference_run, "dataloader_fps", None)
        if dl is not None:
            out["cpu_baseline"]["dataloader_value"] = dl
            out["cpu_baseline"]["dataloader_sample"] = (f"2 batches of {args.cpu_frames} frames through the reference's DataLoader "
                                                        "(TensorDataset, default collate, core.py:470-475) + the same step")
    emit(out)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
