"""Kernel times of the pre-processing backward (cvf_align_vjp, cvf_features_vjp) next to the matching forwards, with CUDA events.

Workloads: C2 (Align, 22 atoms, 2^22 frames), C5 (Align, 1000 atoms, 2^16 frames) and C4 (features + alignment of the 166-atom
chain, 2^22 frames).  Every input is larger than the 126 MB L2, so each launch streams from HBM; each kernel is warmed up, then
timed over --reps back-to-back launches.  Algorithmic bytes per frame: Align forward 24 N (x read, y written), Align backward
36 N (x and g_y read, g_x written); features forward 12 n_used + 4 d_r, features backward 12 n_used + 4 d_r + 12 N.  The
fraction of peak is against bench.measured_peaks().  The device name and power limit are read in the same run.

    python profiles/preproc_vjp_bench.py [--out profiles/preproc_vjp_bench.json] [--reps 20]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "colvars-finder_b200"))

import torch  # noqa: E402

import bench  # noqa: E402
import bench_data as bd  # noqa: E402


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=60).stdout.strip()
        return out or "not measured"
    except (OSError, subprocess.SubprocessError):
        return "not measured"


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "preproc_vjp_bench.json"))
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    from colvarsfinder import _lib, _ops, utils
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    peak, peak_src = bench.measured_peaks()

    def check(code, what):
        _lib.check(code, what)

    rows = []

    def report(workload, kernel, B, bytes_per_frame, ms):
        gbs = B * bytes_per_frame / (ms * 1e-3) / 1e9
        rows.append(dict(workload=workload, kernel=kernel, frames=B, bytes_per_frame=bytes_per_frame, ms=round(ms, 4),
                         gb_s=round(gbs, 1), fraction_of_hbm_peak=round(gbs / peak, 3)))
        print(f"{workload:3s} {kernel:13s} B={B:8d} {bytes_per_frame:6d} B/frame {ms:8.3f} ms {gbs:7.0f} GB/s "
              f"{gbs / peak:6.1%} of {peak:.0f} GB/s", flush=True)

    for workload, n_atoms, log2b in (("C2", 22, 22), ("C5", 1000, 16)):
        base = bd.DIPEPTIDE_NM * 10.0 if n_atoms == 22 else bd.chain_structure(n_atoms, seed=2026)
        B = 1 << log2b
        X = bd.frames(base, B, dev, 1).contiguous()
        assert X.numel() * 4 > 126 * 2 ** 20
        al = utils.Align(base, list(range(n_atoms))).to(dev)
        G = torch.randn_like(X)
        Y, GX = torch.empty_like(X), torch.empty_like(X)
        fwd = lambda: check(L.cvf_align_fwd(X.data_ptr(), B, n_atoms, al.align_idx.data_ptr(), n_atoms, al.ref_pos.data_ptr(),  # noqa: E731
                                            Y.data_ptr(), None, None, stream), "cvf_align_fwd")
        vjp = lambda: check(L.cvf_align_vjp(X.data_ptr(), B, n_atoms, al.align_idx.data_ptr(), n_atoms, al.ref_pos.data_ptr(),  # noqa: E731
                                            G.data_ptr(), GX.data_ptr(), stream), "cvf_align_vjp")
        report(workload, "align_fwd", B, 24 * n_atoms, time_ms(fwd, args.reps))
        report(workload, "align_vjp", B, 36 * n_atoms, time_ms(vjp, args.reps))
        del X, G, Y, GX

    base = bd.chain_structure(166, seed=2026)
    feats, align_idx = bd.c4_features()
    pp = utils.Preprocessing(utils.Align(base[align_idx], align_idx), utils.FeatureMap(feats))
    spec = _ops.PreprocSpec(pp, (166, 3), dev, None)
    s = spec.struct
    B = 1 << 22
    X = bd.frames(base, B, dev, 1).contiguous()
    R = torch.empty(B, s.d_r, device=dev)
    GR = torch.randn(B, s.d_r, device=dev)
    GX = torch.empty_like(X)
    fwd = lambda: check(L.cvf_features_fwd(X.data_ptr(), B, spec.struct_ptr(), R.data_ptr(), stream), "cvf_features_fwd")  # noqa: E731
    vjp = lambda: check(L.cvf_features_vjp(X.data_ptr(), B, spec.struct_ptr(), GR.data_ptr(), GX.data_ptr(), stream),  # noqa: E731
                        "cvf_features_vjp")
    report("C4", "features_fwd", B, 12 * s.n_used + 4 * s.d_r, time_ms(fwd, args.reps))
    report("C4", "features_vjp", B, 12 * s.n_used + 4 * s.d_r + 12 * 166, time_ms(vjp, args.reps))

    res = dict(device=torch.cuda.get_device_name(dev), power_limit=power_limit(), hbm_peak_gb_s=peak, hbm_peak_source=peak_src,
               c4=dict(n_atoms=166, n_used=s.n_used, n_align=s.n_align, d_r=s.d_r), reps=args.reps, results=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "results"}))


if __name__ == "__main__":
    main()
