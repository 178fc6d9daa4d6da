"""Helpers shared by the tests: load the golden vectors written by oracle/gen_golden.py."""
import os

import numpy as np
import torch

from oracle import ref_torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

EIGEN_GENERATOR_CASES = ["eigen_2d_k1", "eigen_2d_k3_diag", "eigen_2d_k2_nosort", "eigen_dipep_k3",
                         "eigen_dipep_subset_diag", "eigen_dipep_features", "eigen_dipep_invariant"]
AE_CASES = ["ae_2d", "ae_dipep"]
REGAE_CASES = ["regae_2d_generator", "regae_2d_lagged", "regae_2d_lagged_k2_frozen", "regae_dipep_generator"]


def load(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))


def eigen_case(name):
    d = load(name)
    k = int(d["k"])
    nl = len(d["layer_dims"]) - 1
    c = dict(X=d["X"], w=d["w"], k=k, layer_dims=[int(v) for v in d["layer_dims"]], alpha=float(d["alpha"]),
             eig_w=[float(v) for v in d["eig_w"]], beta=float(d["beta"]), lag_tau=float(d["lag_tau"]),
             dt=float(d["dt"]), sort=bool(d["sort"]), diag_coeff=d.get("diag_coeff"),
             pp_kind=str(d["pp_kind"]), ref=d.get("ref"), align_idx=d.get("align_idx"), features=None)
    if "feat_types" in d:
        c["features"] = [(str(t), [int(a) for a in row if a >= 0]) for t, row in zip(d["feat_types"], d["feat_atoms"])]
    c["params"] = [[d[f"p_{i}_{j}"] for j in range(2 * nl)] for i in range(k)]
    for tag in ("g32", "g64"):
        c[tag] = [[d[f"{tag}_{i}_{j}"] for j in range(2 * nl)] for i in range(k)]
    for tag in ("r32", "g64"):
        for f in ("loss", "eig", "obj", "pen", "cvec"):
            c[f"{tag}_{f}"] = d[f"{tag}_{f}"]
    return c


def ae_case(name):
    d = load(name)
    ne, nd = len(d["e_dims"]) - 1, len(d["d_dims"]) - 1
    return dict(F=d["F"], w=d["w"], e_dims=[int(v) for v in d["e_dims"]], d_dims=[int(v) for v in d["d_dims"]],
                enc=[d[f"enc_{j}"] for j in range(2 * ne)], dec=[d[f"dec_{j}"] for j in range(2 * nd)],
                g32_enc=[d[f"g32_enc_{j}"] for j in range(2 * ne)], g64_enc=[d[f"g64_enc_{j}"] for j in range(2 * ne)],
                g32_dec=[d[f"g32_dec_{j}"] for j in range(2 * nd)], g64_dec=[d[f"g64_dec_{j}"] for j in range(2 * nd)],
                r32_loss=float(d["r32_loss"]), g64_loss=float(d["g64_loss"]))


def regae_case(name):
    """Golden vectors of RegAutoEncoderTask written by oracle/gen_golden_regae.py."""
    d = load(name)
    K = int(d["K"])
    ne, nd, nr = len(d["e_dims"]) - 1, len(d["d_dims"]) - 1, len(d["r_dims"]) - 1
    c = dict(X=d["X"], w=d["w"], K=K, e_dims=[int(v) for v in d["e_dims"]], d_dims=[int(v) for v in d["d_dims"]],
             r_dims=[int(v) for v in d["r_dims"]], eig_w=[float(v) for v in d["eig_w"]], alpha=float(d["alpha"]),
             gamma=[float(v) for v in d["gamma"]], eta=[float(v) for v in d["eta"]], lag_tau_ae=float(d["lag_tau_ae"]),
             lag_tau_reg=float(d["lag_tau_reg"]), beta=float(d["beta"]), dt=float(d["dt"]), freeze=bool(d["freeze"]),
             pp_kind=str(d["pp_kind"]), ref=d.get("ref"), align_idx=d.get("align_idx"))
    c["enc"] = [d[f"enc_{j}"] for j in range(2 * ne)]
    c["dec"] = [d[f"dec_{j}"] for j in range(2 * nd)]
    c["reg"] = [[d[f"reg_{i}_{j}"] for j in range(2 * nr)] for i in range(K)]
    for tag in ("g32", "g64"):
        c[f"{tag}_enc"] = [d[f"{tag}_enc_{j}"] for j in range(2 * ne)]
        c[f"{tag}_dec"] = [d[f"{tag}_dec_{j}"] for j in range(2 * nd)]
        c[f"{tag}_reg"] = [[d[f"{tag}_reg_{i}_{j}"] for j in range(2 * nr)] for i in range(K)]
    for tag in ("r32", "g64"):
        for f in ("loss", "ae", "g0", "g1", "e0", "e1", "e2", "eig", "cvec"):
            c[f"{tag}_{f}"] = d[f"{tag}_{f}"]
    return c


def rel_l2(a, b):
    a, b = np.asarray(a, dtype=np.float64).ravel(), np.asarray(b, dtype=np.float64).ravel()
    n = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / n) if n > 0 else float(np.linalg.norm(a - b))


def repeated_batch(D, B, seed, offset=0, device=None):
    """(X, w, w_agg, idx): X = D[idx] on the device with idx uniform over the M frames of D, random fp32 weights w, and the
    fp64 weight each distinct frame carries in total (host).  offset=1 returns a contiguous view that starts one frame into
    its allocation (not 16-byte aligned for 12 N-byte frames with N = 2 mod 4)."""
    device = torch.device("cuda", 0) if device is None else device
    D = torch.as_tensor(D, device=device)
    g = torch.Generator(device=device).manual_seed(seed)
    idx = torch.randint(0, D.shape[0], (B,), generator=g, device=device)
    w = torch.exp(0.5 * torch.randn(B, generator=g, device=device)).contiguous()
    buf = torch.empty((B + offset,) + tuple(D.shape[1:]), dtype=D.dtype, device=device)
    X = buf[offset:]
    torch.index_select(D, 0, idx, out=X)
    assert X.is_contiguous() and X.data_ptr() == buf.data_ptr() + offset * X[0].numel() * X.element_size()
    w_agg = torch.zeros(D.shape[0], dtype=torch.float64, device=device).index_add_(0, idx, w.double())
    return X, w, w_agg.cpu().numpy(), idx


def tol(gold, ref32, rel=1e-5, slack=1.0):
    """SURVEY 7.3-D: pass when |ours-gold| <= max(rel*|gold|, slack*|ref32-gold|)."""
    return max(rel * abs(float(gold)), slack * abs(float(ref32) - float(gold)))


class GatheredFeatures(torch.nn.Module):
    """Pre-processing of the gathered transfer-operator oracle: maps frame numbers (carried as float64, the dtype the
    reference formula computes in) to precomputed fp64 features of the distinct frames."""

    def __init__(self, R):
        super().__init__()
        self.R = torch.as_tensor(R, dtype=torch.float64)

    def forward(self, i):
        return self.R[i.long()]


def lag_oracle(R, idx, w, nets, alpha, eig_w, lag, lag_time):
    """fp64 transfer-operator loss of the batch X = D[idx] (frame t paired with t + lag) from the features R of the distinct
    frames: reference formula (oracle/ref_torch.eigen_loss) on the gathered features.  Returns (comb-like dict, grads)."""
    I = torch.as_tensor(np.asarray(idx), dtype=torch.float64)
    wt = torch.as_tensor(np.asarray(w), dtype=torch.float64)
    tn = [[torch.tensor(p, dtype=torch.float64, requires_grad=True) for p in n] for n in nets]
    ref = ref_torch.eigen_loss(I[:-lag], wt[:-lag], tn, GatheredFeatures(R), alpha, eig_w, X_lagged=I[lag:],
                               weight_lagged=wt[lag:], lag_time=lag_time)
    ref[0].backward()
    grads = [[np.zeros(tuple(t.shape)) if t.grad is None else t.grad.numpy() for t in n] for n in tn]
    return dict(loss=float(ref[0]), eig=ref[1].numpy().astype(np.float64), cvec=[int(v) for v in ref[4]]), grads
