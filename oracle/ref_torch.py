"""CPU oracle for the colvars-finder training step.  TEST INFRASTRUCTURE ONLY.

This module is a plain-PyTorch (CPU, autograd) *restatement* of the reference's
hot path.  It is the checker for the CUDA kernels and the CPU baseline timed by
``bench.py``; nothing under ``colvars-finder_b200/`` may import it.

What it restates (reference file:line, all relative to /root/reference):

* ``mlp`` / ``EigenNets`` / ``AutoEncoderNets``  -- colvarsfinder/nn.py:29-59 (Linear+activation
  stack, last layer linear), nn.py:242-293 (k independent scalar nets, outputs concatenated),
  nn.py:61-114 (decoder(encoder(x))).
* ``eigen_loss``            -- colvarsfinder/core.py:387-457 (EigenFunctionTask.loss_func), both the
  generator branch (lag 0, core.py:418-426,438) and the transfer-operator branch (core.py:412-416,428,440).
* ``ae_loss``               -- colvarsfinder/core.py:652-666 (AutoEncoderTask.weighted_MSE_loss).
* ``split_indices``         -- colvarsfinder/core.py:465-481 / 672-685 (sklearn train_test_split on the
  numpy global RNG, drawn twice by the eigen task and once by the AE task).

Parity pin: ``oracle/gen_golden.py`` runs the *actual* reference (imported from /root/reference with
stubs for its two missing imports) on seeded inputs and stores its outputs in ``tests/golden``;
``tests/test_oracle.py`` checks this restatement against those vectors.

PARITY UNPINNED part: the alignment / feature layer (``Align``, ``FeatureMap``).  In the reference
these come from the third-party package ``molann`` (examples/dipeptide/main.ipynb:31-32,335-348),
which is neither vendored under /root/reference nor pinned in setup.cfg:20-24 and is not installed.
The definitions below are this repository's own statement of that layer (SURVEY.md section 8c): Kabsch
alignment through ``torch.linalg.svd`` with the det-sign fix, and position / bond / angle / dihedral
features.  No reference test or golden vector exists for them.
"""
from __future__ import annotations

import itertools
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch


# --------------------------------------------------------------------------------------
# networks  (nn.py:29-59, 61-114, 242-293)
# --------------------------------------------------------------------------------------
def init_mlp_params(layer_dims: Sequence[int], dtype=torch.float32) -> List[torch.Tensor]:
    """Parameters [W1, b1, W2, b2, ...] drawn exactly like a chain of torch.nn.Linear
    constructed in order (nn.py:54-57), so torch.manual_seed reproduces the reference init."""
    out = []
    for i in range(len(layer_dims) - 1):
        lin = torch.nn.Linear(layer_dims[i], layer_dims[i + 1])
        out += [lin.weight.detach().to(dtype).clone(), lin.bias.detach().to(dtype).clone()]
    return out


def mlp(params: Sequence[torch.Tensor], x: torch.Tensor, act=torch.tanh) -> torch.Tensor:
    """Linear layers with ``act`` between them, none after the last (nn.py:54-57)."""
    n = len(params) // 2
    h = x
    for i in range(n):
        h = h @ params[2 * i].t() + params[2 * i + 1]
        if i < n - 1:
            h = act(h)
    return h


def eigen_forward(nets: Sequence[Sequence[torch.Tensor]], r: torch.Tensor, act=torch.tanh) -> torch.Tensor:
    """k scalar nets evaluated on the same features and concatenated -> [B, k] (nn.py:293)."""
    return torch.cat([mlp(p, r, act) for p in nets], dim=1)


def ae_forward(enc: Sequence[torch.Tensor], dec: Sequence[torch.Tensor], r: torch.Tensor) -> torch.Tensor:
    """decoder(encoder(r)) (nn.py:114)."""
    return mlp(dec, mlp(enc, r))


# --------------------------------------------------------------------------------------
# pre-processing layer: alignment + features   (PARITY UNPINNED, see module docstring)
# --------------------------------------------------------------------------------------
class Align(torch.nn.Module):
    """Kabsch alignment of every frame onto a centred reference structure.

    x [B,N,3] -> y [B,N,3]:  c = mean over the align atoms, H = (x_A-c)^T ref,
    U,S,Vh = svd(H), d = sign(det(U Vh)) (no gradient), R = U diag(1,1,d) Vh, y = (x-c) R,
    applied to all N atoms.  Convention of SURVEY.md section 7.3-A / 8c.
    """

    def __init__(self, ref_positions, align_indices):
        super().__init__()
        ref = torch.as_tensor(np.asarray(ref_positions), dtype=torch.float64)
        ref = ref - ref.mean(0, keepdim=True)
        self.register_buffer("ref", ref)
        self.register_buffer("idx", torch.as_tensor(np.asarray(align_indices), dtype=torch.long))

    def rotation(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        xa = x[:, self.idx, :]
        c = xa.mean(1, keepdim=True)
        H = (xa - c).transpose(1, 2) @ self.ref.to(x.dtype)
        U, S, Vh = torch.linalg.svd(H)
        d = torch.sign(torch.linalg.det(U @ Vh)).detach()
        D = torch.ones(x.shape[0], 3, dtype=x.dtype)
        D[:, 2] = d
        R = (U * D[:, None, :]) @ Vh
        return R, c

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        R, c = self.rotation(x)
        return (x - c) @ R


class FeatureMap(torch.nn.Module):
    """Feature map on (aligned) coordinates y [B,N,3] -> [B,d_r].

    ``features`` is a list of (type, atom_indices):
      'position' (any number of atoms) -> their coordinates flattened (3 per atom)
      'bond'     (i,j)       -> |y_j - y_i|
      'angle'    (i,j,k)     -> cos of the angle at j  (or the angle itself if use_angle_value)
      'dihedral' (i,j,k,l)   -> (cos phi, sin phi)     (or phi = atan2(sin,cos) if use_angle_value)
    with r12=y_j-y_i, r23=y_k-y_j, r34=y_l-y_k, n1=r12 x r23, n2=r23 x r34,
    cos phi = n1.n2/(|n1||n2|), sin phi = (n1.r34)|r23|/(|n1||n2|).
    Output is the concatenation in list order.
    """

    def __init__(self, features, use_angle_value: bool = False):
        super().__init__()
        self.features = [(t, [int(a) for a in idx]) for t, idx in features]
        self.use_angle_value = use_angle_value

    def forward(self, y: torch.Tensor) -> torch.Tensor:
        outs = []
        for t, idx in self.features:
            if t == "position":
                outs.append(y[:, idx, :].reshape(y.shape[0], -1))
            elif t == "bond":
                i, j = idx
                outs.append(torch.linalg.norm(y[:, j] - y[:, i], dim=1, keepdim=True))
            elif t == "angle":
                i, j, k = idx
                a, b = y[:, i] - y[:, j], y[:, k] - y[:, j]
                cosv = (a * b).sum(1) / (torch.linalg.norm(a, dim=1) * torch.linalg.norm(b, dim=1))
                outs.append((torch.acos(cosv) if self.use_angle_value else cosv)[:, None])
            elif t == "dihedral":
                i, j, k, l = idx
                r12, r23, r34 = y[:, j] - y[:, i], y[:, k] - y[:, j], y[:, l] - y[:, k]
                n1 = torch.linalg.cross(r12, r23, dim=1)
                n2 = torch.linalg.cross(r23, r34, dim=1)
                den = torch.linalg.norm(n1, dim=1) * torch.linalg.norm(n2, dim=1)
                cosv = (n1 * n2).sum(1) / den
                sinv = (n1 * r34).sum(1) * torch.linalg.norm(r23, dim=1) / den
                if self.use_angle_value:
                    outs.append(torch.atan2(sinv, cosv)[:, None])
                else:
                    outs.append(torch.stack([cosv, sinv], dim=1))
            else:
                raise ValueError(f"unknown feature type {t}")
        return torch.cat(outs, dim=1)


class Preprocess(torch.nn.Module):
    """pp_layer = FeatureMap o Align (either part optional); Identity when both are None."""

    def __init__(self, align: Optional[Align] = None, fmap: Optional[FeatureMap] = None):
        super().__init__()
        self.align, self.fmap = align, fmap

    def forward(self, x):
        if self.align is not None:
            x = self.align(x)
        if self.fmap is not None:
            x = self.fmap(x)
        elif x.dim() == 3:
            x = x.reshape(x.shape[0], -1)
        return x


# --------------------------------------------------------------------------------------
# losses
# --------------------------------------------------------------------------------------
def eigen_loss(X, weight, nets, pp, alpha, eig_w, diag_coeff=None, beta=1.0, sort=True,
               X_lagged=None, weight_lagged=None, lag_time=None, act=torch.tanh):
    """EigenFunctionTask.loss_func (core.py:387-457).

    Returns (loss, eig_vals[k] sorted if ``sort``, non_penalty_loss, penalty, cvec).
    Generator branch when X_lagged is None (X must require grad), transfer-operator branch
    otherwise (lag_time = traj_dt * lag_idx).  The transfer-operator objective keeps the
    reference's indexing (numerator idx, denominator cvec[idx], core.py:440).  ``act`` is the
    activation between the layers of every network (the reference's ``activation`` argument).
    """
    k = len(nets)
    y = eigen_forward(nets, pp(X), act)                                # core.py:403
    tot_w = weight.sum()                                               # core.py:406
    mean = [(y[:, i] * weight).sum() / tot_w for i in range(k)]        # core.py:409
    var = [(y[:, i] ** 2 * weight).sum() / tot_w - mean[i] ** 2 for i in range(k)]  # core.py:410
    generator = X_lagged is None
    if generator:
        tot_dim = X[0].numel()
        a = torch.ones(tot_dim, dtype=X.dtype) if diag_coeff is None else diag_coeff.to(X.dtype)
        grads = [torch.autograd.grad(y[:, i].sum(), X, retain_graph=True, create_graph=True)[0]
                 .reshape(-1, tot_dim) for i in range(k)]              # core.py:424
        dirich = [((grads[i] ** 2 * a).sum(1) * weight).sum() for i in range(k)]
        eig = torch.tensor([float(dirich[i] / (tot_w * beta) / var[i]) for i in range(k)], dtype=X.dtype)  # :426
    else:
        tot_wl = weight_lagged.sum()
        yl = eigen_forward(nets, pp(X_lagged), act)                    # core.py:414
        mean_l = [(yl[:, i] * weight_lagged).sum() / tot_wl for i in range(k)]
        var_l = [(yl[:, i] ** 2 * weight_lagged).sum() / tot_wl - mean_l[i] ** 2 for i in range(k)]
        diff = [(((yl[:, i] - y[:, i]) ** 2) * weight).sum() for i in range(k)]
        eig = torch.tensor([float(diff[i] / tot_w / (var[i] + var_l[i])) for i in range(k)],
                           dtype=X.dtype) / lag_time                  # core.py:428
    cvec = np.arange(k)
    if sort:
        cvec = np.argsort(eig.numpy())                                 # core.py:432
        eig = eig[torch.as_tensor(cvec)]
    if generator:
        obj = sum(eig_w[i] * dirich[cvec[i]] / var[cvec[i]] for i in range(k)) / (tot_w * beta)  # :438
    else:
        obj = sum(eig_w[i] * diff[i] / (var[cvec[i]] + var_l[cvec[i]]) for i in range(k)) / tot_w / lag_time  # :440
    pen = sum((var[i] - 1.0) ** 2 for i in range(k))                   # core.py:446
    for i, j in itertools.combinations(range(k), 2):                   # core.py:449-452
        pen = pen + ((y[:, i] * y[:, j] * weight).sum() / tot_w - mean[i] * mean[j]) ** 2
    loss = obj + alpha * pen                                           # core.py:455
    return loss, eig, obj, pen, cvec


def ae_loss(X, weight, enc, dec):
    """AutoEncoderTask.weighted_MSE_loss (core.py:652-666) on pre-processed features X [B,d_r]."""
    out = ae_forward(enc, dec, X)
    return (weight * ((out - X) ** 2).sum(1)).sum() / weight.sum()


# --------------------------------------------------------------------------------------
# split + batching  (core.py:465-481, 672-685)
# --------------------------------------------------------------------------------------
def split_indices(n: int, test_ratio: float, draws: int = 1):
    """Train/test index arrays exactly as the reference draws them: sklearn train_test_split on
    the numpy *global* RNG; EigenFunctionTask.train calls it twice and keeps the second result
    (core.py:465,468), AutoEncoderTask.train once (core.py:672)."""
    from sklearn.model_selection import train_test_split
    for _ in range(draws):
        tr, te = train_test_split(np.arange(n), test_size=test_ratio)
    return tr, te


def batches(n_split: int, batch_size: int):
    """DataLoader(shuffle=False, drop_last=True) with bs=min(batch_size, n_split) (core.py:470-481)."""
    bs = min(batch_size, n_split)
    return [(s, s + bs) for s in range(0, n_split - bs + 1, bs)], bs


# --------------------------------------------------------------------------------------
# synthetic data of SURVEY.md section 8d
# --------------------------------------------------------------------------------------
DIPEPTIDE_NM = np.array([  # examples/dipeptide/top.gro:3-24 (nm); used x10 -> Angstrom
    [0.200, 0.100, -0.000], [0.200, 0.209, 0.000], [0.149, 0.245, 0.089], [0.149, 0.245, -0.089],
    [0.343, 0.264, -0.000], [0.439, 0.188, -0.000], [0.356, 0.397, -0.000], [0.273, 0.456, -0.000],
    [0.485, 0.461, -0.000], [0.541, 0.432, 0.089], [0.566, 0.422, -0.123], [0.512, 0.452, -0.213],
    [0.663, 0.472, -0.121], [0.581, 0.314, -0.124], [0.471, 0.613, 0.000], [0.360, 0.665, 0.000],
    [0.585, 0.683, 0.000], [0.674, 0.636, -0.000], [0.585, 0.828, 0.000], [0.482, 0.865, 0.000],
    [0.636, 0.865, 0.089], [0.636, 0.865, -0.089]])


def chain_structure(n_atoms: int, seed: int = 2026, bond: float = 1.5) -> np.ndarray:
    """Random-walk chain with fixed bond length (config C4's 166-atom base structure)."""
    rng = np.random.default_rng(seed)
    steps = rng.normal(size=(n_atoms, 3))
    steps *= bond / np.linalg.norm(steps, axis=1, keepdims=True)
    pos = np.cumsum(steps, axis=0)
    return pos - pos.mean(0)


def synth_frames(base: np.ndarray, n: int, seed: int = 2026, trans_sd=5.0, noise_sd=0.3):
    """frame = base Q + t + eps with Q a Haar rotation (QR of a Gaussian, det fixed to +1)."""
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n, 3, 3))
    Q, Rr = np.linalg.qr(A)
    Q = Q * np.sign(np.diagonal(Rr, axis1=1, axis2=2))[:, None, :]
    Q[:, :, 2] *= np.sign(np.linalg.det(Q))[:, None]
    t = rng.normal(scale=trans_sd, size=(n, 1, 3))
    eps = rng.normal(scale=noise_sd, size=(n,) + base.shape)
    return (np.einsum("ni,bij->bnj", base, Q) + t + eps).astype(np.float32)


def boltzmann_weights(n: int, seed: int = 2026, dbeta: float = 0.5) -> np.ndarray:
    """w = exp(-dbeta (E - mean E)) normalised to mean 1 (formula of utils.py:411-412,145)."""
    rng = np.random.default_rng(seed + 1)
    E = rng.normal(size=n)
    w = np.exp(-dbeta * (E - E.mean()))
    return (w / w.mean()).astype(np.float32)
