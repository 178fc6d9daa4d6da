"""CPU check of the per-frame adjoints behind the backward of the pre-processing layers (csrc/cvf_math.cuh:
cvf_align_vjp_frame, cvf_features_vjp_frame), compiled for the host from tests/host_vjp.cpp, against the fp64 closed forms
of oracle/closed_form.py on the same fp32 inputs."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import closed_form as cf
from oracle import ref_torch
from tests._cases import rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = ref_torch.DIPEPTIDE_NM * 10.0
FEATS = [("position", [0, 4, 8]), ("bond", [4, 6]), ("bond", [8, 14]), ("angle", [4, 6, 8]), ("angle", [1, 4, 14]),
         ("dihedral", [4, 6, 8, 14]), ("dihedral", [6, 8, 14, 16]), ("position", [16])]
TYPE_ID = {"position": 0, "bond": 1, "angle": 2, "dihedral": 3}


@pytest.fixture(scope="module")
def hostlib():
    import __graft_entry__ as g
    g.build()
    return C.CDLL(os.path.join(ROOT, "oracle", "_build", "libcvf_hostvjp.so"))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _frames(n, noise_sd, seed):
    return ref_torch.synth_frames(BASE, n, seed=seed, noise_sd=noise_sd).astype(np.float32)


@pytest.mark.parametrize("noise_sd", [0.3, 0.6], ids=["thermal", "noisy"])
@pytest.mark.parametrize("align", [list(range(22)), [1, 4, 6], [1, 4, 6, 8, 10, 14, 16, 18]], ids=["all", "three", "subset"])
def test_align_adjoint_matches_closed_form(hostlib, noise_sd, align):
    B, n = 512, 22
    X = _frames(B, noise_sd, seed=11)
    ref = np.ascontiguousarray(BASE[align] - BASE[align].mean(0), dtype=np.float32)
    G = np.random.default_rng(3).standard_normal((B, n, 3)).astype(np.float32)
    aidx = np.asarray(align, dtype=np.int32)
    out = np.zeros_like(X)
    hostlib.host_align_vjp(_p(X), B, n, _p(aidx), len(align), _p(ref), _p(G), _p(out))
    y, R, c, Kinv, refc = cf.kabsch(X.astype(np.float64), align, ref.astype(np.float64))
    want = cf.align_vjp(G.astype(np.float64), y, R, Kinv, align, refc)
    assert rel_l2(out, want) < 2e-6
    # the rigid-motion invariances hold for the kernel arithmetic, not only for the oracle
    scale = np.abs(out).sum(1).max()
    assert np.abs(out.astype(np.float64).sum(1)).max() < 1e-5 * scale
    torque = np.cross(X.astype(np.float64), out.astype(np.float64)).sum(1)
    assert np.abs(torque).max() < 1e-5 * scale * np.abs(X).max()


@pytest.mark.parametrize("noise_sd", [0.3, 0.6], ids=["thermal", "noisy"])
def test_feature_adjoint_matches_closed_form(hostlib, noise_sd):
    B, n = 512, 22
    Y = _frames(B, noise_sd, seed=12)
    recs = []
    for t, atoms in FEATS:           # the kernels' records: one POSITION record per atom
        recs += [("position", [a]) for a in atoms] if t == "position" else [(t, atoms)]
    table = np.zeros((len(recs), 5), np.int32)
    for i, (t, atoms) in enumerate(recs):
        table[i, 0] = TYPE_ID[t]
        table[i, 1:1 + len(atoms)] = atoms
    d_r = cf.features_fwd(Y[:1].astype(np.float64), FEATS).shape[1]
    U = np.random.default_rng(4).standard_normal((B, d_r)).astype(np.float32)
    out = np.zeros_like(Y)
    hostlib.host_features_vjp(_p(Y), B, n, _p(table), len(recs), d_r, _p(U), _p(out))
    want = cf.features_vjp(U.astype(np.float64), Y.astype(np.float64), FEATS)
    assert rel_l2(out, want) < 2e-6
    unread = sorted(set(range(n)) - {a for _, atoms in FEATS for a in atoms})
    assert unread and not out[:, unread].any()
