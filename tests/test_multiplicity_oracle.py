"""The multiplicity oracle of tests/test_step_at_scale_gpu.py on the host: a batch X = D[idx] of B frames drawn from M distinct
frames has the fp64 loss and gradients of the closed form evaluated on D with the aggregated weights
w_agg[i] = sum_{f: idx_f = i} w_f, and the gathered transfer-operator oracle equals the reference formula on the explicit
lagged batch."""
import numpy as np
import torch

from oracle import closed_form as cf
from oracle import ref_torch
from tests import _cases as C

BASE = ref_torch.DIPEPTIDE_NM * 10.0


def _batch(M, B, seed):
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, M, B)
    w = np.exp(0.5 * rng.normal(size=B)).astype(np.float32).astype(np.float64)
    return idx, w, np.bincount(idx, weights=w, minlength=M)


def _assert_grads_equal(a, b):
    """Equal up to fp64 regrouping: the two sides add the same terms in another order, and gradient sums cancel (the bias
    sums most, to ~1e-4 of their terms), so entries move by ~1e-12 of the largest gradient and a small tensor by up to ~2e-11
    of its own norm."""
    flat_b = [t for n in b for t in n] if isinstance(b[0], list) else list(b)
    flat_a = [t for n in a for t in n] if isinstance(a[0], list) else list(a)
    scale = max(np.abs(t).max() for t in flat_b)
    for ta, tb in zip(flat_a, flat_b):
        assert np.abs(ta - tb).max() <= 1e-11 * scale
        if np.abs(tb).max() >= 1e-9 * scale:       # not the last-layer bias of the generator loss (zero up to rounding)
            assert C.rel_l2(ta, tb) <= 1e-10, C.rel_l2(ta, tb)


def test_eigen_closed_form_of_repeated_frames_equals_aggregated_weights():
    M, B, k = 200, 5000, 3
    D = ref_torch.synth_frames(BASE, M, seed=5).astype(np.float64)
    idx, w, w_agg = _batch(M, B, 6)
    torch.manual_seed(7)
    nets = [[p.numpy() for p in ref_torch.init_mlp_params([66, 20, 20, 20, 1])] for _ in range(k)]
    ppo = cf.Preproc(align_idx=list(range(22)), ref=BASE)
    full, g_full, _ = cf.eigen_loss_and_grads(D[idx], w, nets, ppo, 20.0, [1.0, 0.6, 0.3])
    agg, g_agg, _ = cf.eigen_loss_and_grads(D, w_agg, nets, ppo, 20.0, [1.0, 0.6, 0.3])
    assert list(full["cvec"]) == list(agg["cvec"])
    assert abs(full["loss"] - agg["loss"]) <= 1e-12 * abs(full["loss"])
    np.testing.assert_allclose(agg["eig"], full["eig"], rtol=1e-12, atol=0)
    _assert_grads_equal(g_agg, g_full)


def test_autoencoder_closed_form_of_repeated_frames_equals_aggregated_weights():
    M, B = 200, 5000
    rng = np.random.default_rng(8)
    F = rng.normal(size=(M, 66))
    idx, w, w_agg = _batch(M, B, 9)
    torch.manual_seed(10)
    enc = [p.numpy() for p in ref_torch.init_mlp_params([66, 20, 20, 20, 2])]
    dec = [p.numpy() for p in ref_torch.init_mlp_params([2, 10, 10, 66])]
    lo, ge, gd = cf.ae_loss_and_grads(F[idx], w, enc, dec)
    lo_a, ge_a, gd_a = cf.ae_loss_and_grads(F, w_agg, enc, dec)
    assert abs(lo - lo_a) <= 1e-12 * abs(lo)
    _assert_grads_equal(ge_a + gd_a, ge + gd)


def test_gathered_lag_oracle_equals_reference_on_explicit_batch():
    """The transfer-operator loss pairs frame t with t + lag, so weights do not aggregate: the oracle gathers precomputed
    features of the distinct frames instead.  It must equal the reference formula on the explicit lagged batch."""
    M, B, k, lag, tau = 200, 5000, 3, 3, 1.5
    D = ref_torch.synth_frames(BASE, M, seed=11).astype(np.float64)
    idx, w, _ = _batch(M, B + lag, 12)
    torch.manual_seed(13)
    nets = [[p.numpy() for p in ref_torch.init_mlp_params([66, 20, 20, 20, 1])] for _ in range(k)]
    pp = ref_torch.Preprocess(ref_torch.Align(BASE, list(range(22))), None)
    with torch.no_grad():
        R = pp(torch.as_tensor(D)).numpy()
    gold, g_gold = C.lag_oracle(R, idx, w, nets, 20.0, [1.0, 0.6, 0.3], lag, tau)
    X, wt = torch.as_tensor(D[idx]), torch.as_tensor(w)
    tn = [[torch.tensor(p, dtype=torch.float64, requires_grad=True) for p in n] for n in nets]
    ref = ref_torch.eigen_loss(X[:-lag], wt[:-lag], tn, pp, 20.0, [1.0, 0.6, 0.3], X_lagged=X[lag:], weight_lagged=wt[lag:],
                               lag_time=tau)
    ref[0].backward()
    assert [int(v) for v in ref[4]] == gold["cvec"]
    assert abs(float(ref[0]) - gold["loss"]) <= 1e-12 * abs(gold["loss"])
    np.testing.assert_allclose(gold["eig"], ref[1].numpy(), rtol=1e-12, atol=0)
    _assert_grads_equal(g_gold, [[t.grad.numpy() for t in n] for n in tn])
