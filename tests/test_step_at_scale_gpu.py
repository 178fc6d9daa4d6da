"""The training step at the batch sizes bench.py times, and every fast-path kernel variant in both of its schedules, against an
exact fp64 oracle.

The fast eigenfunction kernels (csrc/cvf_eigen_fast.cu) split their work by batch size.  Pass 1 gives each CTA one (512-frame
tile, network) pair when ceil(B/512) k <= #SMs and otherwise lets each CTA walk whole tiles with all their networks; pass 2 gives
each warp one (32-frame tile, network) pair when ceil(B/512) 16 k <= 2 #SMs nw (nw = 4..8 pass-2 warps) and otherwise lets each
warp walk whole tiles, looping over all networks, prefetching the next network and tile, keeping fp32 totals in tensor memory
across many tiles and sending the networks beyond tensor-memory capacity to fp64 atomics.  Small batches run the first
("split") schedule, the batches users train on the second ("whole").  Every case here states which one it runs and checks it.

The oracle is exact at any batch size for the cost of M frames: a batch is X = D[idx] with M distinct frames D and a random
index map idx, so the fp64 closed form on D with the aggregated weights w_agg[i] = sum_{f: idx_f = i} w_f is the fp64 loss
and gradient of the whole batch (every quantity is a weighted sum over frames; tests/test_multiplicity_oracle.py checks this
on the host).  The index map is random, so every 32-frame tile holds its own frames: a kernel that reads the wrong tile,
network or column does not get the right answer by accident.
"""
import gc

import numpy as np
import pytest
import torch

import bench_data as bd
from oracle import closed_form as cf
from oracle import ref_torch
from oracle.ref_import import FakeTrajectory
from tests import _cases as C

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None
BASE = bd.DIPEPTIDE_NM * 10.0
M = 2048                          # distinct frames behind every eigenfunction batch
B_SMALL = 3001                    # split schedule in both passes on a 148-SM part (6 tiles of 512)
B_LARGE = (1 << 17) + 77          # whole-tile schedule in both passes, with a ragged last tile (257 tiles of 512)
B_BENCH = 1 << 22                 # what bench.py times for C1-C4 and the pre-pass
EIG_W = [1.0, 0.6, 0.3, 0.2, 0.15, 0.1, 0.05, 0.03]


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(autouse=True)
def release_memory():
    yield
    gc.collect()
    torch.cuda.empty_cache()


# --------------------------------------------------------------------------------------------- helpers
def repeated_batch(D, B, seed, offset=0):
    """(X, w, w_agg, idx): X = D[idx] on the device with idx uniform over the M frames of D, random fp32 weights w, and the
    fp64 weight each distinct frame carries in total (host).  offset=1 returns a contiguous view that starts one frame into
    its allocation (not 16-byte aligned for 12 N-byte frames with N = 2 mod 4)."""
    D = torch.as_tensor(D, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(seed)
    idx = torch.randint(0, D.shape[0], (B,), generator=g, device=DEV)
    w = torch.exp(0.5 * torch.randn(B, generator=g, device=DEV)).contiguous()
    buf = torch.empty((B + offset,) + tuple(D.shape[1:]), dtype=D.dtype, device=DEV)
    X = buf[offset:]
    torch.index_select(D, 0, idx, out=X)
    assert X.is_contiguous() and X.data_ptr() == buf.data_ptr() + offset * X[0].numel() * X.element_size()
    w_agg = torch.zeros(D.shape[0], dtype=torch.float64, device=DEV).index_add_(0, idx, w.double())
    return X, w, w_agg.cpu().numpy(), idx


def schedule(B, k):
    """"split" if both passes give out (tile, network) pairs for every pass-2 warp count, "whole" if both walk whole tiles for
    every warp count, "mixed" otherwise (a case must not sit there: which schedule it runs would depend on the shape)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = -(-B // 512)
    p1 = tiles * k <= sms
    p2 = [tiles * 16 * k <= 2 * sms * nw for nw in range(4, 9)]
    if p1 and all(p2):
        return "split"
    if not p1 and not any(p2):
        return "whole"
    return "mixed"


def random_nets(dims, k, seed):
    torch.manual_seed(seed)
    return [[p.numpy() for p in ref_torch.init_mlp_params(dims)] for _ in range(k)]


def load_params(modules, params):
    with torch.no_grad():
        for m, ps in zip(modules, params):
            for p, v in zip(m.parameters(), ps):
                p.copy_(torch.as_tensor(v))


def eigen_task(tmp_path, pp, dims, k, nets, D_host, alpha=20.0, diag=None, lag_tau=0.0, dt=1.0):
    """EigenFunctionTask built as bench.py builds it: a few frames for the constructor, then the step on device tensors."""
    from colvarsfinder import core, nn
    model = nn.EigenFunctions(dims, k)
    load_params(model.eigen_funcs, nets)
    small = np.ascontiguousarray(D_host[:64])
    task = core.EigenFunctionTask(FakeTrajectory(small, np.ones(len(small)), dt=dt), pp, model, str(tmp_path), alpha, EIG_W[:k],
                                  diag_coeff=None if diag is None else torch.as_tensor(diag), lag_tau=lag_tau, k=k, device=DEV,
                                  verbose=False, debug_mode=False)
    return task, model


def eigen_step(task, model, X, w, Xl=None, wl=None):
    model.zero_grad(set_to_none=True)
    out = task.loss_func(X, w, Xl, wl)
    out[0].backward()
    return out, [[p.grad.detach().clone() for p in f.parameters()] for f in model.eigen_funcs]


def assert_eigen_envelope(out, grads, comb, g64, tag):
    """cvec exact; loss <= 1e-6 and eigenvalues <= 2e-6 relative; every gradient tensor <= 5e-5 relative L2; gradients that
    are zero in fp64 (last-layer biases, below 1e-9 of the largest entry) below 1e-5 of that scale.  Prints what was achieved."""
    loss, eig, _, _, cvec = out
    assert list(cvec.cpu().numpy()) == list(comb["cvec"]), (tag, cvec, comb["cvec"])
    e_loss = abs(float(loss) - comb["loss"]) / abs(comb["loss"])
    e = eig.cpu().numpy().astype(np.float64)
    e_eig = float(np.max(np.abs(e - comb["eig"]) / np.abs(comb["eig"])))
    scale = max(np.abs(t).max() for n in g64 for t in n)
    errs, zeros = [], []
    for i in range(len(g64)):
        for j in range(len(g64[i])):
            got = grads[i][j].cpu().numpy()
            if np.abs(g64[i][j]).max() < 1e-9 * scale:
                zeros.append(float(np.abs(got).max() / scale))
            else:
                errs.append(C.rel_l2(got, g64[i][j]))
    print(f"[{tag}] loss {e_loss:.1e}  eig {e_eig:.1e}  grad rel-L2 max {max(errs):.1e} median {np.median(errs):.1e}  "
          f"zero-grad {max(zeros) if zeros else 0.0:.1e}")
    assert e_loss <= 1e-6, (tag, "loss", e_loss)
    assert e_eig <= 2e-6, (tag, "eig", e_eig)
    assert max(errs) <= 5e-5, (tag, "grad", errs)
    assert not zeros or max(zeros) < 1e-5, (tag, "zero-grad", zeros)


def assert_bit_identical(a, b, tag):
    (out_a, g_a), (out_b, g_b) = a, b
    assert torch.equal(out_a[0], out_b[0]) and torch.equal(out_a[1], out_b[1]), (tag, "loss / eigenvalues differ between runs")
    for ga, gb in zip(g_a, g_b):
        for ta, tb in zip(ga, gb):
            assert torch.equal(ta, tb), (tag, "gradients differ between runs")


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


# --------------------------------------------------------------------------------------------- pre-processing of the cases
def _chain(n):
    return bd.chain_structure(n, seed=100 + n)


def _chain24_records():
    feats = [("bond", [i, i + 3]) for i in range(0, 20, 2)]
    feats += [("angle", [i, i + 1, i + 2]) for i in range(0, 22, 3)]
    feats += [("dihedral", [i, i + 1, i + 2, i + 3]) for i in range(0, 21, 4)]
    return feats


DIPEP_RECORDS = [("position", [4]), ("bond", [4, 6]), ("dihedral", [4, 6, 8, 14]), ("position", [8]), ("angle", [6, 8, 14]),
                 ("bond", [1, 18])]


def preprocessing(kind, seed):
    """(drop-in pp layer, oracle Preproc, distinct frames D (fp32 host), diag length) of a case's pre-processing."""
    from colvarsfinder import utils
    if kind[0] == "identity":
        D = np.random.default_rng(seed).normal(size=(M, kind[1])).astype(np.float32)
        return torch.nn.Identity(), cf.Preproc(identity=True), D, kind[1]
    if kind[0] == "align":                 # ("align", base, alignment atoms or None for all): aligned positions
        base, sel = kind[1], kind[2] if kind[2] is not None else list(range(len(kind[1])))
        D = ref_torch.synth_frames(base, M, seed=seed)
        return utils.Align(base[sel], sel), cf.Preproc(align_idx=sel, ref=base[sel]), D, 3 * len(base)
    base, feats, sel = kind[1], kind[2], kind[3]    # ("features", base, records, alignment atoms or None)
    D = ref_torch.synth_frames(base, M, seed=seed)
    fmap = utils.FeatureMap(feats)
    if sel is None:
        return fmap, cf.Preproc(feats=feats), D, 3 * len(base)
    return (utils.Preprocessing(utils.Align(base[sel], sel), fmap), cf.Preproc(align_idx=sel, ref=base[sel], feats=feats), D,
            3 * len(base))


# --------------------------------------------------------------------------------------------- 1. benchmark workloads
def _bench_eigen(tmp_path, name, pp_kind, dims, k, seed):
    pp, ppo, _, _ = preprocessing(pp_kind, seed)
    if name == "C1":
        D = bd.ring_2d(M, DEV, seed)
    else:
        D = bd.frames(pp_kind[1], M, DEV, seed)
    D_host = D.cpu().numpy()
    nets = random_nets(dims, k, seed)
    task, model = eigen_task(tmp_path, pp, dims, k, nets, D_host)
    assert task._ctx.fast_path and schedule(B_BENCH, k) == "whole"
    X, w, w_agg, _ = repeated_batch(D, B_BENCH, seed)
    first = eigen_step(task, model, X, w)
    second = eigen_step(task, model, X, w)
    del X, w
    comb, g64, _ = cf.eigen_loss_and_grads(D_host, w_agg, nets, ppo, 20.0, EIG_W[:k])
    assert_eigen_envelope(first[0], first[1], comb, g64, f"{name} at 2^22")
    assert_bit_identical(first, second, name)
    return task


def test_bench_c1_step_at_bench_size(tmp_path):
    """C1: [2,20,20,20,1], k = 1, Identity, 2^22 frames (about 110 whole tiles per pass-2 warp)."""
    _bench_eigen(tmp_path, "C1", ("identity", 2), [2, 20, 20, 20, 1], 1, seed=11)


def test_bench_c3_step_at_bench_size(tmp_path):
    """C3: [66,20,20,20,1], k = 3, Kabsch on all 22 atoms of the dipeptide, 2^22 frames."""
    _bench_eigen(tmp_path, "C3", ("align", BASE, None), [66, 20, 20, 20, 1], 3, seed=13)


def test_bench_c4_step_at_bench_size(tmp_path):
    """C4: [81,20,20,20,1], k = 3, 45 distances + 18 dihedrals of the 166-atom chain after Kabsch on 40 atoms (the step elides
    the alignment, the oracle goes through it and its Jacobian), 2^22 frames (8 GB of input)."""
    feats, sel = bd.c4_features()
    task = _bench_eigen(tmp_path, "C4", ("features", bd.chain_structure(166, seed=2026), feats, sel), [81, 20, 20, 20, 1], 3,
                        seed=14)
    assert task._ctx.spec.alignment_elided


def _ae_step(tmp_path, e_dims, d_dims, pp, F_small, seed):
    from colvarsfinder import core, nn
    torch.manual_seed(seed)
    enc = [p.numpy() for p in ref_torch.init_mlp_params(e_dims)]
    dec = [p.numpy() for p in ref_torch.init_mlp_params(d_dims)]
    model = nn.AutoEncoder(e_dims, d_dims)
    load_params([model.encoder, model.decoder], [enc, dec])
    task = core.AutoEncoderTask(FakeTrajectory(F_small, np.ones(len(F_small))), pp, model, str(tmp_path), device=DEV,
                                verbose=False, debug_mode=False)
    return task, model, enc, dec


def _assert_ae(loss, model, F_host, w_agg, enc, dec, tag):
    lo, genc, gdec = cf.ae_loss_and_grads(F_host, w_agg, enc, dec)
    got = [p.grad.cpu().numpy() for p in model.encoder.parameters()] + [p.grad.cpu().numpy() for p in model.decoder.parameters()]
    errs = [C.rel_l2(g, go) for g, go in zip(got, genc + gdec)]
    e_loss = abs(float(loss) - lo) / abs(lo)
    print(f"[{tag}] loss {e_loss:.1e}  grad rel-L2 max {max(errs):.1e} median {np.median(errs):.1e}")
    assert e_loss <= 1e-5, (tag, e_loss)
    assert max(errs) <= 2e-5, (tag, errs)


def test_bench_c2_autoencoder_step_at_bench_size(tmp_path):
    """C2: AutoEncoder([66,20,20,20,2],[2,10,10,66]) on aligned dipeptide coordinates, 2^22 frames, on the thread-private
    kernels (cvf_ae_fast.cu).  The features are the task's own pre-pass of the distinct frames, gathered."""
    from colvarsfinder import _lib, utils
    D = bd.frames(BASE, M, DEV, 21)
    D_host = D.cpu().numpy()
    task, model, enc, dec = _ae_step(tmp_path, [66, 20, 20, 20, 2], [2, 10, 10, 66], utils.Align(BASE, list(range(22))),
                                     D_host[:64], seed=21)
    F = task.preprocessing_layer(D).reshape(M, 66).contiguous()
    X, w, w_agg, _ = repeated_batch(F, B_BENCH, 22)
    _lib.profile_read(reset=True)
    loss = task.weighted_MSE_loss(X, w)
    launched = _lib.profile_read(reset=True)
    assert launched["ae_fast_main"][2] > 0 and launched["ae_step"][2] == 0
    loss.backward()
    del X, w
    _assert_ae(loss, model, F.cpu().numpy(), w_agg, enc, dec, "C2 autoencoder at 2^22")


def test_bench_c5_autoencoder_step_at_bench_size(tmp_path):
    """C5: AutoEncoder([3000,512,512,2],[2,512,512,3000]) on standardised features, 2^16 frames = two 32 768-frame chunks of
    the layer-wise tensor-core path (3 x TF32 split, fp32 accumulation in tensor memory)."""
    g = torch.Generator(device=DEV).manual_seed(31)
    F = torch.randn(1024, 3000, generator=g, device=DEV)
    task, model, enc, dec = _ae_step(tmp_path, [3000, 512, 512, 2], [2, 512, 512, 3000], torch.nn.Identity(),
                                     F[:64].cpu().numpy(), seed=31)
    X, w, w_agg, _ = repeated_batch(F, 1 << 16, 32)
    loss = task.weighted_MSE_loss(X, w)
    loss.backward()
    del X, w
    _assert_ae(loss, model, F.cpu().numpy(), w_agg, enc, dec, "C5 autoencoder at 2^16")


def test_bench_c2_prepass_at_bench_size():
    """C2 pre-pass: Kabsch alignment of 2^22 dipeptide frames onto the reference (all 22 atoms); every aligned coordinate
    within 1e-6 Angstrom of the fp64 alignment of its distinct frame."""
    from colvarsfinder import utils
    D = bd.frames(BASE, 4096, DEV, 41)
    yo = torch.as_tensor(cf.kabsch(D.cpu().numpy().astype(np.float64), list(range(22)), BASE)[0], device=DEV)
    X, _, _, idx = repeated_batch(D, B_BENCH, 42)
    align = utils.Align(BASE, list(range(22))).to(DEV)
    out = torch.empty_like(X)
    y = align(X, out=out)
    err = 0.0
    for s in range(0, B_BENCH, 1 << 20):
        err = max(err, float((y[s:s + (1 << 20)].double() - yo[idx[s:s + (1 << 20)]]).abs().max()))
    print(f"[C2 pre-pass at 2^22] max |y - y64| {err:.1e} A")
    assert err <= 1e-6


# --------------------------------------------------------------------------------------------- 2. fast-path variants
# name: (layer dims, k, pre-processing, diag_coeff, which branch the case exists for).  The branch notes follow the host
# planning arithmetic (pass2_warps, tm_per_net in pass2_kernel) on a 227 KB-shared-memory part.
VARIANTS = {
    "v01_dr1_k1": ([1, 20, 20, 20, 1], 1, ("identity", 1), False, "d_r = 1, in-row dW1"),
    "v02_nh2_k8": ([12, 20, 20, 1], 8, ("identity", 12), False, "two hidden layers; all 8 networks in TMEM; 8-network fold"),
    "v03_c1shape_k8": ([2, 20, 20, 20, 1], 8, ("identity", 2), False, "5 networks in TMEM + 3 on atomics, 6 pass-2 warps"),
    "v04_h32_k3_diag": ([5, 32, 32, 32, 1], 3, ("identity", 5), True, "H = 32, 2 in TMEM + 1 on atomics, 4 warps"),
    "v05_h16_k8": ([24, 16, 16, 16, 1], 8, ("identity", 24), False, "H = 16, one exact 24-column dW1 chunk, 8 in TMEM"),
    "v06_dr25_k3": ([25, 20, 20, 20, 1], 3, ("identity", 25), False, "second dW1 chunk one column wide"),
    "v07_chain3_k3": ([9, 20, 20, 20, 1], 3, ("align", _chain(3), None), False, "aligned positions with in-row dW1 (width 12)"),
    "v08_chain4_k4": ([12, 20, 20, 20, 1], 4, ("align", _chain(4), None), False,
                      "aligned positions, exact width 12, 4 networks in TMEM, 7 warps"),
    "v09_chain5_subset_k2": ([15, 16, 16, 16, 1], 2, ("align", _chain(5), [0, 2, 4]), False,
                             "alignment on 3 of 5 atoms, one partial dW1 chunk"),
    "v10_chain16_k8": ([48, 20, 20, 20, 1], 8, ("align", _chain(16), None), False, "two exact dW1 chunks; 4 in TMEM + 4 on atomics"),
    "v11_dipep_k4": ([66, 20, 20, 20, 1], 4, ("align", BASE, None), False, "C3 shape with 3 in TMEM + 1 on atomics"),
    "v12_chain24_k3": ([72, 20, 20, 20, 1], 3, ("align", _chain(24), None), False, "three exact 24-column dW1 chunks"),
    "v13_chain28_k1": ([84, 20, 20, 20, 1], 1, ("align", _chain(28), None), False, "28-column dW1 chunks on aligned positions"),
    "v14_dipep_h32_k1": ([66, 32, 32, 32, 1], 1, ("align", BASE, None), False, "H = 32 at d_r = 66, 5 warps"),
    "v15_dipep_records_diag_k3": ([11, 20, 20, 20, 1], 3, ("features", BASE, DIPEP_RECORDS, None), True,
                                  "feature records with positions and diag_coeff"),
    "v16_chain24_features_k2": ([30, 20, 20, 20, 1], 2, ("features", _chain(24), _chain24_records(), None), False,
                                "strided (non-bulk) feature prep: 3N = 72"),
    "v17_c4_h16_k4": ([81, 16, 16, 16, 1], 4, ("features", bd.chain_structure(166, seed=2026)) + tuple(bd.c4_features()), False,
                      "H = 16 with 28-column dW1 chunks, 4 networks in TMEM"),
}
ON_ATOMICS = {"v03_c1shape_k8", "v04_h32_k3_diag", "v10_chain16_k8", "v11_dipep_k4"}     # re-run: bit-identical results
MISALIGNED = {"v11_dipep_k4", "v15_dipep_records_diag_k3"}                                # also run on a misaligned batch


_VARIANT_PARAMS = [(n, b, 0) for n in sorted(VARIANTS) for b in ("split", "whole")] + \
                  [(n, "whole", 1) for n in sorted(MISALIGNED)]


@pytest.mark.parametrize("name,sched,offset", _VARIANT_PARAMS)
def test_fast_variant_matches_oracle(name, sched, offset, tmp_path):
    """Every fast-path variant at B_SMALL (split schedule) and B_LARGE (whole-tile schedule) against the multiplicity oracle."""
    dims, k, pp_kind, use_diag, _ = VARIANTS[name]
    seed = 1000 + sorted(VARIANTS).index(name)
    pp, ppo, D_host, tot_dim = preprocessing(pp_kind, seed)
    diag = (0.5 + np.random.default_rng(seed).random(tot_dim)).astype(np.float32) if use_diag else None
    nets = random_nets(dims, k, seed)
    task, model = eigen_task(tmp_path, pp, dims, k, nets, D_host, diag=diag)
    assert task._ctx.fast_path, name
    B = B_SMALL if sched == "split" else B_LARGE
    assert schedule(B, k) == sched
    X, w, w_agg, _ = repeated_batch(D_host, B, seed + B, offset)
    assert (X.data_ptr() % 16 != 0) == bool(offset)          # dipeptide frames are 264 bytes: one frame in is 8 bytes off
    first = eigen_step(task, model, X, w)
    if name in ON_ATOMICS and sched == "whole":
        assert_bit_identical(first, eigen_step(task, model, X, w), name)
    del X, w
    comb, g64, _ = cf.eigen_loss_and_grads(D_host, w_agg, nets, ppo, 20.0, EIG_W[:k], diag)
    assert_eigen_envelope(first[0], first[1], comb, g64, f"{name} {sched} B={B}{' misaligned' if offset else ''}")


# --------------------------------------------------------------------------------------------- 3. transfer operator
@pytest.mark.parametrize("case", ["identity_k2_lag2", "c3shape_k3_lag3"])
def test_lag_loss_whole_tile_matches_gathered_oracle(case, tmp_path):
    """Transfer-operator loss (both forward passes, both backward passes seeded through y and y') on 2^17 frame pairs, in the
    whole-tile schedule, against the reference formula in fp64 on the gathered features of the distinct frames."""
    if case == "identity_k2_lag2":
        dims, k, lag, pp_kind = [2, 20, 20, 20, 1], 2, 2, ("identity", 2)
    else:
        dims, k, lag, pp_kind = [66, 20, 20, 20, 1], 3, 3, ("align", BASE, None)
    dt = 0.5
    seed = 51 + k
    pp, ppo, D_host, _ = preprocessing(pp_kind, seed)
    nets = random_nets(dims, k, seed)
    task, model = eigen_task(tmp_path, pp, dims, k, nets, D_host, lag_tau=lag * dt, dt=dt)
    B = 1 << 17
    assert task.lag_idx == lag and task._ctx.fast_path and schedule(B, k) == "whole"
    X, w, _, idx = repeated_batch(D_host, B + lag, seed)
    out, grads = eigen_step(task, model, X[:-lag], w[:-lag], X[lag:], w[lag:])
    idx, w = idx.cpu().numpy(), w.cpu().numpy().astype(np.float64)
    del X
    R = ppo.prepare(D_host.astype(np.float64))["r"]
    gold, g64 = lag_oracle(R, idx, w, nets, 20.0, EIG_W[:k], lag, lag * dt)
    assert_eigen_envelope(out, grads, gold, g64, f"lag {case} B=2^17")
