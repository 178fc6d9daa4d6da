"""The general eigenfunction kernels on every tile layout a network's shape selects, against an fp64 oracle.

Every EigenFunctionTask outside the thread-private fast path (any hidden width other than a uniform 16, 20 or 32, any depth
other than 2 or 3 hidden layers, every activation other than tanh, diag_coeff with an alignment, position records after an
alignment) runs on eigen_kernel<GRAD, 2> in csrc/cvf_eigen.cu.  finish_plan gives it the largest tile of F in {128, 64, 32}
frames whose shared-memory state (layout_plan) fits the device's opt-in shared memory, and refuses the shape when none does.
Every case names its F, checks it with a line-for-line mirror of layout_plan fed the device's cap, and checks the launch
accounting: one eigen_stats(general) and one eigen_grad(general) per step and no launch of the fast path.

The oracle is the multiplicity construction of test_step_at_scale_gpu.py: a batch is X = D[idx] with M distinct frames D, so
the fp64 result on D with the per-frame aggregated weights is the fp64 result of the whole batch at any B.  Tanh networks use
oracle.closed_form.eigen_loss_and_grads, other activations fp64 torch autograd of oracle.ref_torch.eigen_loss.  The bars are
those of the step at scale (loss 1e-6, eigenvalues 2e-6, every gradient tensor 5e-5 relative L2), plus 1e-6 on the batch's
Dirichlet sums SD of pass 1 (1e-5 where an alignment and diag_coeff keep the fp32 Kabsch adjoint in the J phase); each bar gives way to FLOOR_SLACK times the error of torch's own fp32 run of the same batch where
that is larger (small batches whose variance is a cancelling difference; that fp32 run pre-processes in fp64).
"""
import gc
import re

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
M = 2048                          # distinct frames behind every batch
FLOOR_SLACK = 8.0                 # bars give way to this multiple of torch's fp32 error (module docstring)
EIG_W = [1.0, 0.6, 0.3, 0.2, 0.15, 0.1, 0.05, 0.03]
ALPHA = 20.0
BASE = bd.DIPEPTIDE_NM * 10.0
FAST_KERNELS = ("fast_pack", "fast_prep", "fast_pass1", "fast_stats", "fast_pass2", "fast_jjt")


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(autouse=True)
def release_memory():
    yield
    gc.collect()
    torch.cuda.empty_cache()


# --------------------------------------------------------------------------------------------- configuration mirror
def _r4(v):
    return (v + 3) & ~3


def state_bytes(spec, dims, k, F):
    """Shared memory of eigen_kernel at F frames per tile, as layout_plan computes it: k padded parameter blocks, the
    combine vector and the stats reduction scratch (doubles), then rows of F + 4 floats: weight, ones, seed, R (9), K^-1 (6),
    y (k), D (k), the frame (positions Y, and features r unless they alias Y), and the network region: A and G of every
    hidden layer, then max(T and S of every hidden layer, T_1 S_1 followed by V (d_r) and GX (3 n_used unless aliased))."""
    L = len(dims) - 1
    params = k * sum(dims[l + 1] * _r4(dims[l]) + _r4(dims[l + 1]) for l in range(L))
    n_stats = 1 + 2 * k + k * k
    off = _r4(params + _r4(2 * (3 + 5 * k + k * k)) + 2 * 4 * n_stats)
    pos_alias = spec.kind == 1 and bool(spec.positions_only)
    rows = 3 + 9 + 6 + 2 * k
    if spec.kind == 1:
        rows += 3 * spec.n_used + (0 if pos_alias else spec.d_r)
    else:
        rows += spec.d_r
    sum_h = sum(dims[1:L])
    a_g = 2 * sum_h
    t = a_g + (2 * sum_h if L > 1 else 0)
    after1 = a_g + (2 * dims[1] if L > 1 else 0)
    vend = after1 + spec.d_r + (3 * spec.n_used if spec.kind == 1 and not pos_alias else 0)
    return 4 * (off + (rows + max(t, vend)) * (F + 4))


def configuration(spec, dims, k, cap):
    """Frames per tile finish_plan chooses (128, 64 or 32), or None where it refuses the shape."""
    for F in (128, 64, 32):
        if state_bytes(spec, dims, k, F) <= cap:
            return F
    return None


def device_cap():
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# --------------------------------------------------------------------------------------------- pre-processing of the cases
SUB = [0, 4, 6, 8, 10, 14, 16, 18]                  # alignment subset of the dipeptide
RECORDS = [("position", [4]), ("bond", [4, 6]), ("dihedral", [4, 6, 8, 14]), ("position", [8]), ("angle", [6, 8, 14]),
           ("bond", [1, 18])]
RECORDS_SEL = [1, 5, 9, 12, 17, 20]                 # alignment atoms, five of them read by no record
C4_BASE = bd.chain_structure(166, seed=2026)
C4_FEATS, C4_SEL = bd.c4_features()


def preprocessing(kind, seed):
    """(pp layer, closed-form Preproc, torch restatement, distinct frames D (fp32 host), coordinates per frame)."""
    from colvarsfinder import utils
    if kind[0] == "identity":                       # ("identity", d[, scale])
        scale = kind[2] if len(kind) > 2 else 1.0
        D = (scale * np.random.default_rng(seed).normal(size=(M, kind[1]))).astype(np.float32)
        return torch.nn.Identity(), cf.Preproc(identity=True), ref_torch.Preprocess(), D, kind[1]
    if kind[0] == "align":                          # ("align", base, alignment atoms or None for all): aligned positions
        base, sel = kind[1], kind[2] if kind[2] is not None else list(range(len(kind[1])))
        D = ref_torch.synth_frames(base, M, seed=seed)
        return (utils.Align(base[sel], sel), cf.Preproc(align_idx=sel, ref=base[sel]),
                ref_torch.Preprocess(ref_torch.Align(base[sel], sel)), D, 3 * len(base))
    base, feats, sel = kind[1], kind[2], kind[3]    # ("features", base, records, alignment atoms)
    D = ref_torch.synth_frames(base, M, seed=seed)
    return (utils.Preprocessing(utils.Align(base[sel], sel), utils.FeatureMap(feats)),
            cf.Preproc(align_idx=sel, ref=base[sel], feats=feats),
            ref_torch.Preprocess(ref_torch.Align(base[sel], sel), ref_torch.FeatureMap(feats)), D, 3 * len(base))


# --------------------------------------------------------------------------------------------- models and oracle
ACT_MODULES = {"tanh": torch.nn.Tanh, "sigmoid": torch.nn.Sigmoid, "softplus": torch.nn.Softplus, "elu": torch.nn.ELU,
               "relu": torch.nn.ReLU}
ACT_FUNCS = {"tanh": torch.tanh, "sigmoid": torch.sigmoid, "softplus": torch.nn.functional.softplus,
             "elu": torch.nn.functional.elu, "relu": torch.relu}


def random_nets(dims, k, seed):
    torch.manual_seed(seed)
    return [[p.numpy() for p in ref_torch.init_mlp_params(dims)] for _ in range(k)]


def eigen_task(tmp_path, pp, dims, k, nets, D, act="tanh", diag=None, lag_tau=0.0, dt=1.0):
    """EigenFunctionTask with the networks `nets`, built as bench.py builds it."""
    from colvarsfinder import core, nn
    model = nn.EigenFunctions(dims, k, ACT_MODULES[act]())
    with torch.no_grad():
        for f, ps in zip(model.eigen_funcs, nets):
            for p, v in zip(f.parameters(), ps):
                p.copy_(torch.as_tensor(v))
    small = np.ascontiguousarray(D[:64])
    task = core.EigenFunctionTask(FakeTrajectory(small, np.ones(len(small)), dt=dt), pp, model, str(tmp_path), ALPHA,
                                  EIG_W[:k], diag_coeff=None if diag is None else torch.as_tensor(diag), lag_tau=lag_tau,
                                  k=k, device=DEV, verbose=False, debug_mode=False)
    return task, model


def torch_eigen(D, w, nets, pp_t, diag, act, dtype):
    """Loss, eigenvalues, cvec, Dirichlet sums SD and parameter gradients by torch autograd of ref_torch.eigen_loss in
    `dtype`."""
    k = len(nets)
    X = torch.tensor(D, dtype=dtype, requires_grad=True)
    wt = torch.as_tensor(w, dtype=dtype)
    a = None if diag is None else torch.as_tensor(diag, dtype=dtype)
    tn = [[torch.tensor(p, dtype=dtype, requires_grad=True) for p in n] for n in nets]
    f = ACT_FUNCS[act]
    y = ref_torch.eigen_forward(tn, pp_t(X), f)
    SD = []
    for i in range(k):
        g = torch.autograd.grad(y[:, i].sum(), X, retain_graph=True)[0].reshape(len(D), -1)
        SD.append(float((((g * g) if a is None else (g * g * a)).sum(1) * wt).sum()))
    loss, eig, _, _, cvec = ref_torch.eigen_loss(X, wt, tn, pp_t, ALPHA, EIG_W[:k], a, act=f)
    loss.backward()
    grads = [[np.zeros(tuple(p.shape)) if p.grad is None else p.grad.numpy().astype(np.float64) for p in n] for n in tn]
    return dict(loss=float(loss), eig=eig.numpy().astype(np.float64), cvec=[int(v) for v in cvec], SD=np.array(SD)), grads


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def oracle(D, w_agg, nets, ppo, pp_t, diag, act):
    """(fp64 result, fp64 gradients, floors): the floors are the errors of torch's fp32 run of the networks on the batch's
    distinct frames (the pre-processing of that run stays in fp64: torch's fp32 SVD alignment is far less accurate than the
    kernel's fp64 Kabsch step and would hide kernel errors)."""
    nz = w_agg > 0
    Dn, wn = D[nz], w_agg[nz]
    if act == "tanh":
        comb, g64, S = cf.eigen_loss_and_grads(Dn, wn, nets, ppo, ALPHA, EIG_W[:len(nets)], diag)
        ref = dict(loss=comb["loss"], eig=comb["eig"], cvec=[int(v) for v in comb["cvec"]], SD=S["SD"])
    else:
        ref, g64 = torch_eigen(Dn.astype(np.float64), wn, nets, pp_t, diag, act, torch.float64)
    r32, g32 = torch_eigen(Dn, wn.astype(np.float32), nets, lambda X: pp_t(X.double()).float(), diag, act, torch.float32)
    scale = max(np.abs(t).max() for n in g64 for t in n)
    # gradients that are zero in fp64 (the last-layer biases): torch's fp32 value relative to the largest gradient entry
    floors = dict(loss=abs(r32["loss"] - ref["loss"]) / abs(ref["loss"]), eig=_rel(r32["eig"], ref["eig"]),
                  SD=_rel(r32["SD"], ref["SD"]),
                  grads=[[float(np.abs(a).max() / scale) if np.abs(b).max() < 1e-9 * scale else C.rel_l2(a, b)
                          for a, b in zip(na, nb)] for na, nb in zip(g32, g64)])
    return ref, g64, floors


def assert_matches(res, ref, g64, floors, tag, sd_bar=1e-6):
    """cvec exact; loss, eigenvalues, SD and every gradient tensor within their bars (module docstring); gradients that are
    zero in fp64 (the last-layer biases) below 1e-5 of the largest gradient entry, or FLOOR_SLACK times torch's fp32 value."""
    (loss, eig, _, _, cvec), grads, SD = res["out"], res["grads"], res["SD"]
    assert [int(v) for v in cvec.cpu().numpy()] == ref["cvec"], (tag, cvec, ref["cvec"])
    e_loss = abs(float(loss) - ref["loss"]) / abs(ref["loss"])
    e_eig = _rel(eig.cpu().numpy(), ref["eig"])
    e_sd = _rel(SD, ref["SD"])
    scale = max(np.abs(t).max() for n in g64 for t in n)
    errs, zeros = [], []
    for i in range(len(g64)):
        for j in range(len(g64[i])):
            got = grads[i][j].cpu().numpy()
            if np.abs(g64[i][j]).max() < 1e-9 * scale:
                zeros.append((float(np.abs(got).max() / scale), floors["grads"][i][j]))
            else:
                errs.append((C.rel_l2(got, g64[i][j]), floors["grads"][i][j]))
    print(f"[{tag}] loss {e_loss:.1e}  eig {e_eig:.1e}  SD {e_sd:.1e}  grad rel-L2 max {max(e for e, _ in errs):.1e}  "
          f"zero-grad {max(z for z, _ in zeros) if zeros else 0.0:.1e}  (torch fp32: loss {floors['loss']:.1e}, eig {floors['eig']:.1e}, "
          f"SD {floors['SD']:.1e}, grad max {max(f for _, f in errs):.1e})")
    assert e_loss <= max(1e-6, FLOOR_SLACK * floors["loss"]), (tag, "loss", e_loss, floors["loss"])
    assert e_eig <= max(2e-6, FLOOR_SLACK * floors["eig"]), (tag, "eig", e_eig, floors["eig"])
    assert e_sd <= max(sd_bar, FLOOR_SLACK * floors["SD"]), (tag, "SD", e_sd, floors["SD"])
    for e, f in errs:
        assert e <= max(5e-5, FLOOR_SLACK * f), (tag, "gradient", errs)
    for z, f in zeros:
        assert z < max(1e-5, FLOOR_SLACK * f), (tag, "zero-grad", zeros)


def launches(launched, name):
    return launched[name][2]


def step(task, model, X, w, Xl=None, wl=None):
    """Loss outputs, parameter gradients and the launches of one training step."""
    from colvarsfinder import _lib
    torch.cuda.synchronize()
    _lib.profile_read(reset=True)
    model.zero_grad(set_to_none=True)
    out = task.loss_func(X, w, Xl, wl)
    out[0].backward()
    torch.cuda.synchronize()
    launched = _lib.profile_read(reset=True)
    grads = [[p.grad.detach().clone() for p in f.parameters()] for f in model.eigen_funcs]
    return dict(out=out, grads=grads, launched=launched)


def assert_general_launches(launched, tag, stats=1):
    assert launches(launched, "eigen_grad(general)") == 1, (tag, launched)
    if stats is not None:
        assert launches(launched, "eigen_stats(general)") == stats, (tag, launched)
    assert all(launches(launched, n) == 0 for n in FAST_KERNELS), (tag, launched)


def assert_bit_identical(a, b, tag):
    assert torch.equal(a["out"][0], b["out"][0]) and torch.equal(a["out"][1], b["out"][1]), (tag, "loss / eigenvalues differ")
    for ga, gb in zip(a["grads"], b["grads"]):
        for ta, tb in zip(ga, gb):
            assert torch.equal(ta, tb), (tag, "gradients differ")


def float4_tile(spec):
    """load_tile reads whole tiles of an aligned batch with 16-byte loads (Identity, or every atom used in order)."""
    return spec.kind == 0 or bool(spec.used_identity)


def run_case(tmp_path, tag, dims, k, kind, use_diag, act, B, F, seed, nets=None, full_checks=False):
    pp, ppo, pp_t, D, tot_dim = preprocessing(kind, seed)
    diag = (0.5 + np.random.default_rng(seed).random(tot_dim)).astype(np.float32) if use_diag else None
    nets = random_nets(dims, k, seed) if nets is None else nets
    task, model = eigen_task(tmp_path, pp, dims, k, nets, D, act, diag)
    spec = task._ctx.spec.struct
    assert not task._ctx.fast_path, tag
    assert configuration(spec, dims, k, device_cap()) == F, (tag, [state_bytes(spec, dims, k, f) for f in (128, 64, 32)])
    X, w, w_agg, _ = C.repeated_batch(D, B, seed + B)
    _, S = task._ctx.stats(X, w)
    first = step(task, model, X, w)
    first["SD"] = S.cpu().numpy()[1 + k + k * k:]
    assert_general_launches(first["launched"], tag)
    if full_checks:
        second = step(task, model, X, w)
        assert_general_launches(second["launched"], tag)
        assert_bit_identical(first, second, tag + " second run")
        fl = tot_dim
        if float4_tile(spec) and fl % 4 != 0:
            Xm, wm, _, _ = C.repeated_batch(D, B, seed + B, offset=1)
            assert Xm.data_ptr() % 16 != 0 and torch.equal(Xm, X)
            mis = step(task, model, Xm, wm)
            assert_general_launches(mis["launched"], tag)
            assert_bit_identical(first, mis, tag + " misaligned view")
    del X, w
    ref, g64, floors = oracle(D, w_agg, nets, ppo, pp_t, diag, act)
    # With an alignment and diag_coeff the J phase (dg/dx through the Kabsch adjoint, weighted, and back) runs in fp32 over
    # every used atom; there SD is within 1e-5 (8.7e-6 measured for C4's 95 atoms, 2.6e-6 for the dipeptide records).
    assert_matches(first, ref, g64, floors, tag, 1e-5 if spec.kind == 1 and spec.n_align > 0 and use_diag else 1e-6)


# --------------------------------------------------------------------------------------------- 1. layout matrix
# F -> {name: (layer dims, k, pre-processing, diag_coeff)}: every F runs at least two pre-processings; the last Identity shape
# of each F is the widest input [d,24,24,24,1] that still takes it (d = 64, 189 and 321 take the next F or are refused)
LAYOUTS = {
    128: {"id5-24-diag": ([5, 24, 24, 24, 1], 3, ("identity", 5), True),
          "c3-diag": ([66, 20, 20, 20, 1], 3, ("align", BASE, None), True),
          "id7-L1-k8": ([7, 1], 8, ("identity", 7), False),
          "id63-24": ([63, 24, 24, 24, 1], 3, ("identity", 63), False)},
    64: {"dip-30": ([66, 30, 30, 30, 1], 3, ("align", BASE, None), False),
         "dip-sub-diag-k8": ([66, 20, 20, 20, 1], 8, ("align", BASE, SUB), True),
         "id188-24": ([188, 24, 24, 24, 1], 3, ("identity", 188), False)},
    32: {"dip-45": ([66, 45, 45, 45, 1], 3, ("align", BASE, None), False),
         "records-sub-diag-50": ([11, 50, 50, 50, 1], 3, ("features", BASE, RECORDS, RECORDS_SEL), True),
         "c4-diag": ([81, 20, 20, 20, 1], 3, ("features", C4_BASE, C4_FEATS, C4_SEL), True),
         "id5-L8-k8": ([5, 27, 1, 19, 33, 30, 22, 37, 1], 8, ("identity", 5), False),
         "id320-24": ([320, 24, 24, 24, 1], 3, ("identity", 320), False)},
}
# one activation other than tanh per entry, at the largest batch
OTHER_ACT = [(128, "id5-24-diag", "relu"), (64, "dip-30", "sigmoid"), (32, "records-sub-diag-50", "softplus"),
             (32, "id5-L8-k8", "elu")]
BIG = "2gF+17"                    # two tiles per CTA of the full grid and a ragged tail: every CTA walks several tiles


def _layout_params():
    out = []
    for F, shapes in LAYOUTS.items():
        for name in shapes:
            for b in [str(v) for v in sorted({2, 31, 33, F - 1, F + 1})] + [BIG]:
                out.append(pytest.param(F, name, b, "tanh", id=f"F{F}-{name}-B{b}"))
    for F, name, act in OTHER_ACT:
        out.append(pytest.param(F, name, BIG, act, id=f"F{F}-{name}-B{BIG}-{act}"))
    return out


@pytest.mark.parametrize("F,name,bname,act", _layout_params())
def test_general_layout_matches_oracle(F, name, bname, act, tmp_path):
    """The general kernels in every tile layout, at ragged batch sizes around one tile and at two tiles per CTA of the full
    grid plus 17 frames.  At that size a second run is bit-identical, and a misaligned view of the same batch (which moves
    load_tile from 16-byte loads to the per-element gather) gives bit-identical results."""
    dims, k, kind, use_diag = LAYOUTS[F][name]
    B = 2 * sm_count() * F + 17 if bname == BIG else int(bname)
    seed = 100 + 10 * sorted(LAYOUTS).index(F) + list(LAYOUTS[F]).index(name)
    run_case(tmp_path, f"F{F} {name} B={B} {act}", dims, k, kind, use_diag, act, B, F, seed, full_checks=bname == BIG)


# --------------------------------------------------------------------------------------------- 2. saturated activations
def threshold_chain(seed, centre=15.15, spread=0.2, h=12, L=8, d=5):
    """Softplus chain whose pre-activations sit just above 15 in every hidden layer (unit 0 of each layer near 22, past
    Softplus's threshold of 20): the network is nearly linear there, and 1 - softplus'(z) = exp(-z) is a few 1e-7 per
    layer.  Every W_l is small enough that the spread of a layer's pre-activations stays near `spread`."""
    rng = np.random.default_rng(seed)
    c = np.full(h, centre)
    c[0] = 22.0
    nets = []
    for _ in range(2):
        ps, prev = [], None
        for l in range(L):
            nin = d if l == 0 else h
            nout = 1 if l == L - 1 else h
            W = rng.normal(size=(nout, nin)) * (spread / np.sqrt(nin) if l == 0 else 1.0 / np.sqrt(nin))
            b = np.zeros(nout) if l == L - 1 else c.copy()
            if l > 0:
                b = b - W @ prev
            prev = np.log1p(np.exp(c))          # softplus of the centres: what the next layer receives
            ps += [W.astype(np.float32), b.astype(np.float32)]
        nets.append(ps)
    return nets


SATURATED = {"softplus": ("identity", 5, 30.0), "sigmoid": ("identity", 5, 30.0), "elu": ("identity", 5, 30.0),
             "softplus-threshold": ("identity", 5)}


@pytest.mark.parametrize("case", list(SATURATED))
def test_saturated_activations_match_oracle(case, tmp_path):
    """Inputs scaled by 30 put many first-layer pre-activations past Softplus's threshold of 20 and deep into the flat
    parts of Sigmoid and ELU.  `softplus-threshold` runs a constructed 8-layer Softplus chain with pre-activations just
    above 15 (and one unit per layer past 20): its Dirichlet sums would be off by several 1e-6 if the kernel took the
    threshold branch of softplus' below 20."""
    act = case.split("-")[0]
    kind = SATURATED[case]
    if case == "softplus-threshold":
        dims, nets = [5] + [12] * 7 + [1], threshold_chain(77)
    else:
        dims, nets = [5, 24, 24, 24, 1], None
    F = 128
    B = 2 * sm_count() * F + 17
    run_case(tmp_path, f"saturated {case} B={B}", dims, 2, kind, False, act, B, F, 70 + list(SATURATED).index(case), nets)


# --------------------------------------------------------------------------------------------- 3. refusal edge
# family -> (pre-processing, diag_coeff, k, widths h of [d_r,h,h,h,1]: the last that fits and the first that does not)
EDGES = {"identity-2": (("identity", 2), False, 3, 65, 66),
         "dipeptide-aligned": (("align", BASE, None), False, 3, 55, 56),
         "c4-diag": (("features", C4_BASE, C4_FEATS, C4_SEL), True, 3, 38, 39)}


@pytest.mark.parametrize("family", list(EDGES))
def test_refusal_edge(family, tmp_path):
    """The widest hidden layers that fit at F = 32 run and match the oracle; one unit more is refused with a RuntimeError
    that states the bytes needed at 32 frames (equal to the mirror's) and the device's cap, and nothing is launched."""
    from colvarsfinder import _lib
    kind, use_diag, k, h_fit, h_refused = EDGES[family]
    cap = device_cap()
    seed = 200 + list(EDGES).index(family)
    pp, _, _, D, tot_dim = preprocessing(kind, seed)
    d_r = tot_dim if kind[0] != "features" else 81
    fit, refused = [d_r, h_fit, h_fit, h_fit, 1], [d_r, h_refused, h_refused, h_refused, 1]
    B = 2 * sm_count() * 32 + 17
    run_case(tmp_path, f"edge {family} {fit}", fit, k, kind, use_diag, "tanh", B, 32, seed)
    diag = (0.5 + np.random.default_rng(seed).random(tot_dim)).astype(np.float32) if use_diag else None
    task, _ = eigen_task(tmp_path, pp, refused, k, random_nets(refused, k, seed), D, diag=diag)
    spec = task._ctx.spec.struct
    assert configuration(spec, refused, k, cap) is None
    X, w, _, _ = C.repeated_batch(D, 300, seed)
    torch.cuda.synchronize()
    _lib.profile_read(reset=True)
    with pytest.raises(RuntimeError, match="does not fit shared memory") as e:
        task.loss_func(X, w)
    launched = _lib.profile_read(reset=True)
    m = re.search(r"\((\d+) B needed at 32 frames, (\d+) available\)", str(e.value))
    assert m, str(e.value)
    print(f"[edge {family}] {fit} fits; {refused}: {m.group(0)}")
    assert int(m.group(1)) == state_bytes(spec, refused, k, 32) and int(m.group(2)) == cap, (str(e.value), cap)
    assert launches(launched, "eigen_stats(general)") == 0, launched


def test_refuses_k9_and_nine_layers(tmp_path):
    """k = 9 eigenfunctions and 9 linear layers are outside the envelope, and both say so when the task is built."""
    pp, _, _, D, _ = preprocessing(("identity", 3), 9)
    with pytest.raises(RuntimeError, match="k = 9 eigenfunctions is outside the supported envelope"):
        eigen_task(tmp_path, pp, [3, 24, 24, 1], 9, random_nets([3, 24, 24, 1], 9, 9), D)
    dims = [3] + [8] * 8 + [1]
    with pytest.raises(RuntimeError, match="networks with 9 linear layers are outside the supported envelope"):
        eigen_task(tmp_path, pp, dims, 2, random_nets(dims, 2, 9), D)


# --------------------------------------------------------------------------------------------- 4. transfer operator
LAG = {"F128-id5-24": ([5, 24, 24, 24, 1], 3, ("identity", 5), 128),
       "F32-records-sub-50": ([11, 50, 50, 50, 1], 3, ("features", BASE, RECORDS, RECORDS_SEL), 32)}


@pytest.mark.parametrize("case", list(LAG))
def test_lag_loss_on_general_kernel_matches_gathered_oracle(case, tmp_path):
    """The transfer-operator loss (both forward passes, both backward passes seeded through y and y') on the general kernel
    at two tiles per CTA of the full grid plus 17 frame pairs, against the reference formula in fp64 on the gathered features.
    The F = 32 case keeps its alignment (position records).  tlag_terms_kernel counts as an eigen_stats launch, so only the
    eigen_grad launches and the absence of the fast path are checked."""
    dims, k, kind, F = LAG[case]
    lag, dt = 2, 0.5
    seed = 60 + list(LAG).index(case)
    pp, ppo, _, D, _ = preprocessing(kind, seed)
    nets = random_nets(dims, k, seed)
    task, model = eigen_task(tmp_path, pp, dims, k, nets, D, lag_tau=lag * dt, dt=dt)
    spec = task._ctx.spec.struct
    assert task.lag_idx == lag and not task._ctx.fast_path
    assert configuration(spec, dims, k, device_cap()) == F
    B = 2 * sm_count() * F + 17
    X, w, _, idx = C.repeated_batch(D, B + lag, seed)
    r = step(task, model, X[:-lag], w[:-lag], X[lag:], w[lag:])
    assert launches(r["launched"], "eigen_grad(general)") == 2, (case, r["launched"])
    assert all(launches(r["launched"], n) == 0 for n in FAST_KERNELS), (case, r["launched"])
    idx, w = idx.cpu().numpy(), w.cpu().numpy().astype(np.float64)
    del X
    R = ppo.prepare(D.astype(np.float64))["r"]
    gold, g64 = C.lag_oracle(R, idx, w, nets, ALPHA, EIG_W[:k], lag, lag * dt)
    _assert_envelope(r, gold, g64, f"lag {case} B={B}")


def _assert_envelope(r, gold, g64, tag, grad_bar=5e-5):
    """The bars of the step at scale (loss 1e-6, eigenvalues 2e-6, gradients 5e-5 relative L2), no floor."""
    loss, eig, _, _, cvec = r["out"]
    assert [int(v) for v in cvec.cpu().numpy()] == list(gold["cvec"]), (tag, cvec, gold["cvec"])
    e_loss = abs(float(loss) - gold["loss"]) / abs(gold["loss"])
    e_eig = _rel(eig.cpu().numpy(), gold["eig"])
    scale = max(np.abs(t).max() for n in g64 for t in n)
    errs = [C.rel_l2(r["grads"][i][j].cpu().numpy(), g64[i][j]) for i in range(len(g64)) for j in range(len(g64[i]))
            if np.abs(g64[i][j]).max() >= 1e-9 * scale]
    print(f"[{tag}] loss {e_loss:.1e}  eig {e_eig:.1e}  grad rel-L2 max {max(errs):.1e} median {np.median(errs):.1e}")
    assert e_loss <= 1e-6 and e_eig <= 2e-6 and max(errs) <= grad_bar, (tag, e_loss, e_eig, errs)


# --------------------------------------------------------------------------------------------- 5. training sizes
# C4 with diag_coeff keeps its alignment: the fp32 J phase over 95 used atoms leaves 2e-5 to 6.5e-5 relative L2 on every
# gradient tensor (median 2.7e-5 at 2^18 frames, 2.3e-5 max at 9 489 frames), the same at every batch size and layout, so its
# gradient bar is 1e-4; C3 with diag_coeff (22 atoms) stays under 5e-6.
TRAINING = {"c3-diag-2^20": ([66, 20, 20, 20, 1], ("align", BASE, None), 1 << 20, 128, 5e-5),
            "c4-diag-2^18": ([81, 20, 20, 20, 1], ("features", C4_BASE, C4_FEATS, C4_SEL), 1 << 18, 32, 1e-4)}


@pytest.mark.parametrize("case", list(TRAINING))
def test_training_size_matches_oracle(case, tmp_path):
    """C3 and C4 with diag_coeff (which keeps them off the fast path), k = 3, at training batch sizes: 2^20 frames at F = 128,
    and 2^18 frames at F = 32 (about 55 tiles per CTA)."""
    dims, kind, B, F, grad_bar = TRAINING[case]
    k = 3
    seed = 80 + list(TRAINING).index(case)
    pp, ppo, _, D, tot_dim = preprocessing(kind, seed)
    diag = (0.5 + np.random.default_rng(seed).random(tot_dim)).astype(np.float32)
    nets = random_nets(dims, k, seed)
    task, model = eigen_task(tmp_path, pp, dims, k, nets, D, diag=diag)
    assert not task._ctx.fast_path and configuration(task._ctx.spec.struct, dims, k, device_cap()) == F
    X, w, w_agg, _ = C.repeated_batch(D, B, seed)
    r = step(task, model, X, w)
    assert_general_launches(r["launched"], case)
    del X, w
    comb, g64, _ = cf.eigen_loss_and_grads(D, w_agg, nets, ppo, ALPHA, EIG_W[:k], diag)
    _assert_envelope(r, dict(loss=comb["loss"], eig=comb["eig"], cvec=[int(v) for v in comb["cvec"]]), g64,
                     f"{case} ({-(-B // F) / sm_count():.0f} tiles per CTA)", grad_bar)
