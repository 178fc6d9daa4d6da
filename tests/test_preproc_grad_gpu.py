"""First-order gradients through the pre-processing layers (utils.Align, FeatureMap, Preprocessing): the CUDA backward
(cvf_align_vjp, cvf_features_vjp under torch autograd) against the fp64 closed form, the rigid-motion invariances, two
independent CUDA paths, and the exported TorchScript model.

Envelope (SURVEY 7.3-D for gradients): rel-L2 <= max(2e-5, rel-L2 of fp32 autograd through oracle/ref_torch.Preprocess on the
same fp32 inputs).  Large batches are X = D[idx] over M distinct frames D with the cotangent U[idx] (as in
tests/test_step_at_scale_gpu.py): frame f's gradient is the oracle's for frame idx_f, so the fp64 oracle runs on M frames only."""
import copy
import os

import numpy as np
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_torch
from oracle.ref_import import FakeTrajectory
from tests import _cases as C

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None
BASE = ref_torch.DIPEPTIDE_NM * 10.0
ALL = list(range(22))
SUB = [1, 4, 5, 6, 8, 10, 14, 15, 16, 18]
FEATS = C.eigen_case("eigen_dipep_features")["features"]           # bonds, angles, dihedrals and two positions
INVARIANT = C.eigen_case("eigen_dipep_invariant")["features"]      # bonds, angles, dihedrals only
M_MAX = 4099


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__ as g
    g.build()


def _layer(name, base=BASE):
    """(pp_layer of this package, fp64 closed-form oracle, fp32 autograd restatement) of one pre-processing layer."""
    from colvarsfinder import utils
    n = len(base)
    sel = {"align": list(range(n)), "align_subset": list(range(0, n, 7)), "positions": ALL, "subset": SUB, "features": SUB,
           "invariant": ALL, "unaligned": None, "unaligned_invariant": None}[name]
    feats = {"features": FEATS, "invariant": INVARIANT, "unaligned": FEATS, "unaligned_invariant": INVARIANT}.get(name)
    al = None if sel is None else utils.Align(base[sel], sel)
    fm = None if feats is None else utils.FeatureMap(feats)
    if name in ("align", "align_subset"):
        mod = al                                    # the bare module: [B,N,3] -> [B,N,3]
    elif name in ("unaligned", "unaligned_invariant"):
        mod = fm                                    # the bare module: [B,N,3] -> [B,d_r]
    else:
        mod = utils.Preprocessing(al, fm)
    mod = mod.to(DEV)
    ppo = cf.Preproc(align_idx=sel, ref=None if sel is None else base[sel], feats=feats)
    ppt = ref_torch.Preprocess(None if sel is None else ref_torch.Align(base[sel], sel),
                               None if feats is None else ref_torch.FeatureMap(feats))
    return mod, ppo, ppt


LAYERS = ["align", "positions", "subset", "features", "invariant", "unaligned"]


def _frames(M, seed, base=BASE):
    return ref_torch.synth_frames(base, M, seed=seed).astype(np.float32)


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm())


def _oracle(ppo, ppt, D, U):
    """(fp64 closed-form g_x [M,N,3], rel-L2 of the fp32 restatement's g_x against it) for frames D, cotangent U [M, ...]."""
    M = D.shape[0]
    st = ppo.prepare(D.astype(np.float64))
    g64 = ppo.vjp(st, U.reshape(M, -1).astype(np.float64)).reshape(D.shape)
    xt = torch.as_tensor(D).requires_grad_()
    rt = ppt(xt)
    g32, = torch.autograd.grad(rt, xt, torch.as_tensor(U).reshape(rt.shape))
    return g64, _rel(g32, torch.as_tensor(g64))


def _check_vjp(mod, ppo, ppt, D, B, seed):
    """g_x of mod on the batch D[idx] (idx = identity when B = M) against the oracle; returns (error, envelope)."""
    M = D.shape[0]
    g = torch.Generator(device=DEV).manual_seed(seed)
    idx = None if B == M else torch.randint(0, M, (B,), generator=g, device=DEV)
    Dd = torch.as_tensor(D, device=DEV)
    x = (Dd if idx is None else Dd[idx]).clone().requires_grad_()
    out = mod(x)
    U = np.random.default_rng(seed).standard_normal((M,) + tuple(out.shape[1:])).astype(np.float32)
    Ud = torch.as_tensor(U, device=DEV)
    gx, = torch.autograd.grad(out, x, Ud if idx is None else Ud[idx])
    g64, env32 = _oracle(ppo, ppt, D, U)
    want = torch.as_tensor(g64, device=DEV)
    return _rel(gx, want if idx is None else want[idx]), max(2e-5, env32)


# --------------------------------------------------------------------------------------------- 1. parity with the fp64 oracle
@pytest.mark.parametrize("B", [1, 5, 127, 128, 129, 4099, 1 << 20])
@pytest.mark.parametrize("name", LAYERS)
def test_vjp_matches_closed_form(name, B):
    mod, ppo, ppt = _layer(name)
    err, env = _check_vjp(mod, ppo, ppt, _frames(min(B, M_MAX), seed=B), B, seed=B + 1)
    assert err <= env, (name, B, err, env)


# --------------------------------------------------------------------------------------------- 2. both alignment kernels
@pytest.mark.parametrize("n_atoms,name", [(22, "align_subset"), (60, "align"), (120, "align"), (300, "align"),
                                          (300, "align_subset"), (1000, "align"), (1000, "align_subset")])
def test_align_vjp_tile_and_warp_kernels(n_atoms, name):
    """22 / 60 atoms: thread-per-frame tile kernel (tiles of 64 / 32 frames); 120, 300 and 1000 atoms: warp per frame."""
    base = ref_torch.chain_structure(n_atoms) if n_atoms != 22 else BASE
    mod, ppo, ppt = _layer(name, base)
    D = _frames(257, seed=n_atoms, base=base)
    err, env = _check_vjp(mod, ppo, ppt, D, 257, seed=7)
    assert err <= env, (n_atoms, name, err, env)


def test_align_vjp_misaligned_input_view():
    """X[1:] starts 264 bytes into the buffer: not 16-byte aligned, so the tile kernel takes plain loads and stores."""
    mod, ppo, ppt = _layer("align")
    D = _frames(1001, seed=3)
    X = torch.as_tensor(D, device=DEV).requires_grad_()
    x = X[1:]
    assert x.data_ptr() % 16 != 0
    out = mod(x)
    assert torch.equal(out, mod(x.detach().clone()))
    U = np.random.default_rng(3).standard_normal((1000, 22, 3)).astype(np.float32)
    gX, = torch.autograd.grad(out, X, torch.as_tensor(U, device=DEV))
    g64, env32 = _oracle(ppo, ppt, D[1:], U)
    assert not gX[0].any()
    assert _rel(gX[1:], torch.as_tensor(g64, device=DEV)) <= max(2e-5, env32)


# --------------------------------------------------------------------------------------------- 3. invariances
def _random_rotation(seed):
    q, r = np.linalg.qr(np.random.default_rng(seed).standard_normal((3, 3)))
    q = q * np.sign(np.diag(r))
    return q if np.linalg.det(q) > 0 else -q


@pytest.mark.parametrize("name", ["align", "positions", "subset", "features", "invariant"])
def test_gradient_invariances(name):
    """r(x) does not change under a rigid motion of x: sum_j g_j = 0, sum_j x_j x g_j = 0, and x -> xQ + t maps g to gQ."""
    mod, _, _ = _layer(name)
    D = _frames(M_MAX, seed=21)
    x = torch.as_tensor(D, device=DEV).requires_grad_()
    out = mod(x)
    U = torch.randn(out.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
    g, = torch.autograd.grad(out, x, U)
    g64, x64 = g.double(), x.detach().double()
    assert float(g64.sum(1).norm()) <= 1e-5 * float(g64.norm())
    assert float(torch.linalg.cross(x64, g64, dim=2).sum(1).norm()) <= 2e-5 * float(g64.norm()) * float(x64.abs().max())
    Q = torch.as_tensor(_random_rotation(9), dtype=torch.float32, device=DEV)
    t = torch.tensor([3.0, -7.0, 11.0], device=DEV)
    x2 = (x.detach() @ Q + t).requires_grad_()
    g2, = torch.autograd.grad(mod(x2), x2, U)
    assert _rel(g2, g64 @ Q.double()) <= 1e-4


# --------------------------------------------------------------------------------------------- 4. whole models
def _eigen_task(c, tmp, pp):
    from colvarsfinder import core, nn
    model = nn.EigenFunctions(c["layer_dims"], c["k"])
    with torch.no_grad():
        for i in range(c["k"]):
            for p, v in zip(model.eigen_funcs[i].parameters(), c["params"][i]):
                p.copy_(torch.as_tensor(v))
    traj = FakeTrajectory(c["X"], c["w"].astype(np.float64), dt=1.0)
    return core.EigenFunctionTask(traj, pp, model, str(tmp), c["alpha"], c["eig_w"], diag_coeff=None, beta=c["beta"],
                                  sort_eigvals_in_training=c["sort"], k=c["k"], device=DEV, verbose=False, debug_mode=False)


@pytest.mark.parametrize("case,name", [("eigen_dipep_k3", "align"), ("eigen_dipep_features", "features"),
                                       ("eigen_dipep_invariant", "unaligned_invariant"), ("eigen_dipep_invariant", "invariant")])
def test_dirichlet_sums_match_autograd_of_colvar_model(case, name, tmp_path):
    """SD_i = sum_f w_f |grad_x y_i|^2 of pass 1 (the step kernels' own Jacobian products) against the same sum formed from
    torch.autograd.grad through colvar_model(), i.e. through the new backward kernels."""
    c = C.eigen_case(case)
    if name == "features":
        # the golden case has diag_coeff: the Dirichlet sum is then not a plain |grad|^2
        c = dict(c, diag_coeff=None)
    pp, _, _ = _layer(name)
    task = _eigen_task(c, tmp_path, pp)
    k = c["k"]
    X = torch.as_tensor(c["X"], dtype=torch.float32, device=DEV).contiguous()
    w = torch.as_tensor(c["w"], dtype=torch.float32, device=DEV).contiguous()
    _, stats = task._ctx.stats(X, w)
    sd = stats[1 + k + k * k:1 + 2 * k + k * k]
    cv = task.colvar_model()
    x = X.clone().requires_grad_()
    y = cv(x)
    for i in range(k):
        g, = torch.autograd.grad(y[:, i].sum(), x, retain_graph=True)
        mine = float((w.double() * (g.double() ** 2).sum((1, 2))).sum())
        assert abs(mine - float(sd[i])) <= 1e-5 * abs(float(sd[i])), (i, mine, float(sd[i]))


def _model_grads(cv, head, ppt, X, seed):
    """(CUDA-path g_x, fp64 g_x, fp32-reference rel-L2) of a Sequential(pp_layer, head) for a random cotangent."""
    x = torch.as_tensor(X, device=DEV).requires_grad_()
    out = cv(x)
    V = torch.randn(out.shape, generator=torch.Generator().manual_seed(seed))
    g, = torch.autograd.grad(out, x, V.to(DEV))
    res = {}
    for dt in (torch.float64, torch.float32):
        h = copy.deepcopy(head).to("cpu", dt)
        p = copy.deepcopy(ppt).to(dt)
        xt = torch.as_tensor(X, dtype=dt).requires_grad_()
        res[dt], = torch.autograd.grad(h(p(xt)), xt, V.to(dt))
    return g, res[torch.float64], _rel(res[torch.float32], res[torch.float64])


def test_autoencoder_colvar_model_gradient(tmp_path):
    from colvarsfinder import core, nn
    torch.manual_seed(1)
    X = _frames(3000, seed=4)
    mod, _, ppt = _layer("align")
    model = nn.AutoEncoder([66, 20, 20, 20, 2], [2, 10, 10, 66])
    task = core.AutoEncoderTask(FakeTrajectory(X, np.ones(3000)), mod, model, str(tmp_path), device=DEV, verbose=False,
                                debug_mode=False)
    cv = task.colvar_model()
    g, g64, env32 = _model_grads(cv, cv[1], ppt, X, seed=2)
    assert _rel(g, g64.to(DEV)) <= max(2e-5, env32)


def test_regautoencoder_colvar_and_reg_model_gradients(tmp_path):
    from colvarsfinder import core, nn, utils
    c = C.regae_case("regae_dipep_generator")
    model = nn.RegAutoEncoder(c["e_dims"], c["d_dims"], c["r_dims"], c["K"])
    for seq, params in [(model.encoder, c["enc"]), (model.decoder, c["dec"])] + [(model.reg[i], c["reg"][i]) for i in range(c["K"])]:
        with torch.no_grad():
            for p, v in zip(seq.parameters(), params):
                p.copy_(torch.as_tensor(v))
    pp = utils.Align(c["ref"], c["align_idx"])
    task = core.RegAutoEncoderTask(FakeTrajectory(c["X"], c["w"].astype(np.float64), dt=c["dt"]), pp, model, str(tmp_path),
                                   c["eig_w"], alpha=c["alpha"], gamma=c["gamma"], eta=c["eta"], lag_tau_ae=c["lag_tau_ae"],
                                   lag_tau_reg=c["lag_tau_reg"], beta=c["beta"], freeze_encoder=c["freeze"], device=DEV,
                                   verbose=False, debug_mode=False)
    ppt = ref_torch.Preprocess(ref_torch.Align(c["ref"], c["align_idx"]), None)
    X = np.asarray(c["X"], dtype=np.float32)
    for seed, cv in enumerate([task.colvar_model(), task.reg_model()]):
        g, g64, env32 = _model_grads(cv, cv[1], ppt, X, seed=seed)
        assert _rel(g, g64.to(DEV)) <= max(2e-5, env32), seed


def test_gradient_matches_exported_torchscript_model(tmp_path):
    """scripted_cv_gpu.pt (stock torch: SVD alignment, autograd) and the CUDA path give the same gradient: each is within the
    fp32 envelope of the fp64 gradient, so they are within twice that of each other."""
    c = dict(C.eigen_case("eigen_dipep_features"), diag_coeff=None)
    pp, _, ppt = _layer("features")
    task = _eigen_task(c, tmp_path, pp)
    task.save_model(0)
    scripted = torch.jit.load(os.path.join(str(tmp_path), "latest", "scripted_cv_gpu.pt"), map_location=DEV)
    cv = task.colvar_model()
    X = np.asarray(c["X"], dtype=np.float32)
    g, g64, env32 = _model_grads(cv, cv[1], ppt, X, seed=3)
    xs = torch.as_tensor(X, device=DEV).requires_grad_()
    out = scripted(xs)
    gs, = torch.autograd.grad(out, xs, torch.randn(out.shape, generator=torch.Generator().manual_seed(3)).to(DEV))
    env = max(2e-5, env32)
    assert _rel(g, g64.to(DEV)) <= env
    assert _rel(g, gs) <= 2 * max(env, _rel(gs, g64.to(DEV)))


# --------------------------------------------------------------------------------------------- 5. nothing else moved
@pytest.mark.parametrize("name", LAYERS)
def test_forward_unchanged_by_autograd(name):
    mod, _, _ = _layer(name)
    X = torch.as_tensor(_frames(1000, seed=8), device=DEV)
    plain = mod(X)
    recorded = mod(X.clone().requires_grad_())
    with torch.no_grad():
        off = mod(X.clone().requires_grad_())
    assert recorded.grad_fn is not None and plain.grad_fn is None and off.grad_fn is None
    assert torch.equal(plain, recorded) and torch.equal(plain, off)


@pytest.mark.parametrize("name", ["features", "unaligned"])
def test_atoms_no_record_reads_get_exact_zeros(name):
    mod, _, _ = _layer(name)
    B = 4099
    read = set(SUB if name == "features" else []) | {a for _, atoms in FEATS for a in atoms}
    unread = [a for a in range(22) if a not in read]
    assert unread
    x = torch.as_tensor(_frames(B, seed=2), device=DEV).requires_grad_()
    # leave NaN in the memory the caching allocator hands out for g_x: an unwritten entry would show
    torch.full((B, 22, 3), float("nan"), device=DEV)
    out = mod(x)
    g, = torch.autograd.grad(out, x, torch.randn_like(out))
    assert torch.isfinite(g).all()
    assert torch.equal(g[:, unread], torch.zeros_like(g[:, unread]))
    assert (g[:, sorted(read)].abs().sum((0, 2)) > 0).all()


@pytest.mark.parametrize("name,op", [("align", "align_vjp"), ("positions", "align_vjp"), ("features", "features_vjp"),
                                     ("unaligned", "features_vjp")])
def test_second_backward_raises(name, op):
    mod, _, _ = _layer(name)
    x = torch.as_tensor(_frames(64, seed=1), device=DEV).requires_grad_()
    out = mod(x)
    g, = torch.autograd.grad(out, x, torch.randn_like(out), create_graph=True)
    with pytest.raises(RuntimeError, match=f"cvf.{op}"):
        torch.autograd.grad((g * g).sum(), x)


def test_align_module_left_on_the_host_is_refused():
    """The kernels read the reference and the indices on the frames' device: a module that was not moved raises instead."""
    from colvarsfinder import utils
    al = utils.Align(BASE, ALL)
    x = torch.as_tensor(_frames(8, seed=1), device=DEV)
    for xx in (x, x.clone().requires_grad_()):
        with pytest.raises(RuntimeError, match="move the module"):
            al(xx)
    with pytest.raises(RuntimeError, match="move the module"):
        utils.Preprocessing(al, None)(x)


def test_opcheck_of_the_operators():
    from colvarsfinder import _ops, utils
    tests = ("test_schema", "test_autograd_registration", "test_faketensor")
    al = utils.Align(BASE[SUB], SUB).to(DEV)
    x = torch.as_tensor(_frames(200, seed=6), device=DEV)
    g_y = torch.randn_like(x)
    torch.library.opcheck(torch.ops.cvf.align_fwd.default, (x.clone().requires_grad_(), al.ref_pos, al.align_idx), test_utils=tests)
    torch.library.opcheck(torch.ops.cvf.align_vjp.default, (x, al.ref_pos, al.align_idx, g_y.requires_grad_()), test_utils=tests)
    spec = _ops.PreprocSpec(utils.Preprocessing(al, utils.FeatureMap(FEATS)), (22, 3), DEV, None)
    g_r = torch.randn(200, spec.d_r, device=DEV)
    torch.library.opcheck(torch.ops.cvf.features_fwd.default, (x.clone().requires_grad_(), spec.handle), test_utils=tests)
    torch.library.opcheck(torch.ops.cvf.features_vjp.default, (x, g_r.requires_grad_(), spec.handle), test_utils=tests)
