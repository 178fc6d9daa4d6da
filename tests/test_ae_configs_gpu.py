"""The autoencoder step on every kernel configuration a chain's shape selects, against an fp64 oracle.

AutoEncoderTask.weighted_MSE_loss and its backward (cvf_ae_step) run on one of eight configurations, chosen in
csrc/cvf_ae.cu (ae_plan, ae_path) from the chain's shape and the device's opt-in shared memory:
  * the thread-private kernels (cvf_ae_fast.cu) for exactly [d,20,20,20,e] + [e,10,10,d] (tests/test_gpu.py, test_step_at_scale);
  * the general row engine with F = 128, 64 or 32 frames per tile, at one or two CTAs per SM: the largest F whose state fits
    shared memory, or half of it at two CTAs per SM when two such CTAs fit one SM;
  * the layer-wise products (cvf_ae_wide.cu) for chains whose state does not fit shared memory at 32 frames, on tcgen05 with
    the 3 x TF32 split (cvf_gemm_tc.cu, default) or as fp32 SIMT products (cvf_ae_set_wide_path(1)).
Every case names its configuration, checks it with a mirror of ae_plan / ae_path and checks it again from the launch
accounting: the general kernel is one ae_step launch; the layer-wise path issues a known number of ae_step launches and one
reduce_partials launch per chunk for the loss sums plus one per layer per chunk for the gradient.

The oracle is the multiplicity construction of test_step_at_scale_gpu.py: a batch is X = D[idx] with M distinct standardised
frames D, so the fp64 closed form on D with the per-frame aggregated weights is the fp64 result of the whole batch at any B.
Tanh chains use oracle.closed_form.ae_loss_and_grads, other activations and a separate reconstruction target fp64 torch
autograd.  The bars are loss <= 1e-5 relative and every gradient tensor <= 2e-5 relative L2, or FLOOR_SLACK times the error
of torch's fp32 run of the same batch against fp64 where that is larger (SURVEY 7.3-D).  The floor matters for ill-conditioned
batches only:
one frame through a one-unit bottleneck whose value is a cancelling sum of 257 terms (128x257 at B = 1) loses up to 2.4e-4 of
the decoder's first weight gradient in torch's own fp32 run.  A single frame's error is one draw of the rounding, not an
average, so two summation orders can differ several-fold (there: 3.4e-5 on the tensor cores, 5.4e-6 in torch's fp32 run); the
floor is therefore scaled by FLOOR_SLACK.  Well-conditioned batches have floors near 1e-7, where the fixed bars rule.  On every
configuration the loss under torch.no_grad() equals the training loss bit for bit and two runs are bit-identical.
"""
import ctypes
import gc

import numpy as np
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_torch
from tests import _cases as C

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None
M = 2048                          # distinct frames behind every batch
CHUNK = 32768                     # frames per chunk of the layer-wise path (kChunkFrames in cvf_ae_wide.cu)
ACT_TANH = 1                      # CVF_ACT_TANH
E_WORKSPACE = -3                  # CVF_E_WORKSPACE
FLOOR_SLACK = 8.0                 # bars give way to this multiple of torch's fp32 error (module docstring)


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


def state_bytes(chain, F):
    """Shared memory of the general kernel at F frames per tile (ae_layout): the padded weights and biases, the loss partials,
    then rows of F + 4 floats for the weight and error rows, every activation A_0..A_L and every adjoint s_1..s_L."""
    L = len(chain) - 1
    params = sum(chain[l + 1] * _r4(chain[l]) + _r4(chain[l + 1]) for l in range(L))
    rows = 2 + sum(chain) + sum(chain[1:])
    return 4 * (_r4(params + 16) + rows * (F + 4))


def configuration(chain, cap):
    """("general", F, CTAs per SM) or ("layerwise", None, None), as ae_plan / ae_path choose them."""
    Fs = (128, 64, 32)
    fits = [c for c in range(3) if state_bytes(chain, Fs[c]) <= cap]
    if not fits:
        return ("layerwise", None, None)
    c = fits[0]
    if c < 2 and 2 * (state_bytes(chain, Fs[c + 1]) + 1024) <= 228 * 1024:
        return ("general", Fs[c + 1], 2)
    return ("general", Fs[c], 1)


def device_cap():
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# --------------------------------------------------------------------------------------------- models and oracle
ACT_MODULES = {"tanh": torch.nn.Tanh, "sigmoid": torch.nn.Sigmoid, "softplus": torch.nn.Softplus, "elu": torch.nn.ELU,
               "relu": torch.nn.ReLU}
ACT_FUNCS = {"tanh": torch.tanh, "sigmoid": torch.sigmoid, "softplus": torch.nn.functional.softplus,
             "elu": torch.nn.functional.elu, "relu": torch.relu}


def make_model(e_dims, d_dims, act, seed):
    """(model, AEContext, enc, dec): torch's default initialisation for a fixed seed, on the device."""
    from colvarsfinder import _ops, nn
    torch.manual_seed(seed)
    enc = [p.numpy() for p in ref_torch.init_mlp_params(e_dims)]
    dec = [p.numpy() for p in ref_torch.init_mlp_params(d_dims)]
    model = nn.AutoEncoder(e_dims, d_dims, ACT_MODULES[act]())
    with torch.no_grad():
        for p, v in zip(list(model.encoder.parameters()) + list(model.decoder.parameters()), enc + dec):
            p.copy_(torch.as_tensor(v))
    return model, _ops.AEContext(model, DEV), enc, dec


def frames(d, seed):
    return np.random.default_rng(seed).normal(size=(M, d)).astype(np.float32)


def torch_loss_and_grads(D, T, w, enc, dec, act, dtype):
    """Weighted reconstruction loss of the frames D against the targets T (None: D itself) and its parameter gradients, by
    torch autograd in `dtype`."""
    ps = [torch.tensor(np.asarray(p), dtype=dtype, requires_grad=True) for p in list(enc) + list(dec)]
    X = torch.as_tensor(D, dtype=dtype)
    Tt = X if T is None else torch.as_tensor(T, dtype=dtype)
    wt = torch.as_tensor(w, dtype=dtype)
    f = ACT_FUNCS[act]
    out = ref_torch.mlp(ps[len(enc):], ref_torch.mlp(ps[:len(enc)], X, f), f)
    loss = (wt * ((out - Tt) ** 2).sum(1)).sum() / wt.sum()
    loss.backward()
    return float(loss.detach()), [p.grad.numpy().astype(np.float64) for p in ps]


_ORACLE = {}


def oracle(key, D, w_agg, enc, dec, act, T=None):
    """(fp64 loss, fp64 gradients, loss floor, gradient floors), cached per case: both product modes of the layer-wise path
    run the same batch.  The floors are the relative errors of torch's fp32 run (frames with zero aggregated weight add exact
    zeros to it, so it is the fp32 run of the batch's distinct frames)."""
    if key not in _ORACLE:
        if act == "tanh" and T is None:
            lo, genc, gdec = cf.ae_loss_and_grads(D, w_agg, enc, dec)
            g64 = genc + gdec
        else:
            lo, g64 = torch_loss_and_grads(D.astype(np.float64), None if T is None else T.astype(np.float64), w_agg, enc, dec,
                                           act, torch.float64)
        l32, g32 = torch_loss_and_grads(D, T, w_agg.astype(np.float32), enc, dec, act, torch.float32)
        _ORACLE[key] = (lo, g64, abs(l32 - lo) / abs(lo), [C.rel_l2(a, b) for a, b in zip(g32, g64)])
    return _ORACLE[key]


def assert_matches(loss, grads, ref, tag):
    lo, g64, floor_loss, floors = ref
    e_loss = abs(float(loss) - lo) / abs(lo)
    errs = [C.rel_l2(g, go) for g, go in zip(grads, g64)]
    print(f"[{tag}] loss {e_loss:.1e}  grad rel-L2 max {max(errs):.1e} median {np.median(errs):.1e}  "
          f"(torch fp32: loss {floor_loss:.1e}, grad max {max(floors):.1e})")
    assert e_loss <= max(1e-5, FLOOR_SLACK * floor_loss), (tag, "loss", e_loss, floor_loss)
    for i, (e, f) in enumerate(zip(errs, floors)):
        assert e <= max(2e-5, FLOOR_SLACK * f), (tag, "gradient", i, errs, floors)


def step(model, actx, X, w, T=None):
    """Training loss, the parameter gradients and the launches of the step; then the loss under no_grad and its launches."""
    from colvarsfinder import _lib, _ops
    model.zero_grad(set_to_none=True)
    _lib.profile_read(reset=True)
    loss = _ops.ae_loss(actx, X, w, T)
    loss.backward()
    torch.cuda.synchronize()
    launched = _lib.profile_read(reset=True)
    grads = [p.grad.detach().clone() for p in list(model.encoder.parameters()) + list(model.decoder.parameters())]
    with torch.no_grad():
        loss_eval = _ops.ae_loss(actx, X, w, T)
    torch.cuda.synchronize()
    launched_eval = _lib.profile_read(reset=True)
    return dict(loss=loss.detach(), grads=grads, launched=launched, loss_eval=loss_eval, launched_eval=launched_eval)


def assert_repeatable(a, b, tag):
    assert torch.equal(a["loss_eval"], a["loss"]), (tag, "loss under no_grad differs from the training loss")
    assert torch.equal(a["loss"], b["loss"]), (tag, "loss differs between runs")
    for ga, gb in zip(a["grads"], b["grads"]):
        assert torch.equal(ga, gb), (tag, "gradients differ between runs")


def launches(launched, name):
    return launched[name][2]


def shape_tag(e_dims, d_dims):
    return "x".join(str(v) for v in e_dims) + "+" + "x".join(str(v) for v in d_dims[1:])


# --------------------------------------------------------------------------------------------- 1. general row engine
# layout -> shapes that take it on a 227 KB (232 448 B opt-in) part; the last F=32x1 chain is the widest [66,h,h,2] chain that
# still fits (231 328 B at 32 frames), h = 85 goes layer-wise
GENERAL = {
    (128, 1): [([30, 24, 24, 24, 2], [2, 24, 24, 24, 30]), ([30, 33, 33, 2], [2, 33, 33, 30])],
    (64, 2): [([30, 21, 21, 3], [3, 21, 21, 30]), ([30, 3], [3, 30])],
    (32, 2): [([66, 30, 30, 2], [2, 30, 30, 66]), ([12, 37, 37, 37, 1], [1, 37, 37, 37, 12])],
    (64, 1): [([66, 45, 45, 2], [2, 45, 45, 66]), ([71, 52, 52, 1], [1, 52, 52, 71])],
    (32, 1): [([66, 62, 62, 3], [3, 62, 62, 66]), ([500, 2], [2, 500]), ([66, 84, 84, 2], [2, 84, 84, 66])],
}
# one activation other than tanh per layout (index of the shape in GENERAL), and the layout's time-lagged target case (shape 0)
GENERAL_OTHER_ACT = {(128, 1): (1, "sigmoid"), (64, 2): (0, "softplus"), (32, 2): (0, "elu"), (64, 1): (0, "relu"),
                     (32, 1): (2, "sigmoid")}
BIG = "2gF+17"                    # two tiles per CTA of the full grid and a ragged tail: CTAs walk several tiles


def _general_batches(F):
    return [str(b) for b in sorted({1, 31, 33, F - 1, F + 1})] + [BIG]


def _general_params():
    out = []
    for (F, ctas), shapes in GENERAL.items():
        lay = f"F{F}x{ctas}"
        for i, (e, d) in enumerate(shapes):
            for b in _general_batches(F):
                out.append(pytest.param(lay, i, b, "tanh", False, id=f"{lay}-{shape_tag(e, d)}-B{b}-tanh"))
        i, act = GENERAL_OTHER_ACT[(F, ctas)]
        e, d = shapes[i]
        out.append(pytest.param(lay, i, BIG, act, False, id=f"{lay}-{shape_tag(e, d)}-B{BIG}-{act}"))
        e, d = shapes[0]
        out.append(pytest.param(lay, 0, BIG, "tanh", True, id=f"{lay}-{shape_tag(e, d)}-B{BIG}-tanh-target"))
    return out


@pytest.mark.parametrize("layout,shape,bname,act,target", _general_params())
def test_general_layout_matches_oracle(layout, shape, bname, act, target):
    """The general row engine (ae_kernel) in every tile layout, at ragged batch sizes around one tile and at two tiles per CTA
    of the full grid plus 17 frames; one other activation and one separate reconstruction target (cvf_ae_step_target, the
    features of other frames) per layout."""
    F, ctas = (int(v) for v in layout[1:].split("x"))
    e_dims, d_dims = GENERAL[(F, ctas)][shape]
    chain = e_dims + d_dims[1:]
    assert configuration(chain, device_cap()) == ("general", F, ctas), (layout, chain)
    grid = sm_count() * ctas
    B = 2 * grid * F + 17 if bname == BIG else int(bname)
    if bname == BIG:
        assert -(-B // F) > 2 * grid
    seed = 100 + 10 * sorted(GENERAL).index((F, ctas)) + shape
    model, actx, enc, dec = make_model(e_dims, d_dims, act, seed)
    D = frames(e_dims[0], seed)
    X, w, w_agg, idx = C.repeated_batch(D, B, seed + B, device=DEV)
    T_D, T = None, None
    if target:
        T_D = np.ascontiguousarray(D[np.random.default_rng(seed).permutation(M)])
        T = torch.as_tensor(T_D, device=DEV)[idx].contiguous()
    tag = f"{layout} {shape_tag(e_dims, d_dims)} B={B} {act}{' target' if target else ''}"
    first = step(model, actx, X, w, T)
    second = step(model, actx, X, w, T)
    for r in (first, second):
        assert launches(r["launched"], "ae_step") == 1 and launches(r["launched"], "ae_fast_main") == 0, (tag, r["launched"])
        assert launches(r["launched"], "reduce_partials") == 2 and launches(r["launched_eval"], "reduce_partials") == 1, tag
    assert_repeatable(first, second, tag)
    ref = oracle(("general", layout, shape, B, act, target), D, w_agg, enc, dec, act, T_D)
    assert_matches(first["loss"], [g.cpu().numpy() for g in first["grads"]], ref, tag)


# --------------------------------------------------------------------------------------------- 2. layer-wise products
# name -> (encoder, decoder, what the shape is for); d % 4 == 0 with an aligned pointer: the tensor-core path reads the input
# in place, otherwise it stages a padded copy
LAYERWISE = {
    "66x85": ([66, 85, 85, 2], [2, 85, 85, 66], "first chain past the general kernel; staged input; every width below 128"),
    "128x257": ([128, 257, 1], [1, 257, 128], "in place; input ones row in its own tile; K = 257; 1-column N tail; bottleneck 1"),
    "256x256": ([256, 256, 1], [1, 256, 256], "K = 256, one whole chain; hidden ones row in its own tile"),
    "129x255": ([129, 255, 33, 3], [3, 33, 255, 129], "tails of 1 past a tile and past a k-block"),
    "600x3": ([600, 3], [3, 600], "L = 2: no activation; in place; K = 600 is chains of 8 + 8 + 3 k-blocks"),
    "100x130L8": ([100, 130, 130, 130, 1], [1, 130, 130, 130, 100], "L = 8"),
}
LAYERWISE_B = [1, 31, 129, 4099, 32768, 32769, 65665]


def layerwise_launches(L, chunks, grad, tc, in_place):
    """ae_step launches of cvf_ae_wide.cu for a chain of L layers over `chunks` chunks."""
    n = L + (1 if grad else 0)                       # padded weight copies; zeroed gradient
    if tc:
        n += L + (L - 1 if grad else 0)              # weight images of the forward and back-propagation products
    per = L                                          # forward products
    if tc:
        per += (0 if in_place else 1) + 1 + (1 if grad else 0)    # staged input; its K-major and transposed images
    else:
        per += 1 + (L - 1) + 1                       # staged input; ones column of the hidden buffers; loss kernel
    if grad:
        per += 2 * L - 1                             # weight-gradient and back-propagation products
    return n + chunks * per


def _set_wide_path(mode):
    from colvarsfinder import _lib
    _lib.check(_lib.lib().cvf_ae_set_wide_path(mode), "cvf_ae_set_wide_path")


@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("B", LAYERWISE_B)
@pytest.mark.parametrize("name", list(LAYERWISE))
def test_layerwise_matches_oracle(name, B, mode):
    """The layer-wise path in both product modes over one to three chunks (32 768, 32 768 and 129 frames at B = 65 665: split-K
    of the weight gradients with a short last split).  On the shapes the tensor-core path reads in place, the same batch also
    runs as a misaligned contiguous view: it takes the staged route (one more launch per chunk) and gives bit-identical
    results in tensor-core mode."""
    e_dims, d_dims, _ = LAYERWISE[name]
    chain = e_dims + d_dims[1:]
    L, d = len(chain) - 1, chain[0]
    assert configuration(chain, device_cap())[0] == "layerwise", chain
    tc = mode == "tc"
    in_place = tc and d % 4 == 0
    seed = 300 + list(LAYERWISE).index(name)
    model, actx, enc, dec = make_model(e_dims, d_dims, "tanh", seed)
    D = frames(d, seed)
    X, w, w_agg, _ = C.repeated_batch(D, B, seed + B, device=DEV)
    assert X.data_ptr() % 16 == 0
    chunks = -(-B // CHUNK)
    tag = f"layerwise-{mode} {shape_tag(e_dims, d_dims)} B={B}"
    _set_wide_path(0 if tc else 1)
    try:
        first = step(model, actx, X, w)
        second = step(model, actx, X, w)
        mis = None
        if in_place:
            Xm = torch.empty(B * d + 1, dtype=torch.float32, device=DEV)[1:].view(B, d)
            Xm.copy_(X)
            assert Xm.is_contiguous() and Xm.data_ptr() % 16 != 0
            mis = step(model, actx, Xm, w)
    finally:
        _set_wide_path(0)
    for r in (first, second):
        assert launches(r["launched"], "ae_step") == layerwise_launches(L, chunks, True, tc, in_place), (tag, r["launched"])
        assert launches(r["launched_eval"], "ae_step") == layerwise_launches(L, chunks, False, tc, in_place), tag
        assert launches(r["launched"], "reduce_partials") == chunks * (1 + L), (tag, r["launched"])
        assert launches(r["launched_eval"], "reduce_partials") == chunks, tag
        assert launches(r["launched"], "ae_fast_main") == 0, tag
    assert_repeatable(first, second, tag)
    if mis is not None:
        assert launches(mis["launched"], "ae_step") == layerwise_launches(L, chunks, True, tc, False), (tag, mis["launched"])
        assert_repeatable(first, mis, tag + " misaligned view")
    ref = oracle(("layerwise", name, B), D, w_agg, enc, dec, "tanh")
    assert_matches(first["loss"], [g.cpu().numpy() for g in first["grads"]], ref, tag)


def _c_step(chain, params, X, w, ws, ws_bytes, grad):
    from colvarsfinder import _lib
    L = len(chain) - 1
    half = L // 2
    acts = [ACT_TANH] * (half - 1) + [0] + [ACT_TANH] * (L - half - 1) + [0]
    net = _lib.make_mlp(chain, acts)
    sums = torch.zeros(2, dtype=torch.float64, device=DEV)
    rc = _lib.lib().cvf_ae_step(X.data_ptr(), w.data_ptr(), X.shape[0], ctypes.byref(net), params.data_ptr(), sums.data_ptr(),
                                None if grad is None else grad.data_ptr(), ws, ws_bytes, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, sums


def _workspace_bytes(chain, B):
    from colvarsfinder import _lib
    L = len(chain) - 1
    acts = [ACT_TANH] * (L // 2 - 1) + [0] + [ACT_TANH] * (L - L // 2 - 1) + [0]
    return int(_lib.lib().cvf_ae_workspace_bytes(ctypes.byref(_lib.make_mlp(chain, acts)), B))


@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("B,chunk", [(1000, 128), (385, 128), (1000, 384), (385, 384)])
def test_layerwise_small_workspace_chunks(B, chunk, mode):
    """cvf_ae_step through the C ABI with the workspace cvf_ae_workspace_bytes gives for `chunk` frames: the path works in
    chunks of that many frames (B = 385 leaves a last chunk of one frame), and the result matches the oracle."""
    from colvarsfinder import _lib
    e_dims, d_dims, _ = LAYERWISE["128x257"]
    chain = e_dims + d_dims[1:]
    L = len(chain) - 1
    seed = 400 + B
    torch.manual_seed(seed)
    enc = [p.numpy() for p in ref_torch.init_mlp_params(e_dims)]
    dec = [p.numpy() for p in ref_torch.init_mlp_params(d_dims)]
    params = torch.cat([torch.as_tensor(p).reshape(-1) for p in enc + dec]).to(DEV)
    D = frames(chain[0], seed)
    X, w, w_agg, _ = C.repeated_batch(D, B, seed, device=DEV)
    ws_bytes = _workspace_bytes(chain, chunk)
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    grad = torch.zeros(params.numel(), dtype=torch.float64, device=DEV)
    chunks = -(-B // chunk)
    tag = f"layerwise-{mode} {shape_tag(e_dims, d_dims)} B={B} chunks of {chunk}"
    _set_wide_path(0 if mode == "tc" else 1)
    try:
        _lib.profile_read(reset=True)
        rc, sums = _c_step(chain, params, X, w, ws.data_ptr(), ws_bytes, grad)
        launched = _lib.profile_read(reset=True)
    finally:
        _set_wide_path(0)
    _lib.check(rc, "cvf_ae_step")
    assert launches(launched, "reduce_partials") == chunks * (1 + L), (tag, launched)
    assert launches(launched, "ae_step") == layerwise_launches(L, chunks, True, mode == "tc", mode == "tc"), (tag, launched)
    s = sums.cpu().numpy()
    g = grad.cpu().numpy() / s[1]
    sizes = np.cumsum([0] + [p.size for p in enc + dec])
    grads = [g[sizes[i]:sizes[i + 1]].reshape(p.shape) for i, p in enumerate(enc + dec)]
    assert_matches(s[0] / s[1], grads, oracle(("c-abi", B), D, w_agg, enc, dec, "tanh"), tag)


def test_layerwise_workspace_too_small_for_one_chunk():
    """A workspace that leaves no room for a 128-frame chunk is refused with CVF_E_WORKSPACE and its message, and nothing is
    launched."""
    from colvarsfinder import _lib
    e_dims, d_dims, _ = LAYERWISE["128x257"]
    chain = e_dims + d_dims[1:]
    per_frame = (_workspace_bytes(chain, 256) - _workspace_bytes(chain, 128)) // 128
    ws_bytes = _workspace_bytes(chain, 128) - 64 * per_frame
    torch.manual_seed(5)
    params = torch.cat([p.reshape(-1) for p in ref_torch.init_mlp_params(e_dims) + ref_torch.init_mlp_params(d_dims)]).to(DEV)
    X = torch.randn(300, chain[0], device=DEV)
    w = torch.ones(300, device=DEV)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    grad = torch.zeros(params.numel(), dtype=torch.float64, device=DEV)
    _lib.profile_read(reset=True)
    rc, _ = _c_step(chain, params, X, w, ws.data_ptr(), ws_bytes, grad)
    launched = _lib.profile_read(reset=True)
    assert rc == E_WORKSPACE
    assert "128-frame chunk" in _lib.lib().cvf_last_error_string().decode()
    assert sum(v[2] for v in launched.values()) == 0, launched


# --------------------------------------------------------------------------------------------- 3. refusals
def test_layerwise_refuses_other_activations():
    """A chain too wide for shared memory with ReLU: the layer-wise path takes tanh only, and says so."""
    from colvarsfinder import _ops
    e_dims, d_dims, _ = LAYERWISE["66x85"]
    assert configuration(e_dims + d_dims[1:], device_cap())[0] == "layerwise"
    _, actx, _, _ = make_model(e_dims, d_dims, "relu", 7)
    X = torch.randn(64, e_dims[0], device=DEV)
    with pytest.raises(RuntimeError, match="tanh only"):
        _ops.ae_loss(actx, X, torch.ones(64, device=DEV))


def test_layerwise_refuses_separate_target():
    """A separate reconstruction target on a chain too wide for shared memory raises the cvf_ae_step_target error and launches
    nothing, instead of returning a number."""
    from colvarsfinder import _lib, _ops
    e_dims, d_dims, _ = LAYERWISE["66x85"]
    _, actx, _, _ = make_model(e_dims, d_dims, "tanh", 8)
    X = torch.randn(64, e_dims[0], device=DEV)
    T = torch.randn(64, e_dims[0], device=DEV)
    _ops.ae_loss(actx, X, torch.ones(64, device=DEV))          # the workspace exists: only the target is refused below
    torch.cuda.synchronize()
    _lib.profile_read(reset=True)
    with pytest.raises(RuntimeError, match="cvf_ae_step_target: a separate reconstruction target"):
        _ops.ae_loss(actx, X, torch.ones(64, device=DEV), target=T)
    assert launches(_lib.profile_read(reset=True), "ae_step") == 0
