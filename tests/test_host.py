"""CPU-side checks: the shared library exports the C ABI, the per-frame geometry header agrees with the oracle,
host-side descriptors / flat parameter storage / split logic behave like the reference."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    return g


def test_library_exports_every_declared_symbol(built):
    from colvarsfinder import _lib
    header = open(os.path.join(ROOT, "include", "cvf.h")).read()
    declared = set(re.findall(r"\b(cvf_[a-z_0-9]+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name)
    assert lib.cvf_version() == 100
    assert lib.cvf_eigen_num_stats(3) == 1 + 6 + 9 and lib.cvf_eigen_num_combine(3) == 3 + 15 + 9
    m = _lib.make_mlp([66, 20, 20, 20, 1], [1, 1, 1, 0])
    assert lib.cvf_mlp_param_count(C.byref(m)) == 2201
    ae = _lib.make_mlp([66, 20, 2, 20, 66], [1, 0, 1, 0])
    assert lib.cvf_ae_workspace_bytes(C.byref(ae), 1000) > 0
    wide = _lib.make_mlp([3000, 512, 512, 2, 512, 512, 3000], [1, 1, 0, 1, 1, 0])      # layer-wise path: needs room for a chunk
    assert lib.cvf_ae_workspace_bytes(C.byref(wide), 1000) > 1000 * 4 * (3000 + 512 + 512 + 2 + 512 + 512 + 3000)
    assert lib.cvf_ae_workspace_bytes(C.byref(m), 1000) == 0                            # not an R^d -> R^d chain


def test_sass_is_sm100_with_bulk_copies(built):
    cuobjdump = os.path.join(os.path.dirname(built.NVCC), "cuobjdump")      # the toolkit that built the library, not PATH's
    out = subprocess.run([cuobjdump, "-sass", os.path.join(ROOT, "colvars-finder_b200", "colvarsfinder", "libcvf_sm100.so")],
                         capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UBLKCP" in out          # cp.async.bulk (TMA 1-D) in the alignment kernel
    assert "FFMA" in out


def _hostlib(built):
    return C.CDLL(os.path.join(ROOT, "oracle", "_build", "libcvf_hostmath.so"))


def test_rotation_matches_svd_kabsch(built):
    """cvf_rotation (Horn + Jacobi fp32 + Newton fp64) vs numpy SVD Kabsch, incl. reflection-prone frames."""
    h = _hostlib(built)
    base = ref_torch.DIPEPTIDE_NM * 10
    X = ref_torch.synth_frames(base, 4000, seed=5, noise_sd=0.5).astype(np.float64)
    idx = list(range(22))
    y, R, c, Kinv, refc = cf.kabsch(X, idx, base)
    Hm = np.ascontiguousarray(np.einsum("bna,nc->bac", X[:, idx] - c, refc))
    Rf = np.zeros((len(X), 9), np.float32)
    Kf = np.zeros((len(X), 6), np.float32)
    h.host_rotation(Hm.ctypes.data_as(C.c_void_p), len(X), Rf.ctypes.data_as(C.c_void_p), Kf.ctypes.data_as(C.c_void_p))
    Rf = Rf.reshape(-1, 3, 3)
    assert np.abs(Rf - R).max() < 2e-7            # float32 rounding of the stored matrix
    np.testing.assert_allclose(np.linalg.det(Rf.astype(np.float64)), 1.0, atol=1e-6)
    Kfull = np.stack([Kf[:, 0], Kf[:, 1], Kf[:, 2], Kf[:, 1], Kf[:, 3], Kf[:, 4], Kf[:, 2], Kf[:, 4], Kf[:, 5]], 1).reshape(-1, 3, 3)
    assert np.abs(Kfull - Kinv).max() / np.abs(Kinv).max() < 1e-6
    # nearly planar / noisy small subset: det fix must give a proper rotation that still matches
    sub = [1, 4, 6, 8]
    y2, R2, c2, _, ref2 = cf.kabsch(X[:500], sub, base[sub])
    H2 = np.ascontiguousarray(np.einsum("bna,nc->bac", X[:500, sub] - c2, ref2))
    Rg = np.zeros((500, 9), np.float32)
    Kg = np.zeros((500, 6), np.float32)
    h.host_rotation(H2.ctypes.data_as(C.c_void_p), 500, Rg.ctypes.data_as(C.c_void_p), Kg.ctypes.data_as(C.c_void_p))
    assert np.abs(Rg.reshape(-1, 3, 3) - R2).max() < 5e-6


def test_feature_stencils_match_oracle(built):
    h = _hostlib(built)
    rng = np.random.default_rng(3)
    p = rng.normal(size=(256, 4, 3)).astype(np.float32)
    cs = np.zeros((256, 2), np.float32)
    g = np.zeros((256, 4, 3), np.float32)
    h.host_dihedral(p.ctypes.data_as(C.c_void_p), 256, cs.ctypes.data_as(C.c_void_p), g.ctypes.data_as(C.c_void_p))
    vals, grads = cf.feature_stencil(p.astype(np.float64), "dihedral", [0, 1, 2, 3])
    np.testing.assert_allclose(cs, vals, atol=2e-5)
    gphi = -vals[:, 1, None, None] * grads[0] + vals[:, 0, None, None] * grads[1]      # d phi = -sin dcos + cos dsin
    assert np.abs(g - gphi).max() / np.abs(gphi).max() < 1e-4
    q = rng.normal(size=(256, 3, 3)).astype(np.float32)
    ca = np.zeros(256, np.float32)
    ga = np.zeros((256, 2, 3), np.float32)
    h.host_angle(q.ctypes.data_as(C.c_void_p), 256, ca.ctypes.data_as(C.c_void_p), ga.ctypes.data_as(C.c_void_p))
    vals, grads = cf.feature_stencil(q.astype(np.float64), "angle", [0, 1, 2])
    np.testing.assert_allclose(ca, vals[:, 0], atol=1e-5)
    np.testing.assert_allclose(ga[:, 0], grads[0][:, 0], atol=1e-4)
    np.testing.assert_allclose(ga[:, 1], grads[0][:, 2], atol=1e-4)


def test_nn_layout_matches_reference_state_dict():
    from colvarsfinder import nn
    torch.manual_seed(3)
    m = nn.EigenFunctions([5, 7, 7, 1], 2)
    keys = list(m.state_dict().keys())
    assert keys[:4] == ["eigen_funcs.0.1.weight", "eigen_funcs.0.1.bias", "eigen_funcs.0.2.weight", "eigen_funcs.0.2.bias"]
    assert list(m.eigen_funcs[0]._modules.keys()) == ["1", "activation 1", "2", "activation 2", "3"]
    assert nn.chain_spec(m.eigen_funcs[0])[:2] == ([5, 7, 7, 1], [True, True, False])
    ae = nn.AutoEncoder([6, 4, 2], [2, 4, 6])
    assert "encoder.2.bias" in ae.state_dict() and "decoder.1.weight" in ae.state_dict() and ae.encoded_dim == 2
    names = [n for n, _ in ae.get_params_of_cv(1)]
    assert names == ["1.weight", "1.bias", "2.weight", "2.bias"] and ae.get_params_of_cv(1)[2][1].shape == (1, 4)
    with pytest.raises(AssertionError):
        nn.EigenFunctions([5, 3, 2], 1)
    with pytest.raises(AssertionError):
        nn.AutoEncoder([6, 2], [3, 6])
    with pytest.raises(AssertionError):
        nn.create_sequential_nn([4])
    # same seed -> same initial weights as a chain of torch.nn.Linear built in the same order (reference nn.py:54-57,272)
    torch.manual_seed(3)
    ref = ref_torch.init_mlp_params([5, 7, 7, 1])
    for a, b in zip(ref, list(m.eigen_funcs[0].parameters())):
        assert torch.equal(a, b.detach())


def test_regautoencoder_layout_matches_reference():
    """nn.RegAutoEncoder / nn.RegModel (reference nn.py:116-239): state_dict keys, attributes, forward shapes, assertions."""
    from colvarsfinder import nn
    torch.manual_seed(5)
    m = nn.RegAutoEncoder([4, 6, 2], [2, 6, 4], [2, 5, 1], 3)
    keys = list(m.state_dict().keys())
    assert keys[0] == "encoder.1.weight" and "decoder.2.bias" in keys and "reg.2.2.weight" in keys
    assert m.num_reg == 3 and m.encoded_dim == 2 and len(m.reg) == 3
    x = torch.randn(7, 4)
    assert m.forward_ae(x).shape == (7, 4) and m.forward_reg(x).shape == (7, 3) and m(x).shape == (7, 7)
    assert [n for n, _ in m.get_params_of_cv(1)] == ["1.weight", "1.bias", "2.weight", "2.bias"]
    rm = nn.RegModel(m, [2, 0, 1])
    assert torch.equal(rm(x), m.forward_reg(x)[:, [2, 0, 1]])
    assert nn.RegAutoEncoder([4, 2], [2, 4], [2, 1], 0).reg is None
    with pytest.raises(AssertionError):
        nn.RegAutoEncoder([4, 2], [2, 4], [3, 1], 1)
    with pytest.raises(AssertionError):
        nn.RegModel(m, [0, 0, 1])
    # same construction order -> same init stream as the reference class: its initial weights under the same seed are
    # stored in tests/golden/train_regae_2d.npz (oracle/gen_golden_regae.py)
    from tests import _cases
    d = _cases.load("train_regae_2d")
    torch.manual_seed(13)
    r = nn.RegAutoEncoder([2, 20, 20, 20, 1], [1, 20, 20, 2], [1, 20, 20, 1], 1)
    params = list(r.parameters())
    assert len(params) == len([k for k in d if k.startswith("init_")])
    for j, p in enumerate(params):
        np.testing.assert_array_equal(p.detach().numpy(), d[f"init_{j}"])


def test_custom_operators_are_registered():
    """The step is exposed as torch.library operators (namespace cvf) with fake kernels and autograd formulas."""
    from colvarsfinder import _ops  # noqa: F401
    for name in ("eigen_stats", "eigen_grad", "eigen_combine", "eigen_loss", "eigen_tlag_sx", "eigen_tlag_seed", "eigen_tlag_combine", "ae_sums",
                 "align_fwd"):
        assert hasattr(torch.ops.cvf, name), name
    schema = str(torch.ops.cvf.eigen_stats.default._schema)
    assert schema.startswith("cvf::eigen_stats(Tensor X, Tensor w, Tensor params, SymInt handle, SymInt slot) -> (Tensor, Tensor)")
    with pytest.raises(RuntimeError, match="no longer exists"):
        _ops._context(10 ** 9)


def test_device_default_is_the_references_and_raises_clearly(tmp_path):
    """Signature default device=cpu as in the reference (core.py:311,621,797); without a CUDA device the constructor says so."""
    import inspect
    from colvarsfinder import core
    for cls in (core.EigenFunctionTask, core.AutoEncoderTask, core.RegAutoEncoderTask):
        assert inspect.signature(cls.__init__).parameters["device"].default == torch.device("cpu")


def test_flat_params_alias_module_parameters():
    from colvarsfinder import _ops, nn
    m = nn.EigenFunctions([3, 4, 1], 2)
    before = [p.detach().clone() for p in m.parameters()]
    fp = _ops.FlatParams(list(m.eigen_funcs), "cpu")
    assert fp.n == 2 * (3 * 4 + 4 + 4 + 1)
    for p, b in zip(m.parameters(), before):
        assert torch.equal(p.detach(), b)
    with torch.no_grad():
        fp.flat.mul_(2.0)
    for p, b in zip(m.parameters(), before):
        assert torch.equal(p.detach(), 2 * b)
    opt = torch.optim.SGD(m.parameters(), lr=1.0)
    for p in m.parameters():
        p.grad = torch.ones_like(p)
    opt.step()
    assert torch.allclose(fp.flat, torch.cat([(2 * b - 1).reshape(-1) for b in before]))
    m.to(torch.float64)         # breaks the aliasing ...
    m.to(torch.float32)
    fp.check()                  # ... and check() restores it
    assert all(p.data.data_ptr() == fp.flat.data_ptr() + 4 * off for p, off in zip(fp.params, fp.offsets))


def test_preproc_descriptor_lowering():
    from colvarsfinder import _lib, _ops, utils
    base = ref_torch.DIPEPTIDE_NM * 10
    al = utils.Align(base, list(range(22)))
    s = _ops.PreprocSpec(al, (22, 3), "cpu", None)
    assert (s.struct.kind, s.struct.n_used, s.struct.n_align, s.struct.d_r, s.struct.positions_only) == (1, 22, 22, 66, 1)
    assert abs(float(al.ref_pos.sum())) < 1e-4                    # centred reference (main.ipynb:305-328)
    heavy = [1, 4, 5, 6, 8, 10, 14, 15, 16, 18]
    fm = utils.FeatureMap([("dihedral", [4, 6, 8, 14]), ("bond", [1, 4]), ("position", [8, 10])])
    pp = utils.Preprocessing(utils.Align(base[heavy], heavy), fm)
    s = _ops.PreprocSpec(pp, (22, 3), "cpu", torch.arange(66, dtype=torch.float32) + 2)
    used = s._keep[0].tolist()
    assert used[:7] == [4, 6, 8, 14, 1, 10, 5] and sorted(used) == sorted(set(heavy) | {4, 6, 8, 14, 1, 10})
    assert s.struct.positions_only == 0 and s.struct.d_r == 2 + 1 + 6 and s.struct.n_feat == 4
    assert fm.output_dimension() == 9
    diag = s._keep[-1].reshape(-1, 3)
    assert diag[0].tolist() == [2 + 12, 2 + 13, 2 + 14]           # atom 4 -> coordinates 12..14
    s0 = _ops.PreprocSpec(torch.nn.Identity(), (2,), "cpu", None)
    assert (s0.struct.kind, s0.struct.dim) == (0, 2)
    with pytest.raises(RuntimeError):
        _ops.PreprocSpec(torch.nn.Linear(2, 2), (2,), "cpu", None)
    with pytest.raises(ValueError):
        utils.FeatureMap([("bond", [1, 2, 3])])

    class AG:
        def __init__(self, ix, pos):
            self.ix, self.positions = np.asarray(ix), np.asarray(pos)
    a2 = utils.Align.from_atom_groups(AG([10, 12, 14], base[:3]), AG([8, 10, 12, 14], base[:4]))
    assert a2.align_idx.tolist() == [1, 2, 3]


def test_tasks_refuse_cpu_and_unsupported_configs(tmp_path):
    from colvarsfinder import core, nn
    from oracle.ref_import import FakeTrajectory
    traj = FakeTrajectory(np.zeros((10, 2)), np.ones(10), dt=0.1)
    with pytest.raises(RuntimeError, match="cuda"):
        core.EigenFunctionTask(traj, torch.nn.Identity(), nn.EigenFunctions([2, 4, 1], 1), str(tmp_path), 1.0, [1.0],
                               device=torch.device("cpu"), verbose=False)
    with pytest.raises(RuntimeError, match="Tanh"):
        nn.chain_spec(nn.create_sequential_nn([2, 3, 1], torch.nn.GELU()))
    with pytest.raises(RuntimeError, match="Tanh"):
        nn.chain_spec(nn.create_sequential_nn([2, 3, 1], torch.nn.ELU(alpha=0.5)))
    assert nn.chain_spec(nn.create_sequential_nn([2, 3, 3, 1], torch.nn.Softplus()))[1] == [3, 3, 0]


def test_weighted_trajectory_text_and_weights(tmp_path):
    from colvarsfinder.utils import WeightedTrajectory
    t = np.arange(6) * 0.5
    data = np.column_stack([t, np.arange(6), -np.arange(6)])
    np.savetxt(tmp_path / "traj.txt", data)
    np.savetxt(tmp_path / "w.txt", np.array([1.0, 2.0, 3.0, 4.0, 50.0, 0.0]))
    wt = WeightedTrajectory(traj_filename=str(tmp_path / "traj.txt"), verbose=False)
    assert wt.trajectory.shape == (6, 2) and wt.dt == 0.5 and wt.n_frames == 6 and np.all(wt.weights == 1)
    wt = WeightedTrajectory(traj_filename=str(tmp_path / "traj.txt"), weight_filename=str(tmp_path / "w.txt"), min_w=0.05,
                            max_w=4.0, verbose=False)
    assert wt.trajectory.shape == (4, 2) and abs(wt.weights.mean() - 1) < 1e-12
    np.testing.assert_allclose(wt.weights, np.array([1, 2, 3, 4]) / 2.5)
    with pytest.raises(FileNotFoundError):
        WeightedTrajectory(traj_filename=str(tmp_path / "nope.txt"))
    np.savetxt(tmp_path / "w2.txt", np.ones(3))
    with pytest.raises(ValueError):
        WeightedTrajectory(traj_filename=str(tmp_path / "traj.txt"), weight_filename=str(tmp_path / "w2.txt"), verbose=False)


def test_shard_ranges_cover_everything():
    from colvarsfinder import _ops
    for n, w in [(10, 1), (10, 3), (7, 8), (1 << 23, 8)]:
        spans = [_ops.shard_range(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


def test_scriptable_preprocessing_matches_oracle_and_round_trips(tmp_path):
    """utils.scriptable(): the stock-torch restatement of Align / FeatureMap / Preprocessing that save_model exports
    (reference core.py:212-227) agrees with the oracle's pre-processing layer and survives torch.jit.script + save + load."""
    import torch
    from colvarsfinder import utils
    from oracle import ref_torch
    base = ref_torch.DIPEPTIDE_NM * 10.0
    heavy = [1, 4, 5, 6, 8, 10, 14, 15, 16, 18]
    feats = [("bond", [1, 4]), ("position", [4, 8]), ("angle", [4, 6, 8]), ("dihedral", [4, 6, 8, 14]), ("bond", [10, 18]),
             ("dihedral", [6, 8, 14, 16])]
    X = torch.as_tensor(ref_torch.synth_frames(base, 64, seed=5))
    cases = [
        (utils.Align(base, list(range(22))), ref_torch.Preprocess(ref_torch.Align(base, list(range(22))), None)),
        (utils.Preprocessing(utils.Align(base[heavy], heavy), utils.FeatureMap(feats)),
         ref_torch.Preprocess(ref_torch.Align(base[heavy], heavy), ref_torch.FeatureMap(feats))),
        (utils.FeatureMap(feats), ref_torch.Preprocess(None, ref_torch.FeatureMap(feats))),
    ]
    for i, (pp, oracle_pp) in enumerate(cases):
        mod = utils.scriptable(pp)
        want = oracle_pp(X.double()).float()
        got = mod(X)
        assert got.shape == want.shape
        assert torch.allclose(got, want, atol=2e-5, rtol=1e-5), (i, (got - want).abs().max())
        path = str(tmp_path / f"pp{i}.pt")
        torch.jit.script(mod).save(path)
        again = torch.jit.load(path)(X)
        assert torch.equal(again, got)
    ident = torch.nn.Identity()
    assert utils.scriptable(ident) is ident


def test_calc_weights_matches_reference_golden(tmp_path, capsys):
    """utils.calc_weights against the weights file the unmodified reference wrote for the same CSV (oracle/gen_golden_weights.py)."""
    import os
    from colvarsfinder import utils
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "calc_weights.npz"))
    csv = tmp_path / "state.csv"
    with open(csv, "w") as f:
        f.write('#"Time (ps)","Potential Energy (kJ/mole)","Total Energy (kJ/mole)"\n')
        for t, a, b in zip(g["time"], g["pot"], g["tot"]):
            f.write(f"{float(t)!r},{float(a)!r},{float(b)!r}\n")
    for tag in ("a", "b"):
        b_sim, b_sys, col = g[f"args_{tag}"]
        out = tmp_path / f"w_{tag}.txt"
        utils.calc_weights(str(csv), float(b_sim), float(b_sys), traj_weight_filename=str(out), energy_col_idx=int(col))
        got = np.loadtxt(out)
        np.testing.assert_allclose(got, g[f"weights_{tag}"], rtol=1e-12, atol=0)
        assert abs(got.mean() - 1.0) < 1e-12
    assert "Calculate Weights" in capsys.readouterr().out


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the GPU arm): exactly one JSON line on stdout with the
    contract's keys, produced without a GPU."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-frames", "2000"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train-step frames/sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("C3")
