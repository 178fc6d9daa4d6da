"""Trajectory holder and the pre-processing layers r(x) of the B200 training step.

* ``WeightedTrajectory`` -- same contract as the reference's holder (reference utils.py:62-169): ``trajectory``
  ([n,N,3] from an MDAnalysis-like universe or [n,d] from a text file), ``weights`` (mean 1, optionally
  filtered to (min_w, max_w)), ``dt``, ``n_frames``.  Host side only.
* ``Align`` / ``FeatureMap`` / ``Preprocessing`` -- the alignment + feature layer the reference borrows from
  the third-party ``molann`` package (examples/dipeptide/main.ipynb:335-348).  Here they are descriptors:
  the task classes lower them into ``cvf_preproc`` and the CUDA kernels evaluate alignment, features and
  their (transpose-)Jacobians; calling the modules directly runs the stand-alone CUDA pre-pass
  (``cvf_align_fwd`` / ``cvf_features_fwd``), whose autograd backward is ``cvf_align_vjp`` / ``cvf_features_vjp`` (first
  order: ``torch.autograd.grad(cv(x).sum(), x)`` works through ``colvar_model()``).  The integrators / weight calculators of
  the reference's utils.py (data generation) are outside this package's scope.
"""
from __future__ import annotations

import os

import numpy as np
import torch
from typing import List

from . import _lib

_FEATURE_TYPES = {"position": (_lib.FEAT_POSITION, None, 3), "bond": (_lib.FEAT_BOND, 2, 1),
                  "angle": (_lib.FEAT_ANGLE, 3, 1), "dihedral": (_lib.FEAT_DIHEDRAL, 4, 2)}


class WeightedTrajectory:
    """Trajectory data + statistical weights (reference utils.py:62-169)."""

    def __init__(self, universe=None, input_ag=None, traj_filename=None, weight_filename=None, min_w=0.0,
                 max_w=float("inf"), verbose=True, device=None):
        """``device`` (an addition to the reference's signature): a CUDA device on which the weights are normalised, the states
        selected and the trajectory gathered (``cvf_weights_filter``); ``trajectory`` / ``weights`` are then device tensors, which
        the task classes take as they are.  None keeps the reference's host-side numpy arrays."""
        if universe is not None:
            ix = universe.atoms.ix if input_ag is None else input_ag.ix
            self.trajectory = universe.trajectory.timeseries(order='fac')[:, ix, :]
            self.n_frames = universe.trajectory.n_frames
            self.dt = universe.trajectory.dt * 1e-3          # ps -> ns
            if verbose:
                print('\nTrajectory Info:\n  no. of frames in trajectory data: {}\n  stepsize: {:.1f}ps\n'
                      '  shape of trajectory data array: {}\n'.format(self.n_frames, universe.trajectory.dt,
                                                                       self.trajectory.shape))
        else:
            if traj_filename is None or not os.path.exists(traj_filename):
                raise FileNotFoundError('trajectory file not found')
            block = np.loadtxt(traj_filename)                  # column 0: time, the rest: state
            self.n_frames = block.shape[0]
            self.trajectory = block[:, 1:]
            self.dt = block[1, 0] - block[0, 0]
        if weight_filename:
            import pandas as pd
            w = pd.read_csv(weight_filename, usecols=[0], header=None)[0].to_numpy(dtype=np.float64)
            if verbose:   # the reference's summary of the normalised weights (utils.py:147-149)
                print('\nloading weights from file: ', weight_filename)
                print('\nWeights:\n', pd.Series(w / w.mean()).describe(percentiles=[0.2, 0.4, 0.6, 0.8]))
            if self.n_frames != len(w):
                raise ValueError('length in weight file does match the trajectory data!\n')
            if device is not None:
                idx, self.weights = filter_weights(torch.as_tensor(w, device=device), min_w, max_w)
                self.trajectory = torch.as_tensor(self.trajectory, device=device).index_select(0, idx)
            else:
                w = w / w.mean()
                keep = (w > min_w) & (w < max_w)
                self.trajectory = self.trajectory[keep, ...]
                w = w[keep]
                self.weights = w / w.mean()
            if verbose:   # utils.py:160-165
                print('\nAfter selecting states whose weights are in [{:.3e}, {:.3e}] and renormalization:\n'
                      '\nShape of trajectory: {}'.format(min_w, max_w, tuple(self.trajectory.shape)))
                w_sel = self.weights.detach().cpu().numpy() if torch.is_tensor(self.weights) else self.weights
                print('\nWeights:\n', pd.Series(w_sel).describe(percentiles=[0.2, 0.4, 0.6, 0.8]))
        else:
            self.weights = np.ones(self.n_frames)
            if device is not None:
                self.trajectory = torch.as_tensor(self.trajectory, device=device)
                self.weights = torch.ones(self.n_frames, dtype=torch.float64, device=device)


def filter_weights(w, min_w=0.0, max_w=float("inf")):
    """The weight handling of reference utils.py:140-169 on the device: normalise ``w`` (CUDA tensor) to mean 1, keep the states
    with min_w < w < max_w, renormalise the kept weights to mean 1.  Returns (indices of the kept states, their weights)."""
    if not (isinstance(w, torch.Tensor) and w.is_cuda):
        raise RuntimeError("filter_weights: the weights must be a CUDA tensor (this build has no CPU path)")
    w = w.detach().to(torch.float64).contiguous()
    n = w.numel()
    L = _lib.lib()
    ws = torch.empty(int(L.cvf_weights_filter_workspace_bytes(n)), dtype=torch.uint8, device=w.device)
    idx = torch.empty(n, dtype=torch.int64, device=w.device)
    out = torch.empty(n, dtype=torch.float64, device=w.device)
    n_keep = torch.zeros(1, dtype=torch.int64, device=w.device)
    with torch.cuda.device(w.device):
        _lib.check(L.cvf_weights_filter(w.data_ptr(), n, float(min_w), float(min(max_w, 1.7e308)), idx.data_ptr(), out.data_ptr(),
                                        n_keep.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr()), "cvf_weights_filter")
    m = int(n_keep.item())
    return idx[:m], out[:m]


def calc_weights(csv_filename, sampling_beta, sys_beta, traj_weight_filename='weights.txt', energy_col_idx=1):
    """Weights of trajectory data from an energy column of a CSV file (reference utils.py:354-417):
    v_i = exp(-(beta_sys - beta_sim) (V_i - mean V)) / mean, written one per line to ``traj_weight_filename``.
    Host-side data preparation (the file feeds ``WeightedTrajectory(weight_filename=...)``); same arguments, prints and
    output file as the reference."""
    import pandas as pd
    print('\n=============Calculate Weights============')
    print(f'Reading potential from: {csv_filename}')
    vec = pd.read_csv(csv_filename)
    vec.rename(columns={vec.columns[0]: 'Time'}, inplace=True)
    print('\nWhole data:\n', vec.head(8))
    energy_col_name = vec.columns[energy_col_idx]
    print('\nUse {:d}th column to reweight, name: {}'.format(energy_col_idx, energy_col_name))
    energy = vec[energy_col_name].to_numpy(dtype=np.float64)
    print(f'\nsampling beta={sampling_beta}, system beta={sys_beta}')
    nonnormalized = np.exp(-(sys_beta - sampling_beta) * (energy - energy.mean()))
    weights = pd.DataFrame(nonnormalized / np.mean(nonnormalized), columns=['weight'])
    print('\nWeight:\n', weights.head(8), '\n\nSummary of weights:\n', weights.describe())
    weights.to_csv(traj_weight_filename, header=False, index=False)
    print(f'weights saved to: {traj_weight_filename}')


def _stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def _recording(x):
    """True when autograd records the call: grad mode is on and the input requires grad.  Only then do the layers go through
    the cvf:: operators that carry the backward; otherwise they make the plain library call."""
    return torch.is_grad_enabled() and x.requires_grad


def _require_cuda_f32(x, what):
    if not (isinstance(x, torch.Tensor) and x.is_cuda):
        raise RuntimeError(f"{what}: input must be a CUDA tensor (this build has no CPU path)")
    if x.dtype != torch.float32:
        raise RuntimeError(f"{what}: input must be float32, got {x.dtype}")
    return x.contiguous()


class Align(torch.nn.Module):
    """Kabsch alignment of every frame onto a reference structure.

    x [B,N,3] -> (x - c) R with c the centroid of the alignment atoms and R the proper rotation that best
    superimposes them onto ``ref_positions`` (centred internally).  ``align_indices`` index the N input atoms.
    """

    def __init__(self, ref_positions, align_indices):
        super().__init__()
        ref = np.asarray(ref_positions, dtype=np.float64).reshape(-1, 3)
        idx = np.asarray(align_indices, dtype=np.int64).reshape(-1)
        if len(idx) != ref.shape[0]:
            raise ValueError(f"{ref.shape[0]} reference positions for {len(idx)} alignment atoms")
        if len(idx) < 3:
            raise ValueError("alignment needs at least 3 atoms")
        ref = ref - ref.mean(0, keepdims=True)
        self.register_buffer("ref_pos", torch.as_tensor(ref, dtype=torch.float32))
        self.register_buffer("align_idx", torch.as_tensor(idx, dtype=torch.int32))

    @classmethod
    def from_atom_groups(cls, align_atom_group, input_atom_group):
        """molann-style construction (examples/dipeptide/main.ipynb:343-345): atom groups expose .ix and .positions."""
        pos_of = {int(a): i for i, a in enumerate(np.asarray(input_atom_group.ix))}
        local = [pos_of[int(a)] for a in np.asarray(align_atom_group.ix)]
        return cls(np.asarray(align_atom_group.positions), local)

    def show_info(self):
        print('\natom indices used for alignment: \n', self.align_idx.cpu().numpy())
        print('\npositions of reference state used in aligment:\n', self.ref_pos.cpu().numpy())

    def forward(self, x, out=None):
        """Aligned frames; ``out`` (optional, [B,N,3] float32 on the same device) receives them without an allocation.
        Differentiable in ``x`` (first order) when called without ``out``."""
        x = _require_cuda_f32(x, "Align")
        if x.dim() != 3 or x.shape[2] != 3:
            raise RuntimeError(f"Align expects [B,N,3], got {tuple(x.shape)}")
        if out is not None and (out.shape != x.shape or out.dtype != torch.float32 or out.device != x.device or not out.is_contiguous()):
            raise RuntimeError("Align: out must be a contiguous float32 tensor of the input's shape on the input's device")
        from . import _ops      # registers the cvf:: operators and their autograd formulas
        _ops.check_align_args(x, self.ref_pos, self.align_idx, "Align")
        if out is None and _recording(x):
            return torch.ops.cvf.align_fwd(x, self.ref_pos, self.align_idx)
        y = torch.empty_like(x) if out is None else out
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().cvf_align_fwd(x.data_ptr(), x.shape[0], x.shape[1], self.align_idx.data_ptr(),
                                                self.align_idx.numel(), self.ref_pos.data_ptr(), y.data_ptr(), None,
                                                None, _stream_ptr()), "cvf_align_fwd")
        return y

    def rotation(self, x):
        """Aligned frames plus the rotation R [B,3,3] and centroid c [B,3] of every frame."""
        from . import _ops
        x = _require_cuda_f32(x, "Align")
        _ops.check_align_args(x, self.ref_pos, self.align_idx, "Align.rotation")
        y = torch.empty_like(x)
        R = torch.empty(x.shape[0], 3, 3, device=x.device, dtype=torch.float32)
        c = torch.empty(x.shape[0], 3, device=x.device, dtype=torch.float32)
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().cvf_align_fwd(x.data_ptr(), x.shape[0], x.shape[1], self.align_idx.data_ptr(),
                                                self.align_idx.numel(), self.ref_pos.data_ptr(), y.data_ptr(),
                                                R.data_ptr(), c.data_ptr(), _stream_ptr()), "cvf_align_fwd")
        return y, R, c


class FeatureMap(torch.nn.Module):
    """Feature map on (aligned) coordinates [B,N,3] -> [B,d_r].

    ``features``: list of ``(type, atom_indices)`` with type 'position' (any number of atoms, 3 outputs each),
    'bond' (2 atoms, distance), 'angle' (3 atoms, cosine of the angle at the middle atom), 'dihedral'
    (4 atoms, (cos, sin) of the dihedral angle); outputs are concatenated in list order.
    """

    def __init__(self, features):
        super().__init__()
        self.features = []
        for ftype, atoms in features:
            atoms = [int(a) for a in atoms]
            if ftype not in _FEATURE_TYPES:
                raise ValueError(f"unknown feature type {ftype!r} (position, bond, angle, dihedral)")
            need = _FEATURE_TYPES[ftype][1]
            if need is not None and len(atoms) != need:
                raise ValueError(f"feature {ftype!r} takes {need} atoms, got {len(atoms)}")
            self.features.append((ftype, atoms))
        if not self.features:
            raise ValueError("empty feature list")

    def output_dimension(self):
        return sum(3 * len(a) if t == "position" else _FEATURE_TYPES[t][2] for t, a in self.features)

    def records(self):
        """One (type id, atoms) record per kernel feature: multi-atom 'position' entries are split."""
        out = []
        for t, atoms in self.features:
            if t == "position":
                out += [(_lib.FEAT_POSITION, [a]) for a in atoms]
            else:
                out.append((_FEATURE_TYPES[t][0], atoms))
        return out

    def forward(self, x):
        return Preprocessing(None, self)(x)


class Preprocessing(torch.nn.Module):
    """r(x) = features(align(x)); either part may be None (molann.ann.PreprocessingANN analogue,
    examples/dipeptide/main.ipynb:348)."""

    def __init__(self, align_layer=None, feature_layer=None):
        super().__init__()
        if align_layer is not None and not isinstance(align_layer, Align):
            raise TypeError("align_layer must be colvarsfinder.utils.Align")
        if feature_layer is not None and not isinstance(feature_layer, FeatureMap):
            raise TypeError("feature_layer must be colvarsfinder.utils.FeatureMap")
        self.align = align_layer
        self.feature_mapper = feature_layer
        self._spec_cache = {}

    def output_dimension(self, n_atoms):
        return 3 * n_atoms if self.feature_mapper is None else self.feature_mapper.output_dimension()

    def forward(self, x):
        from . import _ops
        x = _require_cuda_f32(x, "Preprocessing")
        if x.dim() != 3 or x.shape[2] != 3:
            raise RuntimeError(f"Preprocessing expects [B,N,3], got {tuple(x.shape)}")
        if self.feature_mapper is None:
            return (self.align(x) if self.align is not None else x).reshape(x.shape[0], -1)
        key = (x.device, x.shape[1])
        if key not in self._spec_cache:
            self._spec_cache[key] = _ops.PreprocSpec(self, x.shape[1:], x.device, None)
        spec = self._spec_cache[key]
        if _recording(x):
            return torch.ops.cvf.features_fwd(x, spec.handle)
        out = torch.empty(x.shape[0], spec.d_r, device=x.device, dtype=torch.float32)
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().cvf_features_fwd(x.data_ptr(), x.shape[0], spec.struct_ptr(), out.data_ptr(),
                                                   _stream_ptr()), "cvf_features_fwd")
        return out


# ------------------------------------------------------------------------------------------ TorchScript export
# save_model (reference core.py:212-227) writes torch.jit.script(Sequential(pp_layer, cv)) for use OUTSIDE this package
# (PLUMED / Colvars load scripted_cv_{cpu,gpu}.pt through libtorch).  The training step never calls these modules: they are the
# same maps r(x) as the CUDA kernels, restated with stock torch ops so that the exported file has no dependency on libcvf.
class _ScriptAlign(torch.nn.Module):
    def __init__(self, ref_pos, align_idx):
        super().__init__()
        self.register_buffer("ref_pos", ref_pos.detach().clone().to(torch.float32))
        self.register_buffer("align_idx", align_idx.detach().clone().to(torch.long))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        xa = x.index_select(1, self.align_idx)
        c = xa.mean(1, keepdim=True)
        h = torch.matmul((xa - c).transpose(1, 2), self.ref_pos.to(x.dtype))
        u, s, vh = torch.linalg.svd(h)
        d = torch.sign(torch.linalg.det(torch.matmul(u, vh))).detach()
        diag = torch.ones_like(s)
        diag[:, 2] = d
        rot = torch.matmul(u * diag.unsqueeze(1), vh)
        return torch.matmul(x - c, rot)


class _ScriptFeatures(torch.nn.Module):
    def __init__(self, features):
        super().__init__()
        groups = {"position": [], "bond": [], "angle": [], "dihedral": []}
        src = []                                   # (group, column inside the group's block) of every output column
        for t, atoms in features:
            if t == "position":
                for a in atoms:
                    j = len(groups[t])
                    groups[t].append([a])
                    src += [(0, 3 * j), (0, 3 * j + 1), (0, 3 * j + 2)]
            elif t == "dihedral":
                j = len(groups[t])
                groups[t].append(atoms)
                src += [(3, 2 * j), (3, 2 * j + 1)]
            else:
                j = len(groups[t])
                groups[t].append(atoms)
                src.append((1 if t == "bond" else 2, j))
        widths = [3 * len(groups["position"]), len(groups["bond"]), len(groups["angle"]), 2 * len(groups["dihedral"])]
        offs = [0, widths[0], widths[0] + widths[1], widths[0] + widths[1] + widths[2]]
        self.register_buffer("perm", torch.tensor([offs[g] + c for g, c in src], dtype=torch.long))
        for name, width in (("position", 1), ("bond", 2), ("angle", 3), ("dihedral", 4)):
            t = torch.tensor(groups[name], dtype=torch.long).reshape(-1, width)
            self.register_buffer(name + "_idx", t)

    def forward(self, y: torch.Tensor) -> torch.Tensor:
        b = y.shape[0]
        parts: List[torch.Tensor] = []
        parts.append(y.index_select(1, self.position_idx[:, 0]).reshape(b, -1))
        p0 = y.index_select(1, self.bond_idx[:, 0])
        p1 = y.index_select(1, self.bond_idx[:, 1])
        parts.append(torch.linalg.norm(p1 - p0, dim=2))
        a0 = y.index_select(1, self.angle_idx[:, 0])
        a1 = y.index_select(1, self.angle_idx[:, 1])
        a2 = y.index_select(1, self.angle_idx[:, 2])
        u = a0 - a1
        v = a2 - a1
        parts.append((u * v).sum(2) / (torch.linalg.norm(u, dim=2) * torch.linalg.norm(v, dim=2)))
        d0 = y.index_select(1, self.dihedral_idx[:, 0])
        d1 = y.index_select(1, self.dihedral_idx[:, 1])
        d2 = y.index_select(1, self.dihedral_idx[:, 2])
        d3 = y.index_select(1, self.dihedral_idx[:, 3])
        r12 = d1 - d0
        r23 = d2 - d1
        r34 = d3 - d2
        n1 = torch.cross(r12, r23, dim=2)
        n2 = torch.cross(r23, r34, dim=2)
        den = torch.sqrt((n1 * n1).sum(2) * (n2 * n2).sum(2))
        cs = (n1 * n2).sum(2) / den
        sn = (n1 * r34).sum(2) * torch.linalg.norm(r23, dim=2) / den
        parts.append(torch.stack([cs, sn], dim=2).reshape(b, -1))
        return torch.cat(parts, dim=1).index_select(1, self.perm)


class _ScriptFlatten(torch.nn.Module):
    def forward(self, y: torch.Tensor) -> torch.Tensor:
        return y.reshape(y.shape[0], -1)


def scriptable(pp_layer):
    """A torch.jit.script-able module computing the same r(x) as ``pp_layer`` with stock torch ops (used by save_model for the
    exported collective-variable file).  Modules that are not defined in this package are returned unchanged."""
    if isinstance(pp_layer, Align):
        return torch.nn.Sequential(_ScriptAlign(pp_layer.ref_pos, pp_layer.align_idx), _ScriptFlatten())
    if isinstance(pp_layer, FeatureMap):
        return _ScriptFeatures(pp_layer.features)
    if isinstance(pp_layer, Preprocessing):
        mods = []
        if pp_layer.align is not None:
            mods.append(_ScriptAlign(pp_layer.align.ref_pos, pp_layer.align.align_idx))
        mods.append(_ScriptFlatten() if pp_layer.feature_mapper is None else _ScriptFeatures(pp_layer.feature_mapper.features))
        return torch.nn.Sequential(*mods)
    return pp_layer
