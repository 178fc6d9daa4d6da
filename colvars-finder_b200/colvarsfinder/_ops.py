"""Glue between the task classes and libcvf_sm100.so: descriptors, flat parameter storage, the ``torch.library`` custom
operators (namespace ``cvf``) that stand where the reference builds its autograd graph, and the one collective per pass.

Operators (each with ``register_fake`` for shape inference and ``register_autograd``, so that the reference's
``loss.backward()`` -- core.py:517,708,1115 -- fills ``param.grad`` from the CUDA passes):

* ``cvf::eigen_stats(X, w, params, handle, slot) -> (y, stats)``   pass 1 + all-reduce; backward = ``cvf::eigen_grad`` (pass 2)
* ``cvf::eigen_combine(stats, handle) -> comb``                    loss / eigenvalues / ordering of core.py:426-455
* ``cvf::eigen_loss(X, w, params, handle) -> (y, comb)``           the two above fused (EigenFunctionTask's generator loss)
* ``cvf::eigen_tlag_sx``, ``cvf::eigen_tlag_combine``              transfer-operator branch (core.py:412-416,428,440)
* ``cvf::ae_sums(F, T, w, params, want_grad, handle) -> (sums, gsum)``  weighted reconstruction error and its gradient
* ``cvf::align_fwd(x, ref, idx) -> y``                             Kabsch alignment (stand-alone pre-pass); backward =
  ``cvf::align_vjp(x, ref, idx, g_y) -> g_x``
* ``cvf::features_fwd(x, handle) -> r``                            features (after alignment) of a PreprocSpec; backward =
  ``cvf::features_vjp(x, g_r, handle) -> g_x``

The two ``*_vjp`` operators are first-order only: they have no autograd formula, so differentiating a gradient that passed
through them raises instead of returning a zero or partial second derivative.

``handle`` is an integer naming the host-side context (descriptors + scratch) of a task: operators take tensors and plain
scalars only.

Data-parallel layout: every rank holds a shard of the frames in its own HBM and the full (replicated)
parameters.  The loss couples frames only through a handful of batch sums, so each pass ends with ONE
``all_reduce(SUM)`` over NCCL -- fp64 batch sums after pass 1, fp64 gradient sums after pass 2 -- and every
rank then runs the same tiny combine kernel / optimizer step.  With one process the collective is skipped.
"""
from __future__ import annotations

import ctypes as C
import itertools
import weakref
from typing import Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .nn import chain_spec


# ------------------------------------------------------------------------------------------ distributed
def world_size() -> int:
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def rank() -> int:
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def backend() -> str:
    return dist.get_backend() if dist.is_available() and dist.is_initialized() else ''


_COLLECTIVES_OFF = False


class no_collectives:
    """Context manager: the step runs as if this rank were alone (its all-reduces become no-ops).  Used by the data-parallel
    parity checks, which compare the sharded step with the same step on the whole batch inside one process."""

    def __enter__(self):
        global _COLLECTIVES_OFF
        self._saved, _COLLECTIVES_OFF = _COLLECTIVES_OFF, True

    def __exit__(self, *exc):
        global _COLLECTIVES_OFF
        _COLLECTIVES_OFF = self._saved


def allreduce_sum_(t: torch.Tensor) -> torch.Tensor:
    """In-place sum over ranks on the current stream (no-op for a single process)."""
    if world_size() > 1 and not _COLLECTIVES_OFF:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def shard_range(n: int, r: int, w: int):
    """Contiguous, near-equal frame shard [lo, hi) of rank r out of w."""
    base, rem = divmod(n, w)
    lo = r * base + min(r, rem)
    return lo, lo + base + (1 if r < rem else 0)


# ------------------------------------------------------------------------------------------ descriptors
class PreprocSpec:
    """``cvf_preproc`` for a pp_layer: Identity, utils.Align, utils.FeatureMap or utils.Preprocessing."""

    def __init__(self, pp_layer, frame_shape, device, diag_coeff):
        from . import utils
        self.device = torch.device(device)
        self._keep = []
        self.alignment_elided = False
        s = _lib.Preproc()
        frame_shape = tuple(int(v) for v in frame_shape)
        tot_dim = int(np.prod(frame_shape))
        diag = None
        if diag_coeff is not None:
            diag = torch.as_tensor(diag_coeff).detach().to("cpu", torch.float32).reshape(-1)
            if diag.numel() != tot_dim:
                raise RuntimeError(f"diag_coeff has {diag.numel()} entries, the state has {tot_dim} coordinates")
            if bool((diag == 1.0).all()):
                diag = None
        if isinstance(pp_layer, torch.nn.Identity):
            if len(frame_shape) != 1:
                raise RuntimeError("Identity pre-processing needs a flat [n, d] trajectory")
            s.kind, s.dim, s.d_r = 0, tot_dim, tot_dim
            if diag is not None:
                s.diag = self._dev(diag)
            self.d_r = tot_dim
        else:
            if isinstance(pp_layer, utils.Align):
                align, fmap = pp_layer, None
            elif isinstance(pp_layer, utils.FeatureMap):
                align, fmap = None, pp_layer
            elif isinstance(pp_layer, utils.Preprocessing):
                align, fmap = pp_layer.align, pp_layer.feature_mapper
            else:
                raise RuntimeError(
                    f"pp_layer of type {type(pp_layer).__name__} is outside the supported envelope of the CUDA step: use "
                    "torch.nn.Identity, colvarsfinder.utils.Align, FeatureMap or Preprocessing (no PyTorch fallback)")
            if len(frame_shape) != 2 or frame_shape[1] != 3:
                raise RuntimeError(f"molecular pre-processing needs [n, N, 3] frames, got frame shape {frame_shape}")
            n_atoms = frame_shape[0]
            if fmap is None:
                records = [(_lib.FEAT_POSITION, [a]) for a in range(n_atoms)]
            else:
                records = fmap.records()
            used, pos = [], {}
            for _, atoms in records:
                for a in atoms:
                    if not 0 <= a < n_atoms:
                        raise RuntimeError(f"feature atom {a} outside the {n_atoms} input atoms")
                    if a not in pos:
                        pos[a] = len(used)
                        used.append(a)
            n_feat_atoms = len(used)
            positions_only = all(t == _lib.FEAT_POSITION for t, _ in records) and len(records) == n_feat_atoms
            align_idx = [] if align is None else [int(a) for a in align.align_idx.cpu().tolist()]
            # Bond lengths, angles and dihedrals do not change under the rigid motion the alignment applies, and with
            # diag_coeff = 1 neither does |grad_x f|^2: r(x) and its Jacobian products are evaluated on the raw frame and
            # the Kabsch step (with its Jacobian) drops out of the training step.  (pp_layer(x) itself still aligns.)
            self.alignment_elided = bool(align_idx) and diag is None and all(t != _lib.FEAT_POSITION for t, _ in records)
            if self.alignment_elided:
                align_idx = []
            for a in align_idx:
                if not 0 <= a < n_atoms:
                    raise RuntimeError(f"alignment atom {a} outside the {n_atoms} input atoms")
                if a not in pos:
                    pos[a] = len(used)
                    used.append(a)
            positions_only = positions_only and len(used) == n_feat_atoms
            s.kind, s.n_atoms, s.n_used = 1, n_atoms, len(used)
            s.used_atoms = self._dev(torch.tensor(used, dtype=torch.int32))
            s.n_align = len(align_idx)
            if align_idx:
                s.align_used = self._dev(torch.tensor([pos[a] for a in align_idx], dtype=torch.int32))
                s.ref = self._dev(align.ref_pos.detach().to("cpu", torch.float32).reshape(-1))
            table = []
            d_r = 0
            for t, atoms in records:
                table.append([t] + [pos[a] for a in atoms] + [0] * (4 - len(atoms)))
                d_r += {_lib.FEAT_POSITION: 3, _lib.FEAT_BOND: 1, _lib.FEAT_ANGLE: 1, _lib.FEAT_DIHEDRAL: 2}[t]
            s.n_feat, s.d_r = len(records), d_r
            for t, _ in records:
                s.n_feat_by_type[t] += 1
            reads = {}
            for t, atoms in records:
                for a in atoms:
                    reads[a] = reads.get(a, 0) + (2 if t == _lib.FEAT_POSITION else 1)
            s.n_self_records = sum(1 for t, atoms in records
                                   if t != _lib.FEAT_POSITION and any(reads[a] == 1 for a in atoms))
            s.n_shared_atoms = sum(1 for c in reads.values() if c > 1)
            s.feat = self._dev(torch.tensor(table, dtype=torch.int32).reshape(-1))
            s.positions_only = 1 if positions_only else 0
            s.used_identity = 1 if used == list(range(n_atoms)) else 0
            if diag is not None:
                g = diag.reshape(n_atoms, 3)[torch.tensor(used, dtype=torch.long)].reshape(-1).contiguous()
                s.diag = self._dev(g)
            self.d_r = d_r
        self.struct = s
        self.handle = _register_context(self)      # the ``handle`` of cvf::features_fwd / cvf::features_vjp

    def _dev(self, t):
        t = t.contiguous().to(self.device)
        self._keep.append(t)
        return t.data_ptr()

    def struct_ptr(self):
        return C.byref(self.struct)


class FlatParams:
    """All parameters of a set of Linear stacks in ONE contiguous fp32 device buffer, in torch's
    ``parameters()`` order; the modules' parameters are re-pointed to views of it, so the optimizer updates the
    buffer the kernels read and nothing is packed per step."""

    def __init__(self, chains, device):
        self.params = []
        self.dims, self.acts = [], []
        for seq in chains:
            dims, acts, lins = chain_spec(seq)
            self.dims.append(dims), self.acts.append(acts)
            for lin in lins:
                self.params += [lin.weight, lin.bias]
        n = sum(p.numel() for p in self.params)
        self.flat = torch.empty(n, dtype=torch.float32, device=device)
        self.offsets = []
        off = 0
        for p in self.params:
            self.offsets.append(off)
            off += p.numel()
        self.n = n
        self.rebind()

    def rebind(self):
        with torch.no_grad():
            for p, off in zip(self.params, self.offsets):
                view = self.flat[off:off + p.numel()].view(p.shape)
                if p.data.data_ptr() != view.data_ptr() or p.data.device != self.flat.device:
                    view.copy_(p.data.to(device=self.flat.device, dtype=torch.float32))
                    p.data = view

    def check(self):
        """Parameters must still alias the flat buffer (e.g. model.to() would break it): re-bind if not."""
        base = self.flat.data_ptr()
        for p, off in zip(self.params, self.offsets):
            if p.data.data_ptr() != base + 4 * off:
                self.rebind()
                return

    def split(self, g):
        return tuple(g[off:off + p.numel()].view(p.shape) for p, off in zip(self.params, self.offsets))


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check_batch(X, weight, what):
    if not (X.is_cuda and weight.is_cuda):
        raise RuntimeError(f"{what}: tensors must live on a CUDA device (this build has no CPU path)")
    if X.dtype != torch.float32:
        raise RuntimeError(f"{what}: data must be float32, got {X.dtype}")
    X = X.detach().contiguous()
    weight = weight.detach().to(torch.float32).contiguous()
    if weight.numel() != X.shape[0]:
        raise RuntimeError(f"{what}: {weight.numel()} weights for {X.shape[0]} states")
    return X, weight


# ------------------------------------------------------------------------------------------ context registry
# Operators registered with torch.library take tensors and scalars; everything else a call needs (descriptor structs, the
# scratch buffer, loss constants) lives in a context object that the operator finds through an integer handle.
_CONTEXTS = weakref.WeakValueDictionary()
_HANDLES = itertools.count(1)


def _register_context(obj) -> int:
    h = next(_HANDLES)
    _CONTEXTS[h] = obj
    return h


def _context(handle: int):
    try:
        return _CONTEXTS[handle]
    except KeyError:
        raise RuntimeError(f"cvf: context {handle} no longer exists (its task object was deleted)") from None


class _PackFlat(torch.autograd.Function):
    """The flat parameter buffer as a differentiable function of the parameters that alias it: forward is free (the
    parameters ARE views of the buffer), backward hands every parameter its slice of the buffer's gradient."""

    @staticmethod
    def forward(ctx, flatp, *params):
        ctx.flatp = flatp
        return flatp.flat.detach()

    @staticmethod
    def backward(ctx, g):
        return (None,) + ctx.flatp.split(g)


# ------------------------------------------------------------------------------------------ eigenfunctions
class EigenContext:
    """Everything constant across steps for one set of k equally-shaped networks on one pre-processing layer: descriptors,
    loss constants, scratch.  ``model`` may be None when the caller packs the parameters itself (RegAutoEncoderTask)."""

    def __init__(self, model, pp_layer, frame_shape, device, alpha, eig_w, beta, diag_coeff, sort, dims=None, acts=None, k=None):
        self.device = torch.device(device)
        if model is not None:
            self.k = len(model.eigen_funcs)
            self.flat = FlatParams(list(model.eigen_funcs), self.device)
            if any(d != self.flat.dims[0] for d in self.flat.dims):
                raise RuntimeError("all eigenfunction networks must share one architecture")
            dims, acts = self.flat.dims[0], self.flat.acts[0]
        else:
            self.k, self.flat = int(k), None
        if self.k > _lib.MAX_K:
            raise RuntimeError(f"k = {self.k} eigenfunctions is outside the supported envelope (<= {_lib.MAX_K})")
        self.mlp = _lib.make_mlp(dims, acts)
        self.spec = PreprocSpec(pp_layer, frame_shape, self.device, diag_coeff)
        if self.spec.d_r != dims[0]:
            raise RuntimeError(f"pre-processing layer outputs {self.spec.d_r} features, the networks take {dims[0]}")
        self.alpha, self.beta, self.sort = float(alpha), float(beta), 1 if sort else 0
        self.eig_w = (C.c_double * self.k)(*[float(v) for v in (list(eig_w) + [0.0] * self.k)[:self.k]])
        L = _lib.lib()
        self.n_stats = L.cvf_eigen_num_stats(self.k)
        self.n_comb = L.cvf_eigen_num_combine(self.k)
        self.n_per_net = int(L.cvf_mlp_param_count(C.byref(self.mlp)))
        self.fast_path = bool(L.cvf_eigen_path(self.spec.struct_ptr(), C.byref(self.mlp), self.k) == 1)
        # scratch slots: 0 for X, 1 for the time-lagged X of the transfer-operator loss (both must survive until backward)
        self._ws = {}
        self.handle = _register_context(self)

    def packed_params(self):
        """[k * n_per_net] parameter vector of a model-backed context, differentiable w.r.t. the model's parameters."""
        self.flat.check()
        return _PackFlat.apply(self.flat, *self.flat.params)

    def _workspace_for(self, B, slot=0):
        """Scratch of the step kernels, grown to the largest batch seen (PyTorch's caching allocator owns it)."""
        ws = self._ws.get(slot)
        if ws is None or B > ws["frames"]:
            need = int(_lib.lib().cvf_eigen_workspace_bytes(self.spec.struct_ptr(), C.byref(self.mlp), self.k, B))
            if need <= 0:
                raise RuntimeError("cvf_eigen_workspace_bytes: unsupported configuration")
            serial = ws["serial"] if ws else 0
            self._ws[slot] = None
            ws = {"buf": torch.empty(need, dtype=torch.uint8, device=self.device), "bytes": need, "frames": B, "serial": serial,
                  "valid": False, "pver": None}
            self._ws[slot] = ws
        return ws

    def _param_version(self, params):
        # the flat buffer's own counter does not see optimizer updates (they go through the parameters' views): add theirs
        v = params._version
        if self.flat is not None and params.data_ptr() == self.flat.flat.data_ptr():
            v += sum(p._version for p in self.flat.params)
        return (params.data_ptr(), v)

    def _own_params(self, params):
        if params is not None:
            return params
        if self.flat is None:
            raise RuntimeError("this context has no model of its own: pass the packed parameter vector")
        self.flat.check()
        return self.flat.flat

    def stats(self, X, weight, params=None, slot=0):
        """Pass 1 on this rank's frames -> (y [k,B] fp32, local stats fp64).  ``params`` defaults to the model's flat buffer."""
        L = _lib.lib()
        B = X.shape[0]
        params = self._own_params(params)
        if params.numel() != self.k * self.n_per_net or params.dtype != torch.float32 or not params.is_contiguous():
            raise RuntimeError(f"cvf::eigen_stats: params must be a contiguous float32 vector of {self.k * self.n_per_net} entries")
        ws = self._workspace_for(B, slot)
        y = torch.empty(self.k, B, dtype=torch.float32, device=self.device)
        stats = torch.empty(self.n_stats, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(L.cvf_eigen_stats(X.data_ptr(), weight.data_ptr(), B, self.spec.struct_ptr(), C.byref(self.mlp), self.k,
                                         params.data_ptr(), y.data_ptr(), stats.data_ptr(), ws["buf"].data_ptr(), ws["bytes"],
                                         _stream()), "cvf_eigen_stats")
        ws["serial"] += 1
        ws["valid"], ws["pver"] = True, self._param_version(params)
        ws["xkey"] = (X.data_ptr(), X.shape[0], X._version, weight.data_ptr(), weight._version)
        return y, stats

    def serial(self, slot=0):
        ws = self._ws.get(slot)
        return ws["serial"] if ws else -1

    def combine(self, stats):
        comb = torch.empty(self.n_comb, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().cvf_eigen_combine(stats.data_ptr(), self.k, self.alpha, self.eig_w, self.beta, self.sort,
                                                    comb.data_ptr(), _stream()), "cvf_eigen_combine")
        return comb

    def grads(self, X, weight, y, comb, seed_extra=None, slot=0, serial=None, params=None):
        """Pass 2 on this rank's frames -> fp64 gradient sums [k * n_per_net].  ``serial`` names the stats() call whose scratch
        may be reused (None: the latest one on the slot)."""
        g = torch.empty(self.k * self.n_per_net, dtype=torch.float64, device=self.device)
        ws = self._workspace_for(X.shape[0], slot)
        params = self._own_params(params)
        if serial is None:
            serial = ws["serial"]
        # the scratch still holds pass 1's intermediates iff the stats() call of THIS loss was the last one on the slot and
        # neither the batch nor the parameters were written since
        valid = 1 if (ws["valid"] and ws["serial"] == serial and ws["pver"] == self._param_version(params) and
                      ws.get("xkey") == (X.data_ptr(), X.shape[0], X._version, weight.data_ptr(), weight._version)) else 0
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().cvf_eigen_grad(X.data_ptr(), weight.data_ptr(), X.shape[0], self.spec.struct_ptr(),
                                                 C.byref(self.mlp), self.k, params.data_ptr(), y.data_ptr(),
                                                 comb.data_ptr(), None if seed_extra is None else seed_extra.data_ptr(),
                                                 g.data_ptr(), ws["buf"].data_ptr(), ws["bytes"], valid, _stream()),
                       "cvf_eigen_grad")
        # pass 2 consumes the scratch (it leaves v = J J^T u where pass 1 left u): a second backward recomputes it
        ws["valid"] = False
        return g

    def tlag_terms(self, y, y_lag, weight, coef=None):
        """sum_f w (y' - y)^2 per network (coef None), or the per-frame seed term coef_i w (y_i - y'_i) of the backward pass."""
        L, B = _lib.lib(), y.shape[1]
        with torch.cuda.device(self.device):
            if coef is None:
                sx = torch.empty(self.k, dtype=torch.float64, device=self.device)
                ws = self._workspace_for(B, 0)
                _lib.check(L.cvf_eigen_tlag_terms(y.data_ptr(), y_lag.data_ptr(), weight.data_ptr(), B, self.k, None, sx.data_ptr(),
                                                  None, ws["buf"].data_ptr(), ws["bytes"], _stream()), "cvf_eigen_tlag_terms")
                return sx
            extra = torch.empty(self.k, B, dtype=torch.float32, device=self.device)
            _lib.check(L.cvf_eigen_tlag_terms(y.data_ptr(), y_lag.data_ptr(), weight.data_ptr(), B, self.k, coef.data_ptr(), None,
                                              extra.data_ptr(), None, 0, _stream()), "cvf_eigen_tlag_terms")
        return extra

    def tlag_combine(self, stats, stats_lag, sx, tau):
        comb = torch.empty(self.n_comb + self.k, dtype=torch.float64, device=self.device)
        comb_lag = torch.empty(self.n_comb, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().cvf_eigen_tlag_combine(stats.data_ptr(), stats_lag.data_ptr(), sx.data_ptr(), self.k, self.alpha,
                                                         self.eig_w, float(tau), self.sort, comb.data_ptr(), comb_lag.data_ptr(),
                                                         _stream()), "cvf_eigen_tlag_combine")
        return comb, comb_lag


def _coef_from_gstats(g_stats, k, n_comb):
    """Gradient w.r.t. the batch sums (S0, S1[k], S2[k,k], SD[k]) -> the coefficient blocks of the combine vector
    (mean = 0, cD = dL/dSD, C2 = dL/dS2 + its transpose, a0 = dL/dS1; include/cvf.h)."""
    coef = torch.zeros(n_comb, dtype=torch.float64, device=g_stats.device)
    g2 = g_stats[1 + k:1 + k + k * k].view(k, k)
    coef[3 + 3 * k:3 + 4 * k] = g_stats[1 + k + k * k:1 + 2 * k + k * k]
    coef[3 + 4 * k:3 + 4 * k + k * k] = (g2 + g2.t()).reshape(-1)
    coef[3 + 4 * k + k * k:3 + 5 * k + k * k] = g_stats[1:1 + k]
    return coef


def _gstats_from_comb(comb, k):
    """The inverse map for a combine vector written by the library (a0 = 0, C2 symmetric): d loss / d (S0, S1, S2, SD)."""
    mean = comb[3 + 2 * k:3 + 3 * k]
    cD = comb[3 + 3 * k:3 + 4 * k]
    C2 = comb[3 + 4 * k:3 + 4 * k + k * k].view(k, k)
    a0 = comb[3 + 4 * k + k * k:3 + 5 * k + k * k]
    return torch.cat([comb.new_zeros(1), a0 - C2 @ mean, (0.5 * C2).reshape(-1), cD])


@torch.library.custom_op("cvf::eigen_stats", mutates_args=())
def eigen_stats_op(X: torch.Tensor, w: torch.Tensor, params: torch.Tensor, handle: int, slot: int) -> Tuple[torch.Tensor, torch.Tensor]:
    ectx = _context(handle)
    y, stats = ectx.stats(X, w, params, slot)
    allreduce_sum_(stats)
    return y, stats


@eigen_stats_op.register_fake
def _(X, w, params, handle, slot):
    ectx = _context(handle)
    return X.new_empty((ectx.k, X.shape[0]), dtype=torch.float32), X.new_empty((ectx.n_stats,), dtype=torch.float64)


@torch.library.custom_op("cvf::eigen_grad", mutates_args=())
def eigen_grad_op(X: torch.Tensor, w: torch.Tensor, y: torch.Tensor, params: torch.Tensor, coef: torch.Tensor,
                  seed_extra: Optional[torch.Tensor], handle: int, slot: int, serial: int) -> torch.Tensor:
    ectx = _context(handle)
    if seed_extra is not None:
        seed_extra = seed_extra.to(torch.float32).contiguous()
    g = ectx.grads(X, w, y, coef.contiguous(), seed_extra, slot, serial, params)
    allreduce_sum_(g)
    return g.to(torch.float32)


@eigen_grad_op.register_fake
def _(X, w, y, params, coef, seed_extra, handle, slot, serial):
    return params.new_empty(params.shape)


def _eigen_stats_setup(ctx, inputs, output):
    X, w, params, handle, slot = inputs
    ctx.save_for_backward(X, w, params, output[0])
    ctx.set_materialize_grads(False)      # an unused y must not turn into a [k, B] tensor of zeros
    ctx.handle, ctx.slot = handle, slot
    ctx.serial = _context(handle).serial(slot)


def _eigen_stats_backward(ctx, g_y, g_stats):
    X, w, params, y = ctx.saved_tensors
    ectx = _context(ctx.handle)
    if g_stats is None and g_y is None:
        return None, None, None, None, None
    if g_stats is None:
        g_stats = torch.zeros(ectx.n_stats, dtype=torch.float64, device=X.device)
    coef = _coef_from_gstats(g_stats.to(torch.float64), ectx.k, ectx.n_comb)
    g = eigen_grad_op(X, w, y, params, coef, g_y, ctx.handle, ctx.slot, ctx.serial)
    return None, None, g, None, None


eigen_stats_op.register_autograd(_eigen_stats_backward, setup_context=_eigen_stats_setup)


@torch.library.custom_op("cvf::eigen_combine", mutates_args=())
def eigen_combine_op(stats: torch.Tensor, handle: int) -> torch.Tensor:
    return _context(handle).combine(stats.contiguous())


@eigen_combine_op.register_fake
def _(stats, handle):
    return stats.new_empty((_context(handle).n_comb,))


def _eigen_combine_setup(ctx, inputs, output):
    ctx.save_for_backward(output)
    ctx.k = _context(inputs[1]).k


def _eigen_combine_backward(ctx, g_comb):
    comb, = ctx.saved_tensors
    return g_comb[0] * _gstats_from_comb(comb, ctx.k), None      # only the loss entry is differentiable


eigen_combine_op.register_autograd(_eigen_combine_backward, setup_context=_eigen_combine_setup)


@torch.library.custom_op("cvf::eigen_tlag_sx", mutates_args=())
def eigen_tlag_sx_op(y: torch.Tensor, y_lag: torch.Tensor, w: torch.Tensor, handle: int) -> torch.Tensor:
    sx = _context(handle).tlag_terms(y.contiguous(), y_lag.contiguous(), w)
    allreduce_sum_(sx)
    return sx


@eigen_tlag_sx_op.register_fake
def _(y, y_lag, w, handle):
    return y.new_empty((y.shape[0],), dtype=torch.float64)


@torch.library.custom_op("cvf::eigen_tlag_seed", mutates_args=())
def eigen_tlag_seed_op(y: torch.Tensor, y_lag: torch.Tensor, w: torch.Tensor, coef: torch.Tensor, handle: int) -> torch.Tensor:
    return _context(handle).tlag_terms(y.contiguous(), y_lag.contiguous(), w, coef=coef.to(torch.float64).contiguous())


@eigen_tlag_seed_op.register_fake
def _(y, y_lag, w, coef, handle):
    return torch.empty_like(y)


def _tlag_sx_setup(ctx, inputs, output):
    y, y_lag, w, handle = inputs
    ctx.save_for_backward(y, y_lag, w)
    ctx.set_materialize_grads(False)
    ctx.handle = handle


def _tlag_sx_backward(ctx, g_sx):
    y, y_lag, w = ctx.saved_tensors
    if g_sx is None:
        return None, None, None, None
    extra = eigen_tlag_seed_op(y, y_lag, w, 2.0 * g_sx, ctx.handle)      # d sx_i / d y_i = 2 w (y_i - y'_i)
    return extra, -extra, None, None


eigen_tlag_sx_op.register_autograd(_tlag_sx_backward, setup_context=_tlag_sx_setup)


@torch.library.custom_op("cvf::eigen_tlag_combine", mutates_args=())
def eigen_tlag_combine_op(stats: torch.Tensor, stats_lag: torch.Tensor, sx: torch.Tensor, tau: float,
                          handle: int) -> Tuple[torch.Tensor, torch.Tensor]:
    return _context(handle).tlag_combine(stats.contiguous(), stats_lag.contiguous(), sx.contiguous(), tau)


@eigen_tlag_combine_op.register_fake
def _(stats, stats_lag, sx, tau, handle):
    ectx = _context(handle)
    return stats.new_empty((ectx.n_comb + ectx.k,)), stats.new_empty((ectx.n_comb,))


def _tlag_combine_setup(ctx, inputs, output):
    ctx.save_for_backward(output[0], output[1])
    ctx.set_materialize_grads(False)
    ctx.k, ctx.n_comb = _context(inputs[4]).k, _context(inputs[4]).n_comb


def _tlag_combine_backward(ctx, g_comb, g_comb_lag):
    comb, comb_lag = ctx.saved_tensors
    if g_comb is None:
        return None, None, None, None, None
    gl = g_comb[0]
    k = ctx.k
    return (gl * _gstats_from_comb(comb, k), gl * _gstats_from_comb(comb_lag, k), gl * 0.5 * comb[ctx.n_comb:ctx.n_comb + k],
            None, None)


eigen_tlag_combine_op.register_autograd(_tlag_combine_backward, setup_context=_tlag_combine_setup)


@torch.library.custom_op("cvf::eigen_loss", mutates_args=())
def eigen_loss_op(X: torch.Tensor, w: torch.Tensor, params: torch.Tensor, handle: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """cvf::eigen_stats + cvf::eigen_combine in one operator (the generator branch of EigenFunctionTask.loss_func) -> (y, combine
    vector, loss as a float32 scalar).  The loss is an output of its own so that no slicing of the combine vector sits on the
    autograd path, and the backward pass reads the coefficient blocks straight out of the combine vector."""
    ectx = _context(handle)
    y, stats = ectx.stats(X, w, params, 0)
    allreduce_sum_(stats)
    comb = ectx.combine(stats)
    return y, comb, comb[0].to(torch.float32)


@eigen_loss_op.register_fake
def _(X, w, params, handle):
    ectx = _context(handle)
    return (X.new_empty((ectx.k, X.shape[0]), dtype=torch.float32), X.new_empty((ectx.n_comb,), dtype=torch.float64),
            X.new_empty((), dtype=torch.float32))


def _eigen_loss_setup(ctx, inputs, output):
    X, w, params, handle = inputs
    ctx.save_for_backward(X, w, params, output[0], output[1])
    ctx.set_materialize_grads(False)
    ctx.handle = handle
    ctx.serial = _context(handle).serial(0)


def _eigen_loss_backward(ctx, g_y, g_comb, g_loss):
    X, w, params, y, comb = ctx.saved_tensors
    if g_comb is not None:
        g_loss = g_comb[0].to(torch.float32) if g_loss is None else g_loss + g_comb[0].to(torch.float32)
    if g_loss is None and g_y is None:
        return None, None, None, None
    if g_loss is None:      # only y was used downstream: zero coefficients, the seeds come from g_y alone
        comb = torch.zeros_like(comb)
    g = eigen_grad_op(X, w, y, params, comb, g_y, ctx.handle, 0, ctx.serial)
    if g_loss is not None:
        g = g * g_loss
    return None, None, g, None


eigen_loss_op.register_autograd(_eigen_loss_backward, setup_context=_eigen_loss_setup)


def _loss_outputs(comb, k, loss=None):
    d = comb.detach()
    out32 = d[:3 + k].to(torch.float32)
    if loss is None:
        loss = comb[0].to(torch.float32)
    return loss, out32[3:3 + k], out32[1], out32[2], d[3 + k:3 + 2 * k].to(torch.int64)


def eigen_loss(ectx: EigenContext, X, weight):
    """EigenFunctionTask.loss_func, generator branch (reference core.py:387-457); ``loss.backward()`` = core.py:517."""
    X, weight = _check_batch(X, weight, "EigenFunctionTask.loss_func")
    _, comb, loss = eigen_loss_op(X, weight, ectx.packed_params(), ectx.handle)
    return _loss_outputs(comb, ectx.k, loss)


def eigen_lag_loss(ectx: EigenContext, tau, X, weight, X_lagged, weight_lagged):
    """Transfer-operator branch of EigenFunctionTask.loss_func (reference core.py:412-416,428,440): forward passes on X and on
    the time-lagged X; backward = two first-order passes seeded through y and y'."""
    X, weight = _check_batch(X, weight, "EigenFunctionTask.loss_func")
    X_lagged, weight_lagged = _check_batch(X_lagged, weight_lagged, "EigenFunctionTask.loss_func (time-lagged data)")
    if X_lagged.shape != X.shape:
        raise RuntimeError(f"time-lagged batch has shape {tuple(X_lagged.shape)}, the batch {tuple(X.shape)}")
    params = ectx.packed_params()
    y, st = eigen_stats_op(X, weight, params, ectx.handle, 0)
    yl, stl = eigen_stats_op(X_lagged, weight_lagged, params, ectx.handle, 1)
    sx = eigen_tlag_sx_op(y, yl, weight, ectx.handle)
    comb, _ = eigen_tlag_combine_op(st, stl, sx, float(tau), ectx.handle)
    return _loss_outputs(comb, ectx.k)


# ------------------------------------------------------------------------------------------ autoencoder
class AEContext:
    def __init__(self, model, device):
        self.device = torch.device(device)
        self.flat = FlatParams([model.encoder, model.decoder], self.device)
        e_dims, d_dims = self.flat.dims
        self.mlp = _lib.make_mlp(list(e_dims) + list(d_dims[1:]), list(self.flat.acts[0]) + list(self.flat.acts[1]))
        L = _lib.lib()
        self.n_params = int(L.cvf_mlp_param_count(C.byref(self.mlp)))
        assert self.n_params == self.flat.n
        self.ws_bytes, self.ws_frames, self.workspace = 0, 0, None
        self.d_r = e_dims[0]
        self.handle = _register_context(self)

    def packed_params(self):
        self.flat.check()
        return _PackFlat.apply(self.flat, *self.flat.params)

    def _workspace_for(self, B):
        if self.workspace is None or B > self.ws_frames:
            need = int(_lib.lib().cvf_ae_workspace_bytes(C.byref(self.mlp), B))
            if need <= 0:
                raise RuntimeError("cvf_ae_workspace_bytes: " + _lib.lib().cvf_last_error_string().decode("utf-8", "replace"))
            self.workspace = None
            self.workspace = torch.empty(need, dtype=torch.uint8, device=self.device)
            self.ws_bytes, self.ws_frames = need, B
        return self.workspace.data_ptr()

    def step(self, F, target, weight, params, want_grad):
        """One pass over this rank's frames -> fp64 [2 + n_params]: sum w|e|^2, sum w, gradient of the first sum."""
        buf = torch.zeros(2 + self.n_params, dtype=torch.float64, device=self.device) if not want_grad else \
            torch.empty(2 + self.n_params, dtype=torch.float64, device=self.device)
        gptr = buf.data_ptr() + 16 if want_grad else None
        ws = self._workspace_for(F.shape[0])
        with torch.cuda.device(self.device):
            if target is None:
                _lib.check(_lib.lib().cvf_ae_step(F.data_ptr(), weight.data_ptr(), F.shape[0], C.byref(self.mlp),
                                                  params.data_ptr(), buf.data_ptr(), gptr, ws, self.ws_bytes, _stream()),
                           "cvf_ae_step")
            else:
                _lib.check(_lib.lib().cvf_ae_step_target(F.data_ptr(), target.data_ptr(), weight.data_ptr(), F.shape[0],
                                                         C.byref(self.mlp), params.data_ptr(), buf.data_ptr(), gptr, ws,
                                                         self.ws_bytes, _stream()), "cvf_ae_step_target")
        return buf


@torch.library.custom_op("cvf::ae_sums", mutates_args=())
def ae_sums_op(F: torch.Tensor, target: Optional[torch.Tensor], w: torch.Tensor, params: torch.Tensor, want_grad: bool,
               handle: int) -> Tuple[torch.Tensor, torch.Tensor]:
    actx = _context(handle)
    if params.numel() != actx.n_params or params.dtype != torch.float32 or not params.is_contiguous():
        raise RuntimeError(f"cvf::ae_sums: params must be a contiguous float32 vector of {actx.n_params} entries")
    buf = actx.step(F, target, w, params, want_grad)
    allreduce_sum_(buf)
    return buf[:2].clone(), buf[2:].clone()


@ae_sums_op.register_fake
def _(F, target, w, params, want_grad, handle):
    return F.new_empty((2,), dtype=torch.float64), F.new_empty((params.numel(),), dtype=torch.float64)


def _ae_sums_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1])
    ctx.set_materialize_grads(False)
    ctx.want_grad = inputs[4]


def _ae_sums_backward(ctx, g_sums, g_gsum):
    if g_sums is None:
        return None, None, None, None, None, None
    if not ctx.want_grad:
        raise RuntimeError("weighted_MSE_loss was evaluated without gradients (torch.no_grad or frozen parameters)")
    gsum, = ctx.saved_tensors
    return None, None, None, (g_sums[0] * gsum).to(torch.float32), None, None


ae_sums_op.register_autograd(_ae_sums_backward, setup_context=_ae_sums_setup)


def ae_loss(actx: AEContext, F, weight, target=None):
    """weighted MSE (reference core.py:652-666; with a target, core.py:876-887); its parameter gradient is formed in the same pass."""
    F, weight = _check_batch(F, weight, "weighted_MSE_loss")
    if F.dim() != 2 or F.shape[1] != actx.d_r:
        raise RuntimeError(f"autoencoder input must be [B,{actx.d_r}], got {tuple(F.shape)}")
    if target is not None:
        target, _ = _check_batch(target, weight, "weighted_MSE_loss (target)")
        if target.shape != F.shape:
            raise RuntimeError(f"reconstruction target has shape {tuple(target.shape)}, the input {tuple(F.shape)}")
    want_grad = torch.is_grad_enabled() and any(p.requires_grad for p in actx.flat.params)
    sums, _ = ae_sums_op(F, target, weight, actx.packed_params(), want_grad, actx.handle)
    return (sums[0] / sums[1]).to(torch.float32)


# ------------------------------------------------------------------------------------------ alignment
def check_align_args(x, ref, align_idx, what):
    """The kernels dereference ref and align_idx on the device of x: a module left on the host (Align(...) without .to(device))
    is refused here instead of faulting on the GPU."""
    if ref.device != x.device or align_idx.device != x.device:
        raise RuntimeError(f"{what}: the reference and alignment indices live on {ref.device} / {align_idx.device}, the frames "
                           f"on {x.device}: move the module to the frames' device (.to(device))")
    if ref.dtype != torch.float32 or align_idx.dtype != torch.int32 or ref.numel() != 3 * align_idx.numel():
        raise RuntimeError(f"{what}: reference must be float32 [n_align,3] and alignment indices int32 [n_align]")


@torch.library.custom_op("cvf::align_fwd", mutates_args=())
def align_fwd_op(x: torch.Tensor, ref: torch.Tensor, align_idx: torch.Tensor) -> torch.Tensor:
    check_align_args(x, ref, align_idx, "cvf::align_fwd")
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().cvf_align_fwd(x.data_ptr(), x.shape[0], x.shape[1], align_idx.data_ptr(), align_idx.numel(),
                                            ref.data_ptr(), y.data_ptr(), None, None, _stream()), "cvf_align_fwd")
    return y


@align_fwd_op.register_fake
def _(x, ref, align_idx):
    return torch.empty_like(x)


@torch.library.custom_op("cvf::align_vjp", mutates_args=())
def align_vjp_op(x: torch.Tensor, ref: torch.Tensor, align_idx: torch.Tensor, g_y: torch.Tensor) -> torch.Tensor:
    """(dy/dx)^T g_y of cvf::align_fwd.  No autograd formula of its own: differentiating it again raises."""
    check_align_args(x, ref, align_idx, "cvf::align_vjp")
    if g_y.shape != x.shape or g_y.dtype != torch.float32 or not g_y.is_contiguous() or g_y.device != x.device:
        raise RuntimeError("cvf::align_vjp: g_y must be a contiguous float32 tensor of the frames' shape and device")
    g_x = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().cvf_align_vjp(x.data_ptr(), x.shape[0], x.shape[1], align_idx.data_ptr(), align_idx.numel(),
                                            ref.data_ptr(), g_y.data_ptr(), g_x.data_ptr(), _stream()), "cvf_align_vjp")
    return g_x


@align_vjp_op.register_fake
def _(x, ref, align_idx, g_y):
    return torch.empty_like(x)


def _align_fwd_setup(ctx, inputs, output):
    x, ref, align_idx = inputs
    ctx.save_for_backward(x, ref, align_idx)


def _align_fwd_backward(ctx, g_y):
    x, ref, align_idx = ctx.saved_tensors
    # the cotangent of .sum() and friends is an expanded view (stride 0): the kernel reads dense frames
    return align_vjp_op(x, ref, align_idx, g_y.contiguous()), None, None


align_fwd_op.register_autograd(_align_fwd_backward, setup_context=_align_fwd_setup)


# ------------------------------------------------------------------------------------------ features
# ``handle`` names a PreprocSpec (PreprocSpec.handle).  utils.FeatureMap builds a temporary Preprocessing, and
# with it a temporary spec, on every call: the autograd context keeps the spec alive until backward has run, and backward uses
# that same spec -- alignment_elided included -- so it differentiates the function the forward computed.
@torch.library.custom_op("cvf::features_fwd", mutates_args=())
def features_fwd_op(x: torch.Tensor, handle: int) -> torch.Tensor:
    spec = _context(handle)
    r = torch.empty(x.shape[0], spec.d_r, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().cvf_features_fwd(x.data_ptr(), x.shape[0], spec.struct_ptr(), r.data_ptr(), _stream()),
                   "cvf_features_fwd")
    return r


@features_fwd_op.register_fake
def _(x, handle):
    return x.new_empty((x.shape[0], _context(handle).d_r))


@torch.library.custom_op("cvf::features_vjp", mutates_args=())
def features_vjp_op(x: torch.Tensor, g_r: torch.Tensor, handle: int) -> torch.Tensor:
    """(dr/dx)^T g_r of cvf::features_fwd.  No autograd formula of its own: differentiating it again raises."""
    spec = _context(handle)
    if tuple(g_r.shape) != (x.shape[0], spec.d_r) or g_r.dtype != torch.float32 or not g_r.is_contiguous() or g_r.device != x.device:
        raise RuntimeError(f"cvf::features_vjp: g_r must be a contiguous float32 [{x.shape[0]},{spec.d_r}] tensor on the frames' device")
    g_x = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().cvf_features_vjp(x.data_ptr(), x.shape[0], spec.struct_ptr(), g_r.data_ptr(), g_x.data_ptr(),
                                               _stream()), "cvf_features_vjp")
    return g_x


@features_vjp_op.register_fake
def _(x, g_r, handle):
    return torch.empty_like(x)


def _features_fwd_setup(ctx, inputs, output):
    x, handle = inputs
    ctx.save_for_backward(x)
    ctx.handle = handle
    ctx.spec = _context(handle)      # strong reference: the registry only holds weak ones


def _features_fwd_backward(ctx, g_r):
    x, = ctx.saved_tensors
    return features_vjp_op(x, g_r.contiguous(), ctx.handle), None


features_fwd_op.register_autograd(_features_fwd_backward, setup_context=_features_fwd_setup)
