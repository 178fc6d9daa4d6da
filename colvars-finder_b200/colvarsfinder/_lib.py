"""ctypes binding of libcvf_sm100.so (C ABI declared in include/cvf.h).

The library is the only compute backend of this package: there is no CPU or PyTorch fallback.  If the
shared object is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcvf_sm100.so")

MAX_LAYERS = 8
MAX_K = 8

FEAT_POSITION, FEAT_BOND, FEAT_ANGLE, FEAT_DIHEDRAL = 0, 1, 2, 3


class Preproc(C.Structure):
    """struct cvf_preproc (include/cvf.h)."""
    _fields_ = [("kind", C.c_int32), ("dim", C.c_int32), ("n_atoms", C.c_int32), ("n_used", C.c_int32),
                ("used_atoms", C.c_void_p), ("n_align", C.c_int32), ("align_used", C.c_void_p), ("ref", C.c_void_p),
                ("n_feat", C.c_int32), ("feat", C.c_void_p), ("d_r", C.c_int32), ("positions_only", C.c_int32), ("used_identity", C.c_int32),
                ("diag", C.c_void_p), ("n_feat_by_type", C.c_int32 * 4), ("n_self_records", C.c_int32), ("n_shared_atoms", C.c_int32)]


class Mlp(C.Structure):
    """struct cvf_mlp (include/cvf.h)."""
    _fields_ = [("n_layers", C.c_int32), ("dims", C.c_int32 * (MAX_LAYERS + 1)), ("act", C.c_int32 * MAX_LAYERS)]


# every symbol include/cvf.h declares: name -> (restype, argtypes)
_P, _I64, _I32, _D, _SZ = C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_size_t
SYMBOLS = {
    "cvf_version": (C.c_int, []),
    "cvf_source_hash": (C.c_char_p, []),
    "cvf_last_error_string": (C.c_char_p, []),
    "cvf_sizeof_preproc": (_SZ, []),
    "cvf_sizeof_mlp": (_SZ, []),
    "cvf_mlp_param_count": (_I64, [C.POINTER(Mlp)]),
    "cvf_align_fwd": (C.c_int, [_P, _I64, _I32, _P, _I32, _P, _P, _P, _P, _P]),
    "cvf_features_fwd": (C.c_int, [_P, _I64, C.POINTER(Preproc), _P, _P]),
    "cvf_align_vjp": (C.c_int, [_P, _I64, _I32, _P, _I32, _P, _P, _P, _P]),
    "cvf_features_vjp": (C.c_int, [_P, _I64, C.POINTER(Preproc), _P, _P, _P]),
    "cvf_eigen_num_stats": (_I32, [_I32]),
    "cvf_eigen_num_combine": (_I32, [_I32]),
    "cvf_eigen_workspace_bytes": (_SZ, [C.POINTER(Preproc), C.POINTER(Mlp), _I32, _I64]),
    "cvf_eigen_path": (C.c_int, [C.POINTER(Preproc), C.POINTER(Mlp), _I32]),
    "cvf_eigen_set_path": (C.c_int, [_I32]),
    "cvf_eigen_stats": (C.c_int, [_P, _P, _I64, C.POINTER(Preproc), C.POINTER(Mlp), _I32, _P, _P, _P, _P, _SZ, _P]),
    "cvf_eigen_combine": (C.c_int, [_P, _I32, _D, C.POINTER(_D), _D, _I32, _P, _P]),
    "cvf_eigen_grad": (C.c_int, [_P, _P, _I64, C.POINTER(Preproc), C.POINTER(Mlp), _I32, _P, _P, _P, _P, _P, _P, _SZ, _I32, _P]),
    "cvf_eigen_tlag_terms": (C.c_int, [_P, _P, _P, _I64, _I32, _P, _P, _P, _P, _SZ, _P]),
    "cvf_eigen_tlag_combine": (C.c_int, [_P, _P, _P, _I32, _D, C.POINTER(_D), _D, _I32, _P, _P, _P]),
    "cvf_ae_workspace_bytes": (_SZ, [C.POINTER(Mlp), _I64]),
    "cvf_ae_step": (C.c_int, [_P, _P, _I64, C.POINTER(Mlp), _P, _P, _P, _P, _SZ, _P]),
    "cvf_ae_step_target": (C.c_int, [_P, _P, _P, _I64, C.POINTER(Mlp), _P, _P, _P, _P, _SZ, _P]),
    "cvf_ae_set_wide_path": (C.c_int, [_I32]),
    "cvf_ae_set_fast_path": (C.c_int, [_I32]),
    "cvf_weights_filter_workspace_bytes": (_SZ, [_I64]),
    "cvf_weights_filter": (C.c_int, [_P, _I64, _D, _D, _P, _P, _P, _P, _SZ, _P]),
    "cvf_fma_probe": (C.c_int, [_P, _I32, C.POINTER(_D), _P]),
    "cvf_profile_enable": (C.c_int, [_I32]),
    "cvf_profile_num_kernels": (_I32, []),
    "cvf_profile_kernel_name": (C.c_char_p, [_I32]),
    "cvf_profile_read": (C.c_int, [C.POINTER(_D), C.POINTER(_I64), C.POINTER(_I64), _I32]),
}

_lib = None


def lib():
    """Load the shared object once; raise (never fall back) if it is not there."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.cvf_sizeof_preproc() != C.sizeof(Preproc) or handle.cvf_sizeof_mlp() != C.sizeof(Mlp):
            raise RuntimeError(f"{LIB_PATH} was built against a different include/cvf.h (struct sizes differ): rebuild it")
        _lib = handle
    return _lib


def check(code: int, what: str):
    if code != 0:
        msg = lib().cvf_last_error_string().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {code}): {msg}")


def profile_read(reset=True):
    """{kernel name: (summed ms of timed launches, timed launches, launches since last reset)} from the library's accounting."""
    L = lib()
    n = L.cvf_profile_num_kernels()
    ms, timed, launches = (_D * n)(), (_I64 * n)(), (_I64 * n)()
    check(L.cvf_profile_read(ms, timed, launches, 1 if reset else 0), "cvf_profile_read")
    return {L.cvf_profile_kernel_name(i).decode(): (ms[i], int(timed[i]), int(launches[i])) for i in range(n)}


def make_mlp(dims, acts) -> Mlp:
    n = len(dims) - 1
    if n < 1 or n > MAX_LAYERS:
        raise RuntimeError(f"networks with {n} linear layers are outside the supported envelope (1..{MAX_LAYERS})")
    m = Mlp()
    m.n_layers = n
    for i, d in enumerate(dims):
        m.dims[i] = int(d)
    for i, a in enumerate(acts):
        m.act[i] = int(a)
    return m
