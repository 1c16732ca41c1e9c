"""ctypes binding of libhop_b200.so (include/hop_b200.h).  No torch types cross this boundary:
only raw device pointers (tensor.data_ptr()), sizes and a cudaStream_t."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HOP_LIB") or os.path.join(_HERE, "libhop_b200.so")   # HOP_LIB: experiment builds only

_vp, _d, _i, _l, _u, _ull = C.c_void_p, C.c_double, C.c_int, C.c_long, C.c_uint, C.c_ulonglong

# name -> (restype, argtypes); must list every symbol declared in include/hop_b200.h
SIGNATURES = {
    "hop_abi_version": (_i, []),
    "hop_version": (C.c_char_p, []),
    "hop_last_error_string": (C.c_char_p, []),
    "hop_device_count": (_i, []),
    "hop_select_supported": (_i, [_i, _i]),
    "hop_select_supported_mode": (_i, [_i, _i, _i]),
    "hop_select_f64": (_i, [_i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _l, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "hop_select_verified_f64": (_i, [_i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _l, _vp, _vp, _vp, _d, _vp, _vp, _vp, _vp, _vp]),
    "hop_select_fused_f64": (_i, [_i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _l, _vp, _vp, _vp, _vp, _vp, _vp, _u,
                                  _d, _d, _i, _vp, _vp, _vp, _vp, _vp]),
    "hop_rollout_f64": (_i, [_i, _i, _vp, _i, _vp, _vp, _l, _d, _vp, _vp]),
    "hop_linearize_f64": (_i, [_i, _i, _vp, _i, _vp, _vp, _l, _i, _d, _d, _d, _d, _vp, _vp, _vp]),
    "hop_select_from_x0_workspace_bytes": (_ull, [_i, _i, _i, _i]),
    "hop_select_from_x0_f64": (_i, [_i, _i, _vp, _i, _i, _i, _vp, _vp, _l, _vp, _vp, _vp, _vp, _vp, _vp, _u, _i, _i, _vp,
                                    _ull, _vp, _vp, _vp, _vp, _vp]),
    "hop_select_from_x0_host_f64": (_i, [_i, _i, _vp, _i, _i, _i, _vp, _vp, _l, _vp, _vp, _vp, _vp, _vp, _vp, _u, _i, _i,
                                         _vp, _vp, _vp, _vp]),
    "hop_chol_inv_f64": (_i, [_i, _i, _vp, _vp, _d, _i, _vp, _vp]),
    "hop_chol_solve_f64": (_i, [_i, _i, _i, _vp, _vp, _vp, _d, _i, _vp, _vp]),
    "hop_affine_residuals_f64": (_i, [_i, _i, _vp, _i, _vp, _vp, _l, _vp, _vp]),
    "hop_build_augmented_f64": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _l, _vp, _vp, _vp, _vp, _u, _d, _d, _vp, _vp,
                                     _vp, _vp]),
    "hop_build_terminal_f64": (_i, [_i, _i, _i, _vp, _vp, _vp, _u, _d, _vp, _vp]),
    "hop_cost_f64": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u, _vp, _vp, _vp]),
    "hop_bruteforce_jt_f64": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _l, _vp, _vp, _vp, _vp, _vp, _vp, _u, _d, _vp, _vp, _vp]),
    "hop_backward_linesearch_f64": (_i, [_i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u, _vp, _vp,
                                         _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hop_linesearch_f64": (_i, [_i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp]),
    "hop_ilqr_workspace_bytes": (_ull, [_i, _i, _i, _i]),
    "hop_ilqr_timeopt_f64": (_i, [_i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u, _i, _d, _i, _i, _vp,
                                  _ull, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hop_test_set_linearize_variant": (_i, [_i]),
    "hop_test_set_backward_variant": (_i, [_i]),
    "hop_test_set_linesearch_variant": (_i, [_i]),
    "hop_test_set_fused_small_variant": (_i, [_i]),
    "hop_test_set_generic_pre": (_i, [_i]),
    "hop_test_set_generic_diag": (_i, [_i]),
    "hop_test_set_tpp_min_batch": (_l, [_l]),
    "hop_probe_fp64_tflops": (_i, [_i, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

_lib = None


class HopError(RuntimeError):
    pass


def load():
    """Load the CUDA library.  Fails loudly when it has not been built (no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HopError(f"{LIB_PATH} is missing: build it with `python time-opt-ilqr_b200/csrc/build.py` "
                       "(or __graft_entry__.build()). The HOP B200 path has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.hop_abi_version() != 1:
        raise HopError("libhop_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().hop_last_error_string().decode("utf-8", "replace")
        raise HopError(f"{what} failed (code {rc}): {msg}")


def require_device():
    lib = load()
    if lib.hop_device_count() <= 0:
        raise HopError("no CUDA device visible: the HOP B200 path has no CPU fallback")
    return lib
