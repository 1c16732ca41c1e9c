"""CPU-only checks of the C-ABI library: it loads, exports every symbol include/hop_b200.h declares,
and refuses to compute without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from hop import _cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "hop_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hop_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_and_bound():
    lib = _cabi.load()
    declared = _declared_symbols()
    assert len(declared) >= 12
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in hop_b200.h but not exported"
        assert name in _cabi.SIGNATURES, f"{name} has no ctypes signature in hop/_cabi.py"
    assert sorted(_cabi.SIGNATURES) == declared
    assert lib.hop_abi_version() == 1
    assert b"sm_100a" in lib.hop_version()


def test_supported_dims_table():
    lib = _cabi.load()
    for d, m in ((3, 1), (4, 2), (5, 1), (12, 4), (13, 4)):
        assert lib.hop_select_supported(d, m) == 1
    assert lib.hop_select_supported(7, 3) == 0


_WINDOWS = {   # (B, N, T_min, T_max) that break 1 <= T_min <= T_max <= N, B >= 0
    "T_max > N": (1, 8, 5, 9), "T_min < 1": (1, 8, 0, 4), "T_max < T_min": (1, 8, 5, 4), "N < 1": (1, 0, 1, 1),
    "B < 0": (-1, 8, 1, 8),
}


def _select(lib, B, N, T_min, T_max, rinv_step_stride=0):
    return lib.hop_select_f64(B, N, 13, 4, T_min, T_max, None, None, None, None, rinv_step_stride, None, None, None, 0,
                              None, None, None, None, None)


def _select_verified(lib, B, N, T_min, T_max, rinv_step_stride=0):
    return lib.hop_select_verified_f64(B, N, 13, 4, T_min, T_max, None, None, None, None, rinv_step_stride, None, None,
                                       None, 1e-6, None, None, None, None, None)


def _select_fused(lib, B, N, T_min, T_max):
    return lib.hop_select_fused_f64(B, N, 12, 4, T_min, T_max, *[None] * 5, 0, *[None] * 6, 0, 1e-9, 1e-12, 0,
                                    None, None, None, None, None)


def _ilqr(lib, B, N, T_min, T_max, sys=2):
    return lib.hop_ilqr_timeopt_f64(B, sys, None, N, T_min, T_max, *[None] * 8, 0, 1, 1e-3, 0, 0, None, 0,
                                    *[None] * 11)


def _from_x0(lib, sys):
    return lib.hop_select_from_x0_f64(1, sys, None, 8, 1, 8, None, None, 0, *[None] * 6, 0, 0, 0, None, 1 << 40,
                                      None, None, None, None, None)


def _from_x0_host(lib, sys):
    return lib.hop_select_from_x0_host_f64(1, sys, None, 8, 1, 8, None, None, 0, *[None] * 6, 0, 0, 0,
                                           None, None, None, None)


def _rejections():
    """(case, call, expected return code, expected message prefix, message keyword)"""
    for entry, call in (("hop_select_f64", _select), ("hop_select_verified_f64", _select_verified),
                        ("hop_select_fused_f64", _select_fused), ("hop_ilqr_timeopt_f64", _ilqr)):
        for what, window in _WINDOWS.items():
            yield f"{entry}: {what}", lambda lib, c=call, w=window: c(lib, *w), -1, entry, b"T_max"
    for entry, call in (("hop_select_f64", _select), ("hop_select_verified_f64", _select_verified)):
        yield f"{entry}: rinv_step_stride", lambda lib, c=call: c(lib, 1, 8, 1, 8, rinv_step_stride=3), -1, entry, \
            b"rinv_step_stride"
    for entry, call in (("hop_select_from_x0_f64", _from_x0), ("hop_select_from_x0_host_f64", _from_x0_host),
                        ("hop_ilqr_timeopt_f64", lambda lib, sys: _ilqr(lib, 1, 8, 1, 8, sys=sys))):
        for sys in (-1, 4):
            yield f"{entry}: system {sys}", lambda lib, c=call, s=sys: c(lib, s), -1, entry, b"unknown system id"


def test_bad_arguments_are_rejected_before_any_device_work():
    # every input below is refused with the same code and message whether or not a device is present
    lib = _cabi.load()
    for case, call, code, entry, keyword in _rejections():
        rc = call(lib)
        msg = lib.hop_last_error_string()
        assert rc == code, f"{case}: rc {rc}, message {msg!r}"
        assert msg.startswith(entry.encode() + b":") and keyword in msg, f"{case}: message {msg!r}"


@pytest.mark.skipif(_cabi.load().hop_device_count() > 0, reason="a GPU is present")
def test_no_cpu_fallback_without_a_device():
    lib = _cabi.load()
    rc = lib.hop_select_f64(1, 8, 13, 4, 1, 8, None, None, None, None, 0, None, None, None, 0, None, None, None, None, None)
    assert rc == -3 and b"no CPU fallback" in lib.hop_last_error_string()
    from hop import api
    with pytest.raises(_cabi.HopError):
        api.select_horizon_host(__import__("hop").cases.make_case("Quadrotor", N=128), np.zeros((2, 12)))
