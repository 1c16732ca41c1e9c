"""HOP_MODE_VERIFIED at the LQR boundary (hop_select_verified_f64) on the host: the near-tie scan on the minimised curve
J + w t against a numpy restatement built on oracle/census.py argmin_gap, the list mode of the generic EXACT kernel against
the full EXACT emulation, and the argument checks of the C-ABI and of the Python entry point, which need no device.
The GPU runs of the same entry point are in tests/test_verified_lqr_gpu.py."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import emul
from _common import perstep_problem
from hop import _cabi, api
from oracle import census

_HERE = os.path.dirname(os.path.abspath(__file__))
_EMUL = os.path.join(_HERE, "emul")
_CSRC = os.path.join(os.path.dirname(_HERE), "time-opt-ilqr_b200", "csrc")
_ip = C.POINTER(C.c_int)
_dp = C.POINTER(C.c_double)
FAST_DM = [(3, 1), (4, 2), (5, 1), (12, 4), (13, 4)]     # hop_select_supported


class TieScanArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("T_min", C.c_int), ("T_max", C.c_int), ("tol", C.c_double), ("J", _dp), ("T_star", _ip),
                ("status", _ip), ("skip", _ip)]


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(tempfile.mkdtemp(prefix="hop_emul_verify_lqr_"), "libhop_emul_verify_lqr.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-DHOP_HOST_EMUL", "-Wno-unknown-pragmas", "-I" + _EMUL, "-I" + _CSRC,
                           "-fPIC", "-shared", "-o", out, os.path.join(_EMUL, "simt_emul.cpp"),
                           os.path.join(_EMUL, "emul_verify_lqr.cpp")])
    return C.CDLL(out)


def tie_scan_w(lib, J, w, T, st, T_min, T_max, tol):
    J = np.ascontiguousarray(J[:, :T_max], dtype=np.float64)
    w = np.ascontiguousarray(w, dtype=np.float64)
    T = np.ascontiguousarray(T, dtype=np.int32); st = np.ascontiguousarray(st, dtype=np.int32)
    B = J.shape[0]
    a = TieScanArgs(B, T_min, T_max, tol, J.ctypes.data_as(_dp), T.ctypes.data_as(_ip), st.ctypes.data_as(_ip), None)
    lst = np.full(B, -1, np.int32); cnt = C.c_int(0)
    assert lib.emul_tie_scan_w(C.byref(a), w.ctypes.data_as(_dp), lst.ctypes.data_as(_ip), C.byref(cnt)) == 0
    return lst[:cnt.value]


def minimised(J, w):
    """v(t) = J(t) + w t with numpy's two roundings (w * t, then the sum), the EXACT body's add_rn(J, mul_rn(w, t))."""
    t = np.arange(1, J.shape[1] + 1, dtype=np.float64)
    return J + w[:, None] * t[None, :]


def scan_numpy(V, T, st, T_min, T_max, tol):
    """include/hop_b200.h, hop_select_verified_f64 step 2, restated with census.argmin_gap on the minimised curve V."""
    W = V[:, T_min - 1:T_max]
    T_scan = np.argmin(W, axis=1) + T_min
    with np.errstate(invalid="ignore", divide="ignore"):
        gap, _ = census.argmin_gap(V, T_scan, T_min, T_max)
        mark = (gap < tol) | ~np.isfinite(W).all(axis=1) | (st != 0) | (T_scan != T)
    return np.nonzero(mark)[0]


def ulp_pair(v1, tol):
    """(v2 with (v2 - v1) / |v1| just below tol, the next double up, whose gap is at or above tol)."""
    hi = v1 * (1.0 + tol)
    while (hi - v1) / abs(v1) >= tol:
        hi = np.nextafter(hi, -np.inf)
    while (hi - v1) / abs(v1) < tol:
        hi = np.nextafter(hi, np.inf)
    return np.nextafter(hi, -np.inf), hi


def raw_for(target, w, t):
    """A raw J(t) with fl(J + fl(w t)) == target exactly (0 < J < target and w t a multiple of 2^-20: target - w t is a
    double, and the sum is exact)."""
    c = w * float(t)
    j = target - c
    for _ in range(64):
        v = j + c
        if v == target:
            return j
        j = np.nextafter(j, np.inf if v < target else -np.inf)
    raise AssertionError("no raw J reaches the target sum")


def synthetic_w(T_min, T_max, tol, seed):
    """Rows whose minimised curve v = J + w t has a unique minimum far from the tolerance and whose raw J slopes down with t
    (so the raw curve's argmin is elsewhere), then one edit per row.  Returns (J, w, T* of v, status, rows by kind)."""
    rng = np.random.default_rng(seed)
    B = 32
    t = np.arange(1, T_max + 1)
    T0 = rng.integers(T_min, T_max + 1, B)
    w = np.round(rng.uniform(0.01, 0.1, B) * 2.0 ** 20) / 2.0 ** 20   # w t exact and on every J grid: targets reachable
    Vd = (1.0 + rng.random(B) + w * T_max)[:, None] * (1.0 + 1e-3 * (t[None, :] - T0[:, None]) ** 2)
    J = Vd - w[:, None] * t[None, :]                             # > 0 and < v, so every v near a target is reachable
    st = np.zeros(B, np.int32)
    kinds = {}

    def v_at(b, col):
        return J[b, col - 1] + w[b] * col

    def set_v(b, col, target):
        J[b, col - 1] = raw_for(target, w[b], col)

    b = 0
    for name, pick in (("v_tie_below", 0), ("v_at_tol", 1)):         # v: one ulp below / at the tolerance; raw J: no tie
        other = T_min if T0[b] != T_min else T_max
        set_v(b, other, ulp_pair(v_at(b, T0[b]), tol)[pick]); kinds[name] = b; b += 1
    # raw J: an exact tie at its own minimum, v: none (the raw minimum lies far from v's, whose curve barely moves)
    ta = int(np.argmin(J[b, T_min - 1:T_max])) + T_min
    tb = ta - 1 if ta > T_min else ta + 1
    J[b, tb - 1] = J[b, ta - 1]; kinds["raw_tie_only"] = b; b += 1
    # v: exact tie, the later horizon is T*; and the earlier one
    set_v(b, T_min if T0[b] != T_min else T_max, v_at(b, T0[b])); kinds["v_exact_tie"] = b; b += 1
    for name, col in (("nan_first", T_min), ("nan_last", T_max)):
        J[b, col - 1] = np.nan; kinds[name] = b; b += 1
    for name, val in (("pinf", np.inf), ("minf", -np.inf)):
        J[b, (T_min + T_max) // 2 - 1] = val; kinds[name] = b; b += 1
    st[b] = 0x200; kinds["lu"] = b; b += 1
    T = T0.astype(np.int32).copy()
    for bb in range(B):                                          # the selection's T*: argmin of v as the kernel computed it
        T[bb] = int(np.argmin(minimised(J[bb:bb + 1], w[bb:bb + 1])[0, T_min - 1:T_max])) + T_min
    T[b] = T[b] + 1 if T[b] < T_max else T[b] - 1; kinds["T_mismatch"] = b; b += 1
    return J, w, T, st, kinds


@pytest.mark.parametrize("tol", [1e-12, 1e-8])
@pytest.mark.parametrize("T_min,T_max", [(5, 100), (1, 31), (40, 128)])
def test_scan_reads_the_minimised_curve(lib, T_min, T_max, tol):
    J, w, T, st, k = synthetic_w(T_min, T_max, tol, seed=T_max)
    V = minimised(J, w)
    want = scan_numpy(V, T, st, T_min, T_max, tol)
    got = tie_scan_w(lib, J, w, T, st, T_min, T_max, tol)
    assert np.array_equal(np.sort(got), want)
    marked = set(want.tolist())
    for name in ("v_tie_below", "v_exact_tie", "nan_first", "nan_last", "pinf", "minf", "lu", "T_mismatch"):
        assert k[name] in marked, name
    assert k["v_at_tol"] not in marked and k["raw_tie_only"] not in marked
    # the raw curve decides otherwise on the designed rows: a scan of J alone (with J's own argmin as T*) marks the raw tie and
    # misses v's
    Tj = (np.argmin(J[:, T_min - 1:T_max], axis=1) + T_min).astype(np.int32)
    raw = set(scan_numpy(J, Tj, st, T_min, T_max, tol).tolist())
    assert k["raw_tie_only"] in raw and k["v_tie_below"] not in raw


def test_scan_without_w_is_the_fused_scan(lib):
    """w = 0 everywhere: v(t) = J(t) + 0 t = J(t), the same decision as the w-less scan."""
    rng = np.random.default_rng(11)
    B, T_min, T_max = 64, 3, 70
    J = 1.0 + rng.random((B, T_max))
    T = (np.argmin(J[:, T_min - 1:], axis=1) + T_min).astype(np.int32)
    for b in range(0, B, 4):                                 # a second horizon 1e-9 above the minimum
        J[b, (T_min if T[b] != T_min else T_max) - 1] = J[b, T[b] - 1] * (1 + 1e-9)
    st = np.zeros(B, np.int32)
    got = tie_scan_w(lib, J, np.zeros(B), T, st, T_min, T_max, 1e-8)
    assert np.array_equal(got, scan_numpy(J, T, st, T_min, T_max, 1e-8)) and got.size > 0


def test_scan_with_a_single_horizon_window(lib):
    rng = np.random.default_rng(3)
    B, T_max = 10, 40
    J = 1.0 + rng.random((B, T_max)); w = rng.uniform(0.01, 0.1, B)
    T = np.full(B, 17, np.int32); st = np.zeros(B, np.int32)
    J[2, 16] = np.nan
    J[3, 16] = -np.inf
    st[4] = 0x100
    J[5, 15] = J[5, 16] + w[5]                               # v(16) == v(17) exactly: outside the window, does not count
    got = tie_scan_w(lib, J, w, T, st, 17, 17, 1e-10)
    want = scan_numpy(minimised(J, w), T, st, 17, 17, 1e-10)
    assert np.array_equal(got, want) and list(want) == [2, 3, 4]


@pytest.mark.parametrize("d,m", FAST_DM)
def test_generic_list_mode_rows_equal_the_full_exact_emulation(lib, d, m):
    """S2 with a per-step R^-1 and w_explicit: the listed instances (given in any order) carry the full EXACT emulation's bits
    plus HOP_ST_FLAG_REEVALUATED, the others keep their sentinels."""
    B, N, T_min = 5, 14, 3
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, B, seed=7 * d + m)
    Jf, Tf, Jsf, stf = emul.select_generic(A, Bm, Q, Rinv, z0, QT, T_min, N, w_explicit=w, ref=True)
    assert not (stf & 0xFF).any()
    listed = np.array([3, 0, 4], np.int32)
    A, Bm, Q, Rinv, z0, w, QT = map(emul._d, (A, Bm, Q, Rinv, z0, w, QT))
    J = np.full((B, N), -123.0); T = np.full(B, -5, np.int32); Js = np.full(B, -7.0); st = np.full(B, 0x7000, np.int32)
    st[listed] = 0
    p = emul._p
    a = emul.SelectArgs(B, N, T_min, N, 1e-9, 8, p(A), p(Bm), p(Q), p(Rinv), p(z0), p(QT), m * m, p(w), p(J),
                        T.ctypes.data_as(_ip), p(Js), st.ctypes.data_as(_ip), None, None, None, 0)
    assert lib.emul_select_generic_ref_list(d, m, C.byref(a), listed.ctypes.data_as(_ip), int(listed.size)) == 0
    for b in range(B):
        if b in listed:
            assert np.array_equal(J[b], Jf[b]) and T[b] == Tf[b] and Js[b] == Jsf[b]
            assert st[b] == (stf[b] | api.ST_FLAG_REEVALUATED)
        else:
            assert (J[b] == -123.0).all() and T[b] == -5 and Js[b] == -7.0 and st[b] == 0x7000


def _call(lib, B=4, N=8, d=13, m=4, T_min=1, T_max=8, stride=0, tol=1e-10):
    return lib.hop_select_verified_f64(B, N, d, m, T_min, T_max, None, None, None, None, stride, None, None, None, tol,
                                       None, None, None, None, None)


def test_abi_rejects_bad_arguments_before_needing_a_device():
    lib = _cabi.load()
    for tol in (0.0, -1.0, float("nan"), float("inf")):
        assert _call(lib, tol=tol) == -1, tol
        assert b"tie_tol" in lib.hop_last_error_string()
    assert _call(lib, d=7, m=3) == -2
    assert _call(lib, d=6, m=2) == -2
    for T_min, T_max in ((0, 8), (5, 4), (1, 9)):
        assert _call(lib, T_min=T_min, T_max=T_max) == -1
    assert _call(lib, B=-1) == -1 and _call(lib, N=0, T_max=0) == -1
    assert _call(lib, stride=3) == -1
    # unchanged: the mode-taking entry point keeps refusing VERIFIED, and the per-mode answers stay those of the fused forms
    assert lib.hop_select_f64(1, 8, 13, 4, 1, 8, None, None, None, None, 0, None, None, None, api.MODE_VERIFIED, None, None,
                              None, None, None) == -1
    assert lib.hop_select_supported_mode(4, 2, api.MODE_VERIFIED) == 0 and lib.hop_select_supported_mode(3, 1, api.MODE_VERIFIED) == 1


def test_python_entry_needs_a_tolerance_exactly_with_verified():
    z = np.zeros((1, 2, 3, 3))
    args = (z, np.zeros((1, 2, 3, 1)), z, np.eye(1), np.zeros(3), z)
    for tol in (None, 0.0, -1e-9, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="tie_tol"):
            api.propagator_all_Jt_aug_batched(*args, mode=api.MODE_VERIFIED, tie_tol=tol)
    for mode in (api.MODE_EXACT, api.MODE_FAST):
        with pytest.raises(ValueError, match="tie_tol"):
            api.propagator_all_Jt_aug_batched(*args, mode=mode, tie_tol=1e-10)
