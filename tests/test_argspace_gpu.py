"""GPU: the selection kernels and their helpers over the argument space include/hop_b200.h documents, through the C-ABI.

  - a different R^-1 per step (R_inv [B][N][m][m]) on every kernel hop_select_f64 routes to, and through the drop-in;
  - HOP_MODE_EXACT / HOP_MODE_FP32 at (d, m) the four cases never reach, at both launch shapes of the EXACT kernel;
  - fused EXACT at odd (n, m), with a non-finite and a jitter-ladder instance;
  - the batched hop_chol_inv_f64 / hop_chol_solve_f64 for every d <= 16;
  - the T* edges of hop_cost_f64, hop_backward_linesearch_f64 and the stand-alone hop_linesearch_f64.
Every test hook a test sets is restored in a finally block.  The emulated run of the first three is
tests/test_argspace_cpu.py, whose module docstring explains the two references of per-step R^-1."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O
from _common import (CASE_NAMES, FUSED_NM, fused_batch, fused_oracle, golden, perstep_problem, perstep_R, reference_b, rel,
                     s2_batch)
from hop import _cabi, api, cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SMS = 148                            # B200: the full-SM launch branch of the EXACT kernel starts at (warps per CTA) * SMs


def _t(a):
    return torch.as_tensor(np.ascontiguousarray(a), device=DEV)


def _np(sel):
    return tuple(x.cpu().numpy() for x in (sel.J, sel.T_star, sel.J_star, sel.status))


def _select(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w, mode):
    return _np(api.propagator_all_Jt_aug_batched(_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), T_min, T_max,
                                                 w_explicit=_t(w), mode=mode))


def _perstep_reference(A, Bm, Q, Rinv, z0, QT, T_max, independent=True):
    """The oracle's per-step curve; with `independent`, also checked against the single-R^-1 reformulation (fp80)."""
    Jo, sto = O.propagator_batch(A, Bm, Q, Rinv, z0, QT, T_use=T_max, nthreads=8)
    assert not sto.any()
    if independent:
        assert rel(Jo, reference_b(A, Bm, Q, Rinv, z0, QT, T_max, f80=True)) <= 1e-12
    return Jo


def _check(out, Jo, w, T_min, tol, exact=False):
    J, T, Js, st = out
    assert not st.any()
    if exact:
        assert np.array_equal(J, Jo)
    assert rel(J, Jo) <= tol
    T_max = Jo.shape[1]
    tot = Jo + w[:, None] * np.arange(1, T_max + 1)
    To = np.argmin(tot[:, T_min - 1:], axis=1) + T_min
    assert np.array_equal(T, To)
    if exact:
        assert np.array_equal(Js, tot[np.arange(len(To)), To - 1])


# ------------------------------------------------------------------ per-step R^-1 on every route of hop_select_f64
@pytest.mark.parametrize("d,m", [(3, 1), (4, 2), (5, 1)])
def test_per_step_rinv_small_blocks_every_route(d, m):
    """d <= 5: the thread-per-problem kernel ignores the R^-1 stride, so hop_select_f64 must never route a per-step R^-1 to
    it -- not by default, and not when the batch threshold is forced to 0.  Every route must equal the reference and the
    lane-group kernel bit for bit.  70 instances: a ragged last warp."""
    N, B, T_min, T_max = 24, 70, 2, 23
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, B)
    Jo = _perstep_reference(A, Bm, Q, Rinv, z0, QT, T_max)
    lib = _cabi.require_device()
    out = {}
    old = lib.hop_test_set_tpp_min_batch(-2)
    try:
        for name, thr in (("default", -1), ("lanes", 1 << 40), ("forced_tpp", 0)):
            lib.hop_test_set_tpp_min_batch(thr)
            for mode in (api.MODE_FAST, api.MODE_GJ):
                out[name, mode] = _select(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w, mode)
    finally:
        lib.hop_test_set_tpp_min_batch(old)
    for key, o in out.items():
        _check(o, Jo, w, T_min, 1e-9)
        for a, b in zip(o, out["lanes", key[1]]):
            assert np.array_equal(a, b), key


@pytest.mark.parametrize("d", [12, 13])
@pytest.mark.parametrize("mode", ["FAST", "GJ"])
def test_per_step_rinv_large_blocks_pre_pass_and_diagonal_switches(d, mode):
    """d in {12, 13}: the pipelined kernel, with and without the input pre-pass (hop_select.cu offsets R^-1 per chunk there)
    and with diagonal Q / QT blocks inverted element-wise or by the sweep; all four combinations give the same bits."""
    m, N, B, T_min, T_max = 4, 20, 37, 3, 19
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, B)
    Jo = _perstep_reference(A, Bm, Q, Rinv, z0, QT, T_max)
    md = getattr(api, "MODE_" + mode)
    lib = _cabi.require_device()
    out = {}
    old_pre, old_diag = lib.hop_test_set_generic_pre(-1), lib.hop_test_set_generic_diag(1)
    try:
        for pre in (0, 1):
            for diag in (0, 1):
                lib.hop_test_set_generic_pre(pre)
                lib.hop_test_set_generic_diag(diag)
                out[pre, diag] = _select(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w, md)
    finally:
        lib.hop_test_set_generic_pre(old_pre)
        lib.hop_test_set_generic_diag(old_diag)
    for key, o in out.items():
        _check(o, Jo, w, T_min, 1e-9)
        for a, b in zip(o, out[0, 1]):
            assert np.array_equal(a, b), key


def test_per_step_rinv_batch_beyond_the_pre_pass_limit():
    """B = 1 100 > 1 024: the default routing switches the pre-pass off; B = 33 keeps it on.  Both at d = 13 and d = 12."""
    for d, B in ((13, 1100), (12, 1100), (13, 33)):
        N, T_min, T_max = 12, 1, 12
        A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, 4, N, B, seed=7)
        Jo = _perstep_reference(A, Bm, Q, Rinv, z0, QT, T_max, independent=B < 100)
        for mode in (api.MODE_FAST, api.MODE_EXACT):
            _check(_select(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w, mode), Jo, w, T_min, 1e-9,
                   exact=mode == api.MODE_EXACT)


@pytest.mark.parametrize("d", [12, 13])
def test_per_step_rinv_scan_mode(d):
    N, B, T_max = 27, 5, 27
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, 4, N, B)
    Jo = _perstep_reference(A, Bm, Q, Rinv, z0, QT, T_max)
    _check(_select(A, Bm, Q, Rinv, z0, QT, 1, T_max, w, api.MODE_SCAN), Jo, w, 1, 1e-9)


@pytest.mark.parametrize("d,m", [(1, 1), (3, 1), (4, 7), (8, 3), (13, 4), (16, 16)])
def test_per_step_rinv_exact_and_fp32(d, m):
    """EXACT: bit-identical to the oracle's per-step path (J, T*, J*).  FP32: within its stated 1e-4."""
    N, B, T_min, T_max = 14, 9, 2, 13
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, B)
    Jo = _perstep_reference(A, Bm, Q, Rinv, z0, QT, T_max)
    _check(_select(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w, api.MODE_EXACT), Jo, w, T_min, 0.0, exact=True)
    J32, _, _, st32 = _select(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w, api.MODE_FP32)
    assert not st32.any() and rel(J32, Jo) <= 1e-4


def test_dropin_propagator_with_a_varying_R_list():
    """horizon_selection.propagator_all_Jt_aug without R_inv_cached and with R_list varying over k sends a per-step R^-1."""
    import importlib
    import os
    import sys
    dropin = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "time-opt-ilqr_b200", "dropin")
    sys.path.insert(0, dropin)
    try:
        hs = importlib.import_module("horizon_selection")
    finally:
        sys.path.remove(dropin)
    d, m, N = 13, 4, 16
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, 1)
    R = perstep_R(100, 1, N, m)[0]
    J = hs.propagator_all_Jt_aug(list(A[0]), list(Bm[0]), list(Q[0]), list(R), z0[0], list(QT[0]))
    Jo = O.propagator_all_Jt(A[0], Bm[0], Q[0], Rinv[0], z0[0], QT[0])
    assert rel(J, Jo) <= 1e-12
    J6 = hs.propagator_all_Jt_aug(list(A[0]), list(Bm[0]), list(Q[0]), list(R), z0[0], list(QT[0]), T_use=6)
    assert rel(J6, Jo[:6]) <= 1e-12
    J1 = hs.propagator_all_Jt_aug(list(A[0]), list(Bm[0]), list(Q[0]), [R[0]] * N, z0[0], list(QT[0]))
    assert rel(J1, Jo) > 1e-3                                           # the R_k matter


# ------------------------------------------------------------------ EXACT / FP32 over (d, m)
DM = sorted({(d, m) for d in (1, 2, 6, 7, 8, 9, 10, 11, 14, 15, 16) for m in (1, d, 16)})
FP32_DIST = {}


@pytest.mark.parametrize("d,m", DM, ids=[f"{d}x{m}" for d, m in DM])
def test_exact_and_fp32_over_block_sizes(d, m):
    """S2 at (d, m) the cases never reach (m > d, m = 16, d = 16 included).  B = 5 takes the `spread` branch of the EXACT
    launch (few warps per CTA); B = 148 * 16 + 3 fills every SM at any slab size and leaves a ragged last CTA.  EXACT is
    bit-identical to the oracle with T*, J* as np.argmin of J(t) + w t; FP32 stays within 1e-4 of EXACT and changes T* only
    where EXACT's argmin gap is below that."""
    N = 8 + (d + m) % 9
    worst = 0.0
    for B in (5, SMS * 16 + 3):
        A, Bm, Q, R, z0, w, QT = s2_batch(range(B), d, m, N)
        Rinv = np.stack([O.chol_inv(r) for r in R])
        Jo, sto = O.propagator_batch(A, Bm, Q, Rinv, z0, QT, nthreads=8)
        assert not sto.any()
        ex = _select(A, Bm, Q, Rinv, z0, QT, 1, N, w, api.MODE_EXACT)
        _check(ex, Jo, w, 1, 0.0, exact=True)
        J32, T32, _, st32 = _select(A, Bm, Q, Rinv, z0, QT, 1, N, w, api.MODE_FP32)
        assert not st32.any()
        worst = max(worst, rel(J32, Jo))
        tot = Jo + w[:, None] * np.arange(1, N + 1)
        for i in np.nonzero(T32 != ex[1])[0]:
            a, b = tot[i, ex[1][i] - 1], tot[i, T32[i] - 1]
            assert abs(b - a) <= 1e-4 * abs(a), (i, ex[1][i], T32[i])
    FP32_DIST[d, m] = worst
    print(f"\nFP32 vs EXACT (d, m) = ({d}, {m}), N = {N}: max relative distance {worst:.3e}")
    assert worst <= 1e-4


# ------------------------------------------------------------------ fused EXACT at odd (n, m)
@pytest.mark.parametrize("n,m", FUSED_NM)
def test_fused_exact_at_odd_dimensions(n, m):
    """Bit-identical to the oracle.  Instance 1 has a NaN in A at step 3 (status 1, the curve NaN from t = 4 on, T* = 4 as
    np.argmin lets NaN win); instance 2 has w < 0, so the first augmented stage block needs the jitter ladder (0x100)."""
    N, B, T_min, T_max = 7, 5, 2, 6
    g = fused_batch(10 * n + m, B, n, m, N)
    g["A"][1, 3, 0, 0] = np.nan
    g["w"][2] = -1e-6
    sel = api.select_fused_batched(_t(g["A"]), _t(g["Bm"]), _t(g["X"]), _t(g["U"]), _t(g["xg"]), _t(g["w"]), g["u_ref"],
                                   g["Q"], g["R"], g["alpha"], T_min, T_max, g["wrap_idx"], a_resid=_t(g["a"]),
                                   mode=api.MODE_EXACT)
    J, T, Js, st = _np(sel)
    assert st[1] == 1 and st[2] == 0x100 and st[0] == 0 and st[3] == 0 and st[4] == 0
    ok = [0, 2, 3, 4]
    sub = {k: (v[ok] if k in ("A", "Bm", "X", "xg", "w", "a") else v) for k, v in g.items()}
    Jo, To = fused_oracle(sub, T_min, T_max)
    assert np.array_equal(J[ok], Jo) and np.array_equal(T[ok], To)
    assert np.array_equal(Js[ok], Jo[np.arange(len(ok)), To - 1])
    Jp, _ = O.select_fused(g["A"][1, :3], g["Bm"][1, :3], g["X"][1, :4], g["U"][:3], g["xg"][1], g["u_ref"], g["Q"], g["R"],
                           g["alpha"], g["w"][1], 1, 3, g["wrap_idx"], a_resid=g["a"][1, :3])
    assert np.array_equal(J[1, :3], Jp) and np.isnan(J[1, 3:]).all() and T[1] == 4


# ------------------------------------------------------------------ batched chol_inv / chol_solve
def _chol_batch(d, rng, B=300):
    """SPD, ladder-needing (one eigenvalue -1e-6), never PD (-I: the LU fallback of the inverse) and NaN matrices, mixed."""
    A = np.empty((B, d, d))
    kinds = np.arange(B) % 6
    for i in range(B):
        M = rng.standard_normal((d, d))
        S = M @ M.T / d + 0.5 * np.eye(d)
        if kinds[i] == 3:                                   # PD again once the jitter exceeds 1e-6
            V, _ = np.linalg.qr(rng.standard_normal((d, d)))
            ev = rng.uniform(0.5, 2.0, d); ev[0] = -1e-6
            S = (V * ev) @ V.T
        elif kinds[i] == 4:
            S = -np.eye(d) - 0.1 * (M @ M.T) / d
        elif kinds[i] == 5:
            S[rng.integers(d), rng.integers(d)] = np.nan
        E = 1e-3 * rng.standard_normal((d, d))
        A[i] = S if kinds[i] == 5 else S + (E - E.T)        # not symmetric (sym() is part of the op), same symmetric part
    return A, kinds


def _oracle_status(rc, info, max_tries=8):
    if rc == O.HOP_ERR_NONFINITE:
        return 1
    return rc | (0x100 if info > 0 else 0) | (0x200 if info >= max_tries else 0)


CHOL_BITS = {}


@pytest.mark.parametrize("d", range(1, 17))
def test_batched_chol_inv_and_chol_solve(d):
    """hop_chol_inv_f64 / hop_chol_solve_f64 (one thread per matrix) against O.chol_inv / O.chol_solve: the exact status word
    and 1e-12 on the values; whether the values are also bit-identical is printed (the device and the oracle follow the same
    operation order; the device may contract a product and a sum into one FMA)."""
    lib = _cabi.require_device()
    rng = np.random.default_rng(d)
    A, kinds = _chol_batch(d, rng)
    B = A.shape[0]
    Ad = _t(A)
    X = torch.full((B, d, d), -7.0, dtype=torch.float64, device=DEV)
    st = torch.full((B,), -1, dtype=torch.int32, device=DEV)
    _cabi.check(lib.hop_chol_inv_f64(B, d, C.c_void_p(Ad.data_ptr()), C.c_void_p(X.data_ptr()), 1e-9, 8,
                                     C.c_void_p(st.data_ptr()), None), "hop_chol_inv_f64")
    torch.cuda.synchronize()
    X, st = X.cpu().numpy(), st.cpu().numpy()
    same = True
    seen = set()
    for i in range(B):
        Xo = np.empty((d, d)); info = C.c_int(0)
        rc = O.lib().hopo_chol_inv(d, O._p(O._d(A[i])), O._p(Xo), C.c_double(1e-9), 8, C.byref(info))
        so = _oracle_status(rc, info.value)
        assert st[i] == so, (i, kinds[i], hex(st[i]), hex(so))
        seen.add(so)
        if rc == 0:
            assert np.abs(X[i] - Xo).max() <= 1e-12 * np.abs(Xo).max(), (i, kinds[i])
            same = same and np.array_equal(X[i], Xo)
    assert {0, 1, 0x300} <= seen and (d == 1 or 0x100 in seen)
    for c in sorted({1, d, 16}):
        Bm = rng.standard_normal((B, d, c))
        Bd = _t(Bm)
        Y = torch.full((B, d, c), -7.0, dtype=torch.float64, device=DEV)
        st = torch.full((B,), -1, dtype=torch.int32, device=DEV)
        _cabi.check(lib.hop_chol_solve_f64(B, d, c, C.c_void_p(Ad.data_ptr()), C.c_void_p(Bd.data_ptr()),
                                           C.c_void_p(Y.data_ptr()), 1e-9, 8, C.c_void_p(st.data_ptr()), None),
                    "hop_chol_solve_f64")
        torch.cuda.synchronize()
        Y, st = Y.cpu().numpy(), st.cpu().numpy()
        for i in range(B):
            Yo = np.empty((d, c)); info = C.c_int(0)
            rc = O.lib().hopo_chol_solve(d, c, O._p(O._d(A[i])), O._p(O._d(Bm[i])), O._p(Yo), C.c_double(1e-9), 8)
            if rc == O.HOP_ERR_NONFINITE:
                assert st[i] == 1, (i, c)
            elif rc == O.HOP_ERR_LINALG:
                assert st[i] == 0x102, (i, c, hex(st[i]))           # every try failed: ladder flag + LinAlgError
            else:
                assert (st[i] & 0xFF) == 0 and ((st[i] == 0x100) == (kinds[i] == 3)), (i, c, hex(st[i]))
                assert np.abs(Y[i] - Yo).max() <= 1e-12 * np.abs(Yo).max(), (i, c)
                same = same and np.array_equal(Y[i], Yo)
    CHOL_BITS[d] = same
    print(f"\nchol_inv / chol_solve d = {d}: values bit-identical to the oracle: {same}")


# ------------------------------------------------------------------ T* edges of the HOP-DDP pieces
def _case_arrays(name, B):
    g = golden("case_" + name)
    case = cases.make_case(name, N=int(g["N"]))
    rep = lambda a: np.repeat(a[None], B, 0)                                        # noqa: E731
    return g, case, int(g["N"]), rep(g["A_fwd"]), rep(g["B_fwd"]), rep(g["X"]), rep(g["U"])


@pytest.mark.parametrize("name", CASE_NAMES)
def test_cost_and_backward_pass_at_horizon_edges(name):
    """T* > N is clamped to N; T* <= 0 gives cost = inf and ok = 0; the backward pass leaves every row >= T* of k / K as the
    caller filled it (a NaN sentinel here)."""
    g, case, N, A, Bm, X, U = _case_arrays(name, 5)
    F, x0, xg, u_ref, Q, R, alpha, w, *_ = case
    n, m = x0.size, u_ref.size
    Ts = np.array([-1, 0, 1, N, N + 5], np.int32)
    J = api.cost_timeopt_true_batched(case, _t(X), _t(U), torch.as_tensor(Ts)).cpu().numpy()
    for i, T in enumerate(Ts):
        Jo = O.cost_timeopt_true(X[i], U[i], xg, u_ref, Q, R, alpha, w, min(T, N), case[11])
        if T <= 0:
            assert J[i] == np.inf and Jo == np.inf
        else:
            assert abs(J[i] - Jo) <= 1e-12 * abs(Jo), (T, J[i], Jo)
    lib = _cabi.require_device()
    c = api._case_consts(case, 5, torch.device(DEV))
    k = torch.full((5, N, m), np.nan, dtype=torch.float64, device=DEV)
    K = torch.full((5, N, m, n), np.nan, dtype=torch.float64, device=DEV)
    i32 = lambda v: torch.full((5,), v, dtype=torch.int32, device=DEV)             # noqa: E731
    ok, err, acc = i32(-1), i32(-1), i32(-1)
    Xn, Un = torch.empty((5, N + 1, n), dtype=torch.float64, device=DEV), torch.empty((5, N, m), dtype=torch.float64, device=DEV)
    Jn, lm, Td = torch.empty(5, dtype=torch.float64, device=DEV), _t(np.full(5, 1e-3)), _t(Ts)
    Ad, Bd, Xd, Ud = _t(A), _t(Bm), _t(X), _t(U)
    p = lambda t: C.c_void_p(t.data_ptr())                                          # noqa: E731
    _cabi.check(lib.hop_backward_linesearch_f64(5, F.hop_sys, c["params"].ctypes.data_as(C.c_void_p), N, p(Ad), p(Bd), p(Xd),
                                                p(Ud), p(c["xg"]), p(c["w"]), p(c["u_ref"]), p(c["Q"]), p(c["R"]), p(c["Qf"]),
                                                c["wrap"], p(Td), p(lm), p(k), p(K), p(ok), p(err), p(Xn), p(Un), p(Jn), p(acc),
                                                None), "hop_backward_linesearch_f64")
    torch.cuda.synchronize()
    k, K, ok, err = k.cpu().numpy(), K.cpu().numpy(), ok.cpu().numpy(), err.cpu().numpy()
    assert not err.any()
    for i, T in enumerate(Ts):
        Tc = min(T, N)
        if T <= 0:
            assert ok[i] == 0 and np.isnan(k[i]).all() and np.isnan(K[i]).all()
            continue
        ko, Ko, oko = O.backward_pass(A[i], Bm[i], X[i], U[i], xg, u_ref, Q, R, alpha, Tc, 1e-3, case[11])
        assert ok[i] == int(oko)
        assert np.isnan(k[i, Tc:]).all() and np.isnan(K[i, Tc:]).all()
        if oko:
            assert np.abs(k[i, :Tc] - ko).max() <= 1e-9 * np.abs(ko).max()
            assert np.abs(K[i, :Tc] - Ko).max() <= 1e-9 * np.abs(Ko).max()


@pytest.mark.parametrize("name", CASE_NAMES)
def test_standalone_linesearch_with_an_ok_mask(name):
    """hop_linesearch_f64 with the gains of the fused entry point and ok = [1, 0, 1, 0, 1] (and the backward pass's ok),
    horizons T0, T0 / 2 and N + 3 (clamped to N).  Masked instances keep their sentinels in X_new, U_new, J_new and report
    accepted = 0 (include/hop_b200.h); the others equal the fused entry point's line search bit for bit and the oracle's
    forward_linesearch, in both line-search kernels (five step sizes side by side / one thread trying them in turn)."""
    B = 5
    g, case, N, A, Bm, X, U = _case_arrays(name, B)
    F, x0, xg, u_ref, Q, R, alpha, w, *_ = case
    n, m = x0.size, u_ref.size
    T0 = int(g["T0"])
    Ts = np.array([T0, T0, max(1, T0 // 2), T0, N + 3], np.int32)
    lib = _cabi.require_device()
    c = api._case_consts(case, B, torch.device(DEV))
    p = lambda t: C.c_void_p(t.data_ptr())                                          # noqa: E731
    mask = np.array([1, 0, 1, 0, 1], np.int32)
    r = api.backward_linesearch_batched(case, _t(A), _t(Bm), _t(X), _t(U), torch.as_tensor(Ts), 1e-3)
    mask &= r["ok"].cpu().numpy().astype(np.int32)         # the fused entry point leaves the outputs of ok = 0 untouched
    assert mask.sum() >= 2
    res = {}
    old = lib.hop_test_set_linesearch_variant(0)
    try:
        for variant in (0, 1):
            lib.hop_test_set_linesearch_variant(variant)
            r = api.backward_linesearch_batched(case, _t(A), _t(Bm), _t(X), _t(U), torch.as_tensor(Ts), 1e-3)
            Xn = torch.full((B, N + 1, n), -7.0, dtype=torch.float64, device=DEV)
            Un = torch.full((B, N, m), -7.0, dtype=torch.float64, device=DEV)
            Jn = torch.full((B,), -7.0, dtype=torch.float64, device=DEV)
            acc = torch.full((B,), -7, dtype=torch.int32, device=DEV)
            Td, okd, Xd, Ud = _t(Ts), _t(mask), _t(X), _t(U)
            _cabi.check(lib.hop_linesearch_f64(B, F.hop_sys, c["params"].ctypes.data_as(C.c_void_p), N, p(Xd), p(Ud), p(c["xg"]),
                                               p(c["w"]), p(c["u_ref"]), p(c["Q"]), p(c["R"]), p(c["Qf"]), c["wrap"], p(Td),
                                               p(r["k"]), p(r["K"]), p(okd), p(Xn), p(Un), p(Jn), p(acc), None), "hop_linesearch_f64")
            torch.cuda.synchronize()
            res[variant] = {key: v.cpu().numpy() for key, v in (("X_new", Xn), ("U_new", Un), ("J_new", Jn), ("accepted", acc))}
            res[variant]["fused"] = {key: r[key].cpu().numpy() for key in ("X_new", "U_new", "J_new", "accepted", "k", "K")}
    finally:
        lib.hop_test_set_linesearch_variant(old)
    for variant, o in res.items():
        f = o["fused"]
        for i in range(B):
            if not mask[i]:
                assert (o["X_new"][i] == -7.0).all() and (o["U_new"][i] == -7.0).all() and o["J_new"][i] == -7.0
                assert o["accepted"][i] == 0                  # a skipped instance is reported as not accepted
                continue
            for key in ("X_new", "U_new", "J_new", "accepted"):
                assert np.array_equal(o[key][i], f[key][i]), (variant, i, key)
            Tc = min(int(Ts[i]), N)
            Xo, Uo, Jo, acco = O.forward_linesearch(F.hop_sys, F.hop_params, X[i], U[i], xg, u_ref, Q, R, alpha, w, Tc,
                                                    f["k"][i, :Tc], f["K"][i, :Tc], case[11])
            assert bool(o["accepted"][i]) == acco
            assert abs(o["J_new"][i] - Jo) <= 1e-9 * abs(Jo)
            assert np.abs(o["U_new"][i] - Uo).max() <= 1e-8 * max(1.0, np.abs(Uo).max())
    for key in ("X_new", "U_new", "J_new", "accepted"):
        assert np.array_equal(res[0][key], res[1][key]), key
