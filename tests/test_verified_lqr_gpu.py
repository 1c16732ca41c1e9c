"""HOP_MODE_VERIFIED at the LQR boundary on the device (hop_select_verified_f64 through propagator_all_Jt_aug_batched):
checked against HOP_MODE_EXACT and HOP_MODE_FAST on identical device inputs, on every FAST route of hop_select_f64."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O
from _common import perstep_R, s1_x0
from hop import _cabi, api, cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RE = api.ST_FLAG_REEVALUATED
S2_TOL = 1e-10                 # S2: FAST within 2.7e-14 of EXACT on v (include/hop_b200.h)
QUAD_TOL = 1e-7                # quadrotor embedding at the boundary: FAST within 4.7e-9 (include/hop_b200.h)


def _np(sel):
    return tuple(x.cpu().numpy() for x in (sel.J, sel.T_star, sel.J_star, sel.status))


def _check_against_exact_and_fast(v, e, f):
    """v, e, f = (J, T*, J*, status) of VERIFIED, EXACT, FAST on the same inputs (tests/test_verified_gpu.py).  Returns the
    re-evaluated mask."""
    Jv, Tv, Jsv, stv = v
    Je, Te, Jse, ste = e
    Jf, Tf, Jsf, stf = f
    re = (stv & RE) != 0
    assert np.array_equal(Tv, Te), np.nonzero(Tv != Te)[0][:16]
    assert np.array_equal(stv & 0xFF, ste & 0xFF)
    assert np.array_equal(Jv[re], Je[re], equal_nan=True) and np.array_equal(Jsv[re], Jse[re], equal_nan=True)
    assert np.array_equal(stv[re], ste[re] | RE)
    keep = ~re
    assert np.array_equal(Jv[keep], Jf[keep]) and np.array_equal(Jsv[keep], Jsf[keep]) and np.array_equal(Tv[keep], Tf[keep])
    assert not stv[keep].any() and not stf[keep].any()
    return re


def s2_device(B, d, m, N, seed, perstep=False):
    """S2 as tests/run_configs.py configuration 5 generates it (on the device), optionally with a per-step R^-1."""
    gen = torch.Generator(device=DEV); gen.manual_seed(seed)
    A = torch.eye(d, dtype=torch.float64, device=DEV).expand(B, N, d, d) + \
        0.05 / np.sqrt(d) * torch.randn((B, N, d, d), dtype=torch.float64, device=DEV, generator=gen)
    Bm = 0.05 * torch.randn((B, N, d, m), dtype=torch.float64, device=DEV, generator=gen)
    Q = torch.diag_embed(0.5 + 1.5 * torch.rand((B, N, d), dtype=torch.float64, device=DEV, generator=gen))
    QT = (50.0 * torch.eye(d, dtype=torch.float64, device=DEV)).expand(B, N, d, d).contiguous()
    Rd = 0.05 + 0.45 * torch.rand((B, m), dtype=torch.float64, device=DEV, generator=gen)
    Rinv = torch.diag_embed(1.0 / (Rd + 1e-9))
    if perstep:
        Rinv = torch.as_tensor(np.linalg.inv(perstep_R(seed, B, N, m)), device=DEV)
    z0 = torch.randn((B, d), dtype=torch.float64, device=DEV, generator=gen)
    w = 0.01 + 0.09 * torch.rand((B,), dtype=torch.float64, device=DEV, generator=gen)
    return [A, Bm, Q, Rinv, z0, QT], w


def three(args, T_min, T_max, w, tol):
    run = lambda mode, **k: _np(api.propagator_all_Jt_aug_batched(*args, T_min, T_max, w_explicit=w, mode=mode, **k))  # noqa: E731
    return run(api.MODE_VERIFIED, tie_tol=tol), run(api.MODE_EXACT), run(api.MODE_FAST)


class hooks:
    """Forces a FAST route through the hop_test_set_* hooks and restores the defaults afterwards."""
    def __init__(self, tpp=None, pre=None, diag=None):
        self.set = {"tpp": tpp, "pre": pre, "diag": diag}

    def __enter__(self):
        lib = _cabi.require_device()
        self.old = (lib.hop_test_set_tpp_min_batch(self.set["tpp"] if self.set["tpp"] is not None else -2),
                    lib.hop_test_set_generic_pre(self.set["pre"]) if self.set["pre"] is not None else None,
                    lib.hop_test_set_generic_diag(self.set["diag"]) if self.set["diag"] is not None else None)
        return self

    def __exit__(self, *exc):
        lib = _cabi.require_device()
        lib.hop_test_set_tpp_min_batch(self.old[0])
        if self.old[1] is not None:
            lib.hop_test_set_generic_pre(self.old[1])
        if self.old[2] is not None:
            lib.hop_test_set_generic_diag(self.old[2])


ROUTES = [(3, 1, dict(tpp=0)), (3, 1, dict(tpp=1 << 40)), (4, 2, dict(tpp=0)), (4, 2, dict(tpp=1 << 40)),
          (5, 1, dict(tpp=0)), (5, 1, dict(tpp=1 << 40)),
          (12, 4, dict(pre=0, diag=1)), (12, 4, dict(pre=1, diag=1)), (12, 4, dict(pre=1, diag=0)),
          (13, 4, dict(pre=0, diag=1)), (13, 4, dict(pre=0, diag=0)), (13, 4, dict(pre=1, diag=1))]
RID = ["d3-tpp", "d3-lanes", "d4-tpp", "d4-lanes", "d5-tpp", "d5-lanes", "d12-pipe", "d12-pre", "d12-pre-nodiag",
       "d13-pipe", "d13-pipe-nodiag", "d13-pre"]


@pytest.mark.parametrize("perstep", [False, True], ids=["rinv", "rinv-per-step"])
@pytest.mark.parametrize("with_w", [True, False], ids=["w", "no-w"])
@pytest.mark.parametrize("d,m,route", ROUTES, ids=RID)
def test_every_fast_route_against_exact_and_fast(d, m, route, with_w, perstep):
    B, N, T_min = (3000 if d <= 5 else 1500), 48, 5
    args, w = s2_device(B, d, m, N, seed=17 * d + m + 3 * perstep)
    with hooks(**route):
        v, e, f = three(args, T_min, N, w if with_w else None, S2_TOL)
    re = _check_against_exact_and_fast(v, e, f)
    print(f"\nd={d} {route} w={with_w} per-step={perstep}: re-evaluated {int(re.sum())} of {B}, "
          f"FAST T* != EXACT T* on {int((f[1] != e[1]).sum())}")


@pytest.mark.parametrize("d,m", [(4, 2), (13, 4)])
def test_constructed_ties_are_re_evaluated(d, m):
    """w taken per instance from the EXACT curve so that two adjacent horizons of v = J + w t tie within 1e-13 relative."""
    B, N, T_min = 2048, 48, 3
    args, _ = s2_device(B, d, m, N, seed=91 + d)
    Je = _np(api.propagator_all_Jt_aug_batched(*args, T_min, N, mode=api.MODE_EXACT))[0]
    rng = np.random.default_rng(d)
    t1 = rng.integers(T_min + 2, N - 2, B)
    w = (Je[np.arange(B), t1 - 1] - Je[np.arange(B), t1]) / 1.0            # v(t1) == v(t1 + 1) up to rounding
    wt = torch.as_tensor(w, device=DEV)
    v, e, f = three(args, T_min, N, wt, S2_TOL)
    re = _check_against_exact_and_fast(v, e, f)
    V = Je + w[:, None] * np.arange(1, N + 1)[None, :]
    rows = np.arange(B)
    Te = e[1].astype(np.int64)
    tied = ((Te == t1) | (Te == t1 + 1)) & (np.abs(V[rows, t1 - 1] - V[rows, t1]) <= 1e-13 * np.abs(V[rows, t1]))
    assert tied.sum() > B // 16, int(tied.sum())               # where J is locally convex the tie is v's minimum (13 - 24 %)
    assert re[tied].all(), np.nonzero(tied & ~re)[0][:16]
    print(f"\nd={d}: {int(tied.sum())} constructed ties, all re-evaluated; re-evaluated {int(re.sum())}, "
          f"FAST T* != EXACT T* on {int((f[1] != e[1]).sum())}")


def test_everything_re_evaluated_beyond_one_machine_fill():
    """tie_tol = 1e300 marks every instance; B exceeds one fill of the list-mode grid at d = 13 (19.3 KB slab: at most 11
    one-warp CTAs per SM), so warps take several listed instances (grid stride)."""
    d, m, N, T_min = 13, 4, 24, 2
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 12 * sms + 517
    args, w = s2_device(B, d, m, N, seed=5, perstep=False)
    for wx in (w, None):
        v, e, f = three(args, T_min, N, wx, 1e300)
        re = _check_against_exact_and_fast(v, e, f)
        assert re.all()
        assert np.array_equal(v[0], e[0]) and np.array_equal(v[2], e[2]) and np.array_equal(v[3], e[3] | RE)


@pytest.mark.parametrize("d,m", [(5, 1), (12, 4)])
def test_tiny_tolerance_re_evaluates_only_the_broken_instances(d, m):
    """tie_tol = 1e-300: nothing is a near-tie; only the instances with a NaN block, a forced jitter ladder or a forced LU
    fallback are re-evaluated (their status or window marks them)."""
    B, N, T_min = 1200, 40, 4
    args, w = s2_device(B, d, m, N, seed=23 + d)
    A, Bm, Q = args[0].clone(), args[1], args[2].clone()
    A[7, 11, 0, 1] = float("nan")                               # non-finite input
    Q[100, 3, 1, 1] = -1e-4                                     # Cholesky of Q_3 climbs the jitter ladder
    Q[200, 9, 0, 0] = -1.0                                      # every rung fails: LU fallback
    args = [A, Bm, Q] + args[3:]
    v, e, f = three(args, T_min, N, w, 1e-300)
    re = _check_against_exact_and_fast(v, e, f)
    assert np.nonzero(re)[0].tolist() == [7, 100, 200], np.nonzero(re)[0][:16]
    assert e[3][7] & 0xFF == 1 and e[3][100] & 0x100 and e[3][200] & 0x200


def test_quadrotor_embedding_at_the_documented_tolerance():
    """S1 linearisations materialised at the boundary (hop_build_augmented_f64 / hop_build_terminal_f64), no explicit w:
    T* equals EXACT's on every instance at QUAD_TOL, and two VERIFIED runs are bit-identical."""
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    T_max = min(T_max, N)
    B, n, m = 8192, 12, 4
    sel = api.HorizonSelector(case, B, device=DEV, mode=api.MODE_FAST)
    sel(torch.as_tensor(s1_x0(B, seed=2), device=DEV))
    X, A, Bm = sel.views()
    d = n + 1
    A_aug = torch.empty((B, N, d, d), dtype=torch.float64, device=DEV); Q_aug = torch.empty_like(A_aug)
    QT = torch.empty_like(A_aug); B_aug = torch.empty((B, N, d, m), dtype=torch.float64, device=DEV)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=DEV)  # noqa: E731
    xg_t, w_t, ur_t, Q_t = t(np.broadcast_to(xg, (B, n))), t(np.full(B, float(w))), t(u_ref), t(Q)
    Qf_t = t(O.as_terminal_weight(alpha, n))
    p_ = lambda a: C.c_void_p(a.data_ptr())  # noqa: E731
    lib = _cabi.require_device()
    _cabi.check(lib.hop_build_augmented_f64(B, N, n, m, p_(A), p_(Bm), None, p_(X), p_(sel.U), sel.ustride, p_(xg_t), p_(w_t), p_(ur_t),
                                            p_(Q_t), O.wrap_mask(wrap_idx), 1e-9, 1e-12, p_(A_aug), p_(B_aug), p_(Q_aug), None),
                "hop_build_augmented_f64")
    _cabi.check(lib.hop_build_terminal_f64(B, N, n, p_(X), p_(xg_t), p_(Qf_t), O.wrap_mask(wrap_idx), 1e-12, p_(QT), None),
                "hop_build_terminal_f64")
    torch.cuda.synchronize()
    z0 = np.zeros(d); z0[-1] = 1.0
    args = [A_aug, B_aug, Q_aug, t(O.chol_inv(0.5 * (R + R.T))), t(z0), QT]
    v, e, f = three(args, T_min, T_max, None, QUAD_TOL)
    re = _check_against_exact_and_fast(v, e, f)
    v2 = _np(api.propagator_all_Jt_aug_batched(*args, T_min, T_max, mode=api.MODE_VERIFIED, tie_tol=QUAD_TOL))
    for a, b in zip(v, v2):
        assert np.array_equal(a, b, equal_nan=True)
    print(f"\nquadrotor embedding x{B}: re-evaluated {int(re.sum())}, FAST T* != EXACT T* on {int((f[1] != e[1]).sum())}")


def test_determinism_and_empty_batch():
    args, w = s2_device(4096, 13, 4, 64, seed=1)
    a = _np(api.propagator_all_Jt_aug_batched(*args, 1, 64, w_explicit=w, mode=api.MODE_VERIFIED, tie_tol=1e-6))
    b = _np(api.propagator_all_Jt_aug_batched(*args, 1, 64, w_explicit=w, mode=api.MODE_VERIFIED, tie_tol=1e-6))
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert ((a[3] & RE) != 0).any()
    lib = _cabi.require_device()
    assert lib.hop_select_verified_f64(0, 8, 13, 4, 1, 8, None, None, None, None, 0, None, None, None, 1e-10, None, None, None,
                                       None, None) == 0
