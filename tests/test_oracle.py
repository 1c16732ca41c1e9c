"""Pins the CPU oracle (oracle/, plain-C restatement) against golden vectors recorded from the
real reference (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

import oracle as O
from _common import CASE_NAMES, J_TOL, golden, rel, s2_instance, s1_x0
from hop import cases


def _case(name):
    g = golden("case_" + name)
    tup = cases.make_case(name, N=int(g["N"]))
    return g, tup


def test_chol_inv_ladder_and_fallback_match_reference():
    u = golden("utils")
    seen = set()
    for A, X, kind in zip(u["mats"], u["invs"], u["kinds"]):
        d = int(str(kind).split(":")[1])
        Xo, info = O.chol_inv(A[:d, :d], return_info=True)
        seen.add(info)
        assert np.linalg.norm(Xo - X[:d, :d]) <= 1e-10 * np.linalg.norm(X[:d, :d]), kind
    assert 0 in seen and 8 in seen and any(0 < s < 8 for s in seen)  # first-try, ladder, LU fallback all hit


def test_chol_inv_rejects_nonfinite():
    with pytest.raises(FloatingPointError):
        O.chol_inv(np.array([[1.0, np.nan], [0.0, 1.0]]))


def test_chol_solve_and_wrap_match_reference():
    u = golden("utils")
    for A, B, X, (d, c) in zip(u["sA"], u["sB"], u["sX"], u["sdims"]):
        assert np.abs(O.chol_solve(A[:d, :d], B[:d, :c]) - X[:d, :c]).max() < 1e-12
    got = np.array([O.angle_normalize(a) for a in u["angles"]])
    assert np.array_equal(got, u["wrapped"])          # floored modulo, bit-exact
    assert O.angle_normalize(np.pi) == -np.pi and O.angle_normalize(-np.pi) == -np.pi


@pytest.mark.parametrize("name", CASE_NAMES)
def test_dynamics_match_reference(name):
    dy = golden("dynamics")
    g, tup = _case(name)
    F = tup[0]
    xs, us, fs = dy[name + "_x"], dy[name + "_u"], dy[name + "_f"]
    fo = np.stack([O.dynamics(F.hop_sys, F.hop_params, x, u) for x, u in zip(xs, us)])
    fh = np.stack([F(x, u) for x, u in zip(xs, us)])      # host twin shipped in hop/cases.py
    for f in (fo, fh):
        assert np.array_equal(np.isnan(f), np.isnan(fs))
        assert np.nanmax(np.abs(f - fs)) <= 4.5e-16 * max(1.0, np.nanmax(np.abs(fs)))


@pytest.mark.parametrize("name", CASE_NAMES)
def test_case_constants_match_reference(name):
    g, (F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, extra) = _case(name)
    for mine, ref in ((x0, "x0"), (xg, "xg"), (u_ref, "u_ref"), (Q, "Q"), (R, "R"), (np.asarray(alpha, float), "alpha")):
        assert np.array_equal(mine, g[ref])
    assert (w, N, T_min, T_max, F.dt) == (float(g["w"]), int(g["N"]), int(g["T_min"]), int(g["T_max"]), float(g["dt"]))
    assert list(wrap_idx) == list(g["wrap_idx"]) and extra is None


@pytest.mark.parametrize("name", CASE_NAMES)
def test_rollout_linearize_augment_match_reference(name):
    g, (F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _) = _case(name)
    s, p, U, X = F.hop_sys, F.hop_params, g["U"], g["X"]
    assert np.abs(O.rollout(s, p, x0, U) - X).max() <= 1e-13
    A, B = O.linearize(s, p, X, U, central=False)
    Ac, Bc = O.linearize(s, p, X, U, central=True)
    for mine, ref in ((A, "A_fwd"), (B, "B_fwd"), (Ac, "A_cen"), (Bc, "B_cen")):
        assert np.abs(mine - g[ref]).max() <= 1e-9 * max(1.0, np.abs(g[ref]).max())
    a = O.affine_residuals(s, p, X, U)
    assert np.abs(a - g["a_resid"]).max() <= 1e-13
    A_aug, B_aug, Q_aug, z0, R_inv = O.build_augmented(g["A_fwd"], g["B_fwd"], a, X, U, xg, u_ref, Q, R, w, wrap_idx)
    QT = O.build_terminal(X, xg, alpha, wrap_idx)
    ks = g["ks"]
    for mine, ref in ((A_aug[ks], "A_aug_ks"), (B_aug[ks], "B_aug_ks"), (Q_aug[ks], "Q_aug_ks"), (QT[ks], "QT_ks"),
                      (R_inv, "R_inv"), (z0, "z0")):
        assert np.abs(mine - g[ref]).max() <= 1e-12 * max(1.0, np.abs(g[ref]).max())
    assert abs(O.cost_timeopt_true(X, U, xg, u_ref, Q, R, alpha, w, int(g["T0"]), wrap_idx) - float(g["cost0"])) \
        <= 1e-12 * abs(float(g["cost0"]))


@pytest.mark.parametrize("name", CASE_NAMES)
def test_selection_curve_and_argmin_match_reference(name):
    g, (F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _) = _case(name)
    J, T = O.select_fused(g["A_fwd"], g["B_fwd"], g["X"], g["U"], xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx,
                          a_resid=g["a_resid"])
    Jr, Tr = g["J_curve0"], int(g["T0"])
    tol_win, tol_star, dT = J_TOL[name]
    assert abs(T - Tr) <= dT
    assert abs(J[Tr - 1] - Jr[Tr - 1]) <= tol_star * abs(Jr[Tr - 1])
    if tol_win is not None:
        assert rel(J[T_min - 1:T_max], Jr[T_min - 1:T_max]) <= tol_win
    # the fp80 evaluation of the same jittered algorithm agrees on T* wherever the problem is well posed
    J80, T80 = O.select_fused(g["A_fwd"], g["B_fwd"], g["X"], g["U"], xg, u_ref, Q, R, alpha, w, T_min, T_max,
                              wrap_idx, a_resid=g["a_resid"], f80=True)
    assert abs(T80 - Tr) <= dT


@pytest.mark.parametrize("name", CASE_NAMES)
def test_backward_and_linesearch_match_reference(name):
    g, (F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _) = _case(name)
    T0 = int(g["T0"])
    k, K, ok = O.backward_pass(g["A_fwd"], g["B_fwd"], g["X"], g["U"], xg, u_ref, Q, R, alpha, T0, 1e-3, wrap_idx)
    assert ok
    assert np.abs(k - g["k_list"]).max() <= 1e-10 * np.abs(g["k_list"]).max()
    assert np.abs(K - g["K_list"]).max() <= 1e-10 * np.abs(g["K_list"]).max()
    X1, U1, J1, acc = O.forward_linesearch(F.hop_sys, F.hop_params, g["X"], g["U"], xg, u_ref, Q, R, alpha, w, T0,
                                           g["k_list"], g["K_list"], wrap_idx)
    assert acc == bool(g["acc1"])
    assert abs(J1 - float(g["J1"])) <= 1e-12 * abs(float(g["J1"]))
    assert np.abs(U1 - g["U1"]).max() <= 1e-11 * max(1.0, np.abs(g["U1"]).max())
    assert np.abs(X1[:T0 + 1] - g["X1"][:T0 + 1]).max() <= 1e-10   # beyond T* the open-loop tail may be unstable
    Jbf = O.bruteforce_all_Jt(g["A_fwd"], g["B_fwd"], g["X"], g["U"], xg, u_ref, Q, R, alpha, w,
                              len(g["J_bruteforce48"]), 1e-6, wrap_idx)
    assert rel(Jbf, g["J_bruteforce48"]) <= 1e-10


@pytest.mark.parametrize("name", ["DoubleIntegrator", "Quadrotor", "Segway_Balance"])
def test_full_hop_ddp_solve_matches_reference(name):
    """solver.ilqr_timeopt_ourmethod with run_suite defaults: T_hist exact, J_hist to 1e-9."""
    g, (F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _) = _case(name)
    r = O.ilqr_timeopt_batch(F.hop_sys, F.hop_params, N, T_min, T_max, x0[None], g["U"], xg, u_ref, Q, R, alpha, w,
                             wrap_idx, max_iter=12, use_central_diff=False)
    assert r["status"][0] == 0
    nh = int(r["n_hist"][0])
    assert list(r["T_hist"][0, :nh]) == list(g["sol_T_hist"])
    assert rel(r["J_hist"][0, :nh], g["sol_J_hist"]) <= 1e-9
    assert int(r["T_star"][0]) == int(g["sol_T_star"])
    T = int(g["sol_T_star"])
    assert np.abs(r["U"][0, :T] - g["sol_U"][:T]).max() <= 1e-6 * max(1.0, np.abs(g["sol_U"]).max())
    assert np.abs(r["X"][0, :T + 1] - g["sol_X"][:T + 1]).max() <= 1e-6


def test_full_solve_cartpole_is_noise_limited():
    """Cartpole: the reference's own curve noise (3e-5 at T*) exceeds its argmin gap (1.3e-5), so the
    T_hist of an independent fp64 implementation may differ by one step per iteration (SURVEY.md s.9)."""
    g, (F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _) = _case("Cartpole_SwingUp")
    r = O.ilqr_timeopt_batch(F.hop_sys, F.hop_params, N, T_min, T_max, x0[None], g["U"], xg, u_ref, Q, R, alpha, w,
                             wrap_idx, max_iter=12, use_central_diff=False)
    nh = int(r["n_hist"][0])
    assert r["status"][0] == 0 and nh == len(g["sol_T_hist"])
    assert np.abs(r["T_hist"][0, :nh] - g["sol_T_hist"]).max() <= 1
    assert rel(r["J_hist"][0, :nh], g["sol_J_hist"]) <= 2e-2


def test_s2_synthetic_matches_reference_to_1e_12():
    g = golden("s2_synthetic")
    n = 0
    for key in g.files:
        if not key.startswith("J_"):
            continue
        d, m, N, s = (int(tok[1:]) for tok in key.split("_")[1:])
        A, B, Q, R, z0, w, QT = s2_instance(s, d, m, N)
        assert w == float(g["w_" + key[2:]])
        J = O.propagator_all_Jt(A, B, Q, O.chol_inv(R), z0, QT)
        assert rel(J, g[key]) <= 1e-12
        Jw = J + w * np.arange(1, N + 1)
        assert np.argmin(Jw) == np.argmin(g[key] + w * np.arange(1, N + 1))
        n += 1
    assert n == 12


def test_s1_quadrotor_batch_matches_reference():
    g = golden("s1_quadrotor_batch")
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = cases.make_case("Quadrotor", N=128)
    assert np.array_equal(s1_x0(16), g["x0"])
    U = np.tile(u_ref, (N, 1))
    J, T, st = O.select_from_x0_batch(F.hop_sys, F.hop_params, N, T_min, T_max, g["x0"], U, xg, u_ref, Q, R, alpha, w,
                                      wrap_idx, nthreads=4)
    assert not st.any() and np.array_equal(T, g["T"])
    assert rel(J[:, T_min - 1:], g["J"][:, T_min - 1:]) <= 1e-6


def test_argmin_window_first_minimum_and_nan():
    J = np.array([5.0, 3.0, 1.0, 1.0, 2.0])
    assert O.argmin_window(J, 1, 5) == 3 and O.argmin_window(J, 4, 5) == 4
    J[3] = np.nan
    assert O.argmin_window(J, 1, 5) == 4       # np.argmin: NaN wins


def test_oracle_reproduces_4096_reference_selections_of_the_headline_workload():
    """tests/golden/s1_quadrotor_ref4096.npz: the REAL reference on 4096 S1 instances (quadrotor N=128, the first 4096 of
    bench.py's rank-0 batch).  The oracle must select the same horizon on every one and reproduce J at T*-2..T*+2 to 1e-8
    (measured: 0 mismatches, 3.2e-9)."""
    from _common import s1_x0
    from hop import cases
    g = golden("s1_quadrotor_ref4096")
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = cases.make_case("Quadrotor", N=128)
    B = g["T"].shape[0]
    assert B == 4096
    J, T, st = O.select_from_x0_batch(F.hop_sys, F.hop_params, N, T_min, T_max, s1_x0(B, seed=int(g["seed"])),
                                      np.tile(u_ref, (N, 1)), xg, u_ref, Q, R, alpha, w, wrap_idx, nthreads=8)
    Tr = g["T"].astype(np.int64)
    assert not st.any() and np.array_equal(T, Tr)
    cols = Tr[:, None] + np.arange(-2, 3)[None, :]
    J5 = J[np.arange(B)[:, None], np.clip(cols, 1, T_max) - 1]
    assert np.nanmax(np.abs(J5 - g["J_pm2"]) / np.abs(g["J_pm2"])) <= 1e-8


def test_oracle_with_nonzero_affine_residuals_matches_the_reference():
    from hop import cases
    g = golden("resid_Quadrotor")
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = cases.make_case("Quadrotor", N=128)
    assert np.abs(g["a_resid"]).max() > 1e-4
    for b in range(g["X"].shape[0]):
        a = O.affine_residuals(F.hop_sys, F.hop_params, g["X"][b], g["U"][b])
        assert np.abs(a - g["a_resid"][b]).max() <= 1e-15
    J, T, st = O.select_fused_batch(g["A"], g["B"], g["X"], g["U"], xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx,
                                    a_resid=g["a_resid"], nthreads=4)
    assert not st.any() and np.array_equal(T, g["T"])
    assert rel(J[:, T_min - 1:70], g["J"][:, T_min - 1:70]) <= 2e-7        # (beyond T = 70 the tail is noise-dominated)
    assert rel(J[np.arange(4), T - 1], g["J"][np.arange(4), T - 1]) <= 5e-8
    J0, _, _ = O.select_fused_batch(g["A"], g["B"], g["X"], g["U"], xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx, nthreads=4)
    assert rel(J0[:, T_min - 1:70], g["J"][:, T_min - 1:70]) > 1e-5        # the residuals matter


@pytest.mark.parametrize("name", ["Segway_Balance", "Cartpole_SwingUp", "Quadrotor"])
def test_oracle_full_solves_match_the_reference_on_sampled_initial_states(name):
    """tests/golden/ddp_batch.npz: full HOP-DDP solves of the REAL reference (run_suite defaults) on sampled initial states --
    Segway 25 trials, Cartpole 48, Quadrotor (N = 128) 16 (configurations 2-4 at a size the reference finishes in minutes).
    An instance is well-posed when the oracle reproduces its own T_hist under six rounding-level perturbations
    (oracle/census.py); the reference (another BLAS, another summation order) is one more such perturbation.
    Segway / Quadrotor: T_hist identical to the reference on EVERY well-posed instance, J_hist <= 1e-9.  Cartpole (|E_k| ~ 5e8):
    the oracle's distance to the reference must not exceed its own worst self-flip rate (+ 3 instances), >= 85 % identical
    among the well-posed ones, J_hist <= 1e-6 where T_hist agrees (measured: 36/48 overall, 28/31, 2.3e-8)."""
    from oracle import census
    g = golden("ddp_batch")
    case = cases.make_case(name, N=128) if name == "Quadrotor" else cases.make_case(name)
    x0s = g[name + "_x0"]
    B = len(x0s)
    o, well, self_flip, _ = census.ddp_oracle_census(case, case[8], x0s, 12, nthreads=8)
    ref = {"n_hist": g[name + "_n_hist"], "T_hist": g[name + "_T_hist"]}
    same = np.array([census.same_history(o, ref, b) for b in range(B)])
    relJ = [rel(o["J_hist"][b, :o["n_hist"][b]], g[name + "_J_hist"][b, :o["n_hist"][b]]) for b in range(B) if same[b]]
    if name == "Cartpole_SwingUp":
        assert 1.0 - same.mean() <= max(self_flip.values()) + 3.0 / B + 0.1, (same.sum(), self_flip)
        assert (same & well).sum() >= 0.85 * well.sum()
        assert max(relJ) <= 1e-6
    else:
        assert well.sum() >= 0.8 * B
        assert (same & well).sum() == well.sum(), np.nonzero(well & ~same)[0]
        assert max(relJ) <= 1e-9
        assert (o["T_star"][well] == g[name + "_T_star"][well]).all()


@pytest.mark.parametrize("f80", [False, True])
def test_per_step_rinv_constant_over_k_is_bit_identical_to_one_rinv(f80):
    """R_inv [N, m, m] (a different R^-1 per step, horizon_selection.py:60-61) reloads R^-1 at every step; with the same R^-1
    at every step it must give the bits of the single-R^-1 path, in both precisions and through the batched entry."""
    from _common import s2_batch
    d, m, N, B = 5, 3, 12, 3
    A, Bm, Q, R, z0, w, QT = s2_batch(range(B), d, m, N)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    for b in range(B):
        J1 = O.propagator_all_Jt(A[b], Bm[b], Q[b], Rinv[b], z0[b], QT[b], f80=f80)
        Jk = O.propagator_all_Jt(A[b], Bm[b], Q[b], np.repeat(Rinv[b][None], N, 0), z0[b], QT[b], f80=f80)
        assert np.isfinite(J1).all() and np.array_equal(J1, Jk)
    if not f80:
        Jb, st = O.propagator_batch(A, Bm, Q, np.repeat(Rinv[:, None], N, 1), z0, QT, nthreads=2)
        Jo, sto = O.propagator_batch(A, Bm, Q, Rinv, z0, QT)
        assert not st.any() and not sto.any() and np.array_equal(Jb, Jo)
    with pytest.raises(ValueError):                       # a per-step R^-1 must cover every step
        O.propagator_all_Jt(A[0], Bm[0], Q[0], np.repeat(Rinv[0][None], N - 1, 0), z0[0], QT[0])


@pytest.mark.parametrize("m", [9, 16])
def test_select_fused_takes_control_dimensions_up_to_16(m):
    from _common import fused_batch
    n, N = 15, 6
    g = fused_batch(3, 2, n, m, N)
    for b in range(2):
        J, T = O.select_fused(g["A"][b], g["Bm"][b], g["X"][b], g["U"], g["xg"][b], g["u_ref"], g["Q"], g["R"], g["alpha"],
                              g["w"][b], 2, N - 1, g["wrap_idx"], a_resid=g["a"][b])
        assert np.isfinite(J).all() and 2 <= T <= N - 1 and T == np.argmin(J[1:N - 1]) + 2
    J, T, st = O.select_fused_batch(g["A"], g["Bm"], g["X"], g["U"], g["xg"], g["u_ref"], g["Q"], g["R"], g["alpha"], g["w"],
                                    2, N - 1, g["wrap_idx"], a_resid=g["a"])
    assert not st.any() and np.isfinite(J).all()


def test_select_fused_rejects_dimensions_beyond_its_arrays():
    """m > 16 or n > 15 is an argument error, not a write past the oracle's stack arrays."""
    from _common import fused_batch
    for n, m in ((15, 17), (16, 4)):
        g = fused_batch(4, 1, n, m, 4)
        with pytest.raises(RuntimeError, match="error code 4"):
            O.select_fused(g["A"][0], g["Bm"][0], g["X"][0], g["U"], g["xg"][0], g["u_ref"], g["Q"], g["R"], g["alpha"],
                           g["w"][0], 1, 4, g["wrap_idx"])
        with pytest.raises(RuntimeError, match="error code 4"):
            O.build_augmented(g["A"][0], g["Bm"][0], None, g["X"][0], g["U"], g["xg"][0], g["u_ref"], g["Q"], g["R"],
                              g["w"][0])
        with pytest.raises(RuntimeError, match="error code 4"):
            O.backward_pass(g["A"][0], g["Bm"][0], g["X"][0], g["U"], g["xg"][0], g["u_ref"], g["Q"], g["R"], g["alpha"], 3)
        assert np.isnan(O.cost_timeopt_true(g["X"][0], g["U"], g["xg"][0], g["u_ref"], g["Q"], g["R"], g["alpha"],
                                            g["w"][0], 3))
