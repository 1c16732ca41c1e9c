"""GPU parity tests: the CUDA path (through the C-ABI) against the CPU oracle and the reference
goldens.  Tolerances: T* exact; J within 1e-9 relative on the well-conditioned synthetic family
(north star), and within the reference's own reproducibility on the augmented cases (J_TOL)."""
import numpy as np
import pytest
import torch

import oracle as O
from _common import CASE_NAMES, J_TOL, golden, rel, s1_x0, s2_batch
from hop import api, cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(a):
    return torch.as_tensor(np.ascontiguousarray(a), device=DEV)


@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_FAST])
@pytest.mark.parametrize("d,m,N,B", [(3, 1, 32, 9), (4, 2, 64, 33), (5, 1, 64, 7), (12, 4, 128, 5), (13, 4, 128, 6),
                                     (13, 4, 256, 3), (4, 2, 256, 2)])
def test_select_generic_matches_oracle_on_s2(d, m, N, B, mode):
    A, Bm, Q, R, z0, w, QT = s2_batch(range(B), d, m, N)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    sel = api.propagator_all_Jt_aug_batched(_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 1, N, w_explicit=_t(w), mode=mode)
    Jo, sto = O.propagator_batch(A, Bm, Q, Rinv, z0, QT, nthreads=4)
    J = sel.J.cpu().numpy()
    assert not sel.status.cpu().numpy().any() and not sto.any()
    if mode == api.MODE_EXACT:
        assert np.array_equal(J, Jo)                               # reference operation order: bit-identical to the oracle
    assert rel(J, Jo) <= 1e-9                                      # north-star tolerance
    tot = Jo + w[:, None] * np.arange(1, N + 1)
    assert np.array_equal(sel.T_star.cpu().numpy(), np.argmin(tot, axis=1) + 1)
    assert np.allclose(sel.J_star.cpu().numpy(), tot.min(axis=1), rtol=1e-9)


def test_select_generic_matches_reference_golden_s2():
    g = golden("s2_synthetic")
    from _common import s2_instance
    for key in g.files:
        if not key.startswith("J_"):
            continue
        d, m, N, s = (int(tok[1:]) for tok in key.split("_")[1:])
        A, Bm, Q, R, z0, w, QT = s2_instance(s, d, m, N)
        sel = api.propagator_all_Jt_aug_batched(_t(A[None]), _t(Bm[None]), _t(Q[None]), _t(O.chol_inv(R)), _t(z0),
                                                _t(QT[None]), 1, N)
        assert rel(sel.J.cpu().numpy()[0], g[key]) <= 1e-9


@pytest.mark.parametrize("name", CASE_NAMES)
@pytest.mark.parametrize("traj", ["nominal", "converged"])
@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_GJ, api.MODE_FAST])
def test_select_fused_matches_reference_golden(name, traj, mode):
    g = golden("case_" + name)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = cases.make_case(name, N=int(g["N"]))
    if traj == "nominal":
        X, U, A, Bm, Jr, Tr = g["X"], g["U"], g["A_fwd"], g["B_fwd"], g["J_curve0"], int(g["T0"])
    else:
        X, U = g["sol_X"], g["sol_U"]
        A, Bm = O.linearize(F.hop_sys, F.hop_params, X, U)
        Jr, Tr = g["conv_J_curve"], int(g["conv_T"])
    sel = api.select_fused_batched(_t(A[None]), _t(Bm[None]), _t(X[None]), _t(U[None]), xg, w, u_ref, Q, R, alpha,
                                   T_min, T_max, wrap_idx, mode=mode)
    J = sel.J.cpu().numpy()[0]
    tol_win, tol_star, dT = J_TOL[name]
    assert (int(sel.status[0]) & 0xFF) == 0
    if mode == api.MODE_EXACT:      # identical inputs => identical bits
        Jo, To = O.select_fused(A, Bm, X, U, xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx)
        assert np.array_equal(J, Jo) and int(sel.T_star[0]) == To
    assert abs(int(sel.T_star[0]) - Tr) <= dT
    assert abs(J[Tr - 1] - Jr[Tr - 1]) <= max(tol_star, 3e-5 if name == "Cartpole_SwingUp" else 0) * abs(Jr[Tr - 1])
    if tol_win is not None:
        assert rel(J[T_min - 1:T_max], Jr[T_min - 1:T_max]) <= tol_win


@pytest.mark.parametrize("d,m,N,T_max", [(12, 4, 128, 128), (13, 4, 128, 128), (13, 4, 64, 61), (13, 4, 16, 5)])
def test_scan_mode_matches_sequential_sweep_and_oracle(d, m, N, T_max):
    """HOP_MODE_SCAN: chunked parallel scan over the horizon (one CTA of 8 warps per problem).  Chunk 0 follows the sequential
    sweep (bit-identical to the sequential body: tests/test_emul_kernel.py; the default kernel here is the pipelined one, whose
    cost evaluation is an elimination instead of an inverse); later chunks differ by re-association only (well-conditioned
    S2: 1e-9, the north-star tolerance)."""
    A, Bm, Q, R, z0, w, QT = s2_batch(range(7), d, m, N)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    args = (_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 1, T_max)
    seq = api.propagator_all_Jt_aug_batched(*args, w_explicit=_t(w), mode=api.MODE_FAST)
    scan = api.propagator_all_Jt_aug_batched(*args, w_explicit=_t(w), mode=api.MODE_SCAN)
    Js, Jp = seq.J.cpu().numpy(), scan.J.cpu().numpy()
    Lc = -(-T_max // 8)
    assert not scan.status.cpu().numpy().any()
    assert rel(Jp[:, :Lc], Js[:, :Lc]) <= 1e-12
    assert rel(Jp, Js) <= 1e-9
    assert torch.equal(scan.T_star, seq.T_star)
    Jo, _ = O.propagator_batch(A, Bm, Q, Rinv, z0, QT, T_use=T_max)
    assert rel(Jp, Jo) <= 1e-9
    assert np.array_equal(scan.T_star.cpu().numpy(), np.argmin(Jo + w[:, None] * np.arange(1, T_max + 1), axis=1) + 1)


def test_scan_mode_is_refused_where_it_is_not_instantiated():
    from hop import _cabi
    A, Bm, Q, R, z0, w, QT = s2_batch(range(2), 4, 2, 8)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    with pytest.raises(_cabi.HopError):
        api.propagator_all_Jt_aug_batched(_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 1, 8, mode=api.MODE_SCAN)


@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_GJ])
def test_generic_and_fused_agree_bitwise_in_T_and_closely_in_J(mode):
    """The fused kernel builds the augmented blocks itself; feeding the oracle-built blocks to the
    generic kernel must give the same selection (EXACT: the same bits)."""
    g = golden("case_Quadrotor")
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = cases.make_case("Quadrotor", N=128)
    A_aug, B_aug, Q_aug, z0, R_inv = O.build_augmented(g["A_fwd"], g["B_fwd"], g["a_resid"], g["X"], g["U"], xg, u_ref, Q,
                                                       R, w, wrap_idx)
    QT = O.build_terminal(g["X"], xg, alpha, wrap_idx)
    s1 = api.propagator_all_Jt_aug_batched(_t(A_aug[None]), _t(B_aug[None]), _t(Q_aug[None]), _t(R_inv), _t(z0),
                                           _t(QT[None]), T_min, T_max, mode=mode)
    s2 = api.select_fused_batched(_t(g["A_fwd"][None]), _t(g["B_fwd"][None]), _t(g["X"][None]), _t(g["U"][None]), xg, w,
                                  u_ref, Q, R, alpha, T_min, T_max, wrap_idx, a_resid=_t(g["a_resid"][None]), mode=mode)
    assert int(s1.T_star[0]) == int(s2.T_star[0]) == int(g["T0"])
    if mode == api.MODE_EXACT:
        assert torch.equal(s1.J, s2.J)
    assert rel(s1.J.cpu().numpy()[0, T_min - 1:], s2.J.cpu().numpy()[0, T_min - 1:]) <= 1e-6


@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_FAST])
def test_ladder_fallback_and_nonfinite_status_on_gpu(mode):
    d, m, N = 4, 2, 8
    A, Bm, Q, R, z0, w, QT = s2_batch(range(11), d, m, N)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    Q[1, 3] = np.diag([1.0, 1.0, 1.0, -1e-4])
    QT[2, 5] = -np.eye(d)
    A[9, 2, 1, 1] = np.nan
    sel = api.propagator_all_Jt_aug_batched(_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 1, N, mode=mode)
    Jo, sto = O.propagator_batch(A, Bm, Q, Rinv, z0, QT)
    st = sel.status.cpu().numpy()
    assert st[0] == 0 and st[1] == 0x100 and st[2] == 0x300 and (st[9] & 0xFF) == 1 and sto[9] == 1
    ok = [i for i in range(11) if i != 9]
    assert rel(sel.J.cpu().numpy()[ok], Jo[ok]) <= 1e-9
    if mode == api.MODE_EXACT:      # the ladder and the LU fallback in the reference's operation order too
        assert np.array_equal(sel.J.cpu().numpy()[ok], Jo[ok])
    with pytest.raises(FloatingPointError):
        sel.raise_for_status()


@pytest.mark.parametrize("d,m,N,B", [(3, 1, 32, 70), (4, 2, 64, 97), (5, 1, 48, 33)])
def test_thread_per_problem_and_lane_group_kernels_agree_bit_for_bit(d, m, N, B):
    """hop_select_f64 routes large batches of small blocks (d <= 5) to the thread-per-problem kernel
    (hop_select_tpp_body.cuh); it performs the same IEEE operations per element as the lane-group kernel, so J, T*, J*
    and status are identical -- ragged last warp, T_min > 1, T_max < N, jitter ladder, LU fallback and a NaN included."""
    from hop import _cabi
    lib = _cabi.require_device()
    A, Bm, Q, R, z0, w, QT = s2_batch(range(B), d, m, N)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    Q[1, 3] = np.diag(np.r_[np.ones(d - 1), -1e-4])       # ladder
    QT[2, 5] = -np.eye(d)                                  # LU fallback
    A[B - 1, 7, 1, 1] = np.nan                             # FloatingPointError in the reference
    args = (_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 2, N - 1)
    out = {}
    old = lib.hop_test_set_tpp_min_batch(-2)
    try:
        for name, thr in (("lanes", 1 << 40), ("threads", 0)):
            lib.hop_test_set_tpp_min_batch(thr)
            sel = api.propagator_all_Jt_aug_batched(*args, w_explicit=_t(w), mode=api.MODE_FAST)
            out[name] = tuple(x.cpu().numpy() for x in (sel.J, sel.T_star, sel.J_star, sel.status))
    finally:
        lib.hop_test_set_tpp_min_batch(old)
    st = out["lanes"][3]
    assert st[1] == 0x100 and st[2] == 0x300 and (st[B - 1] & 0xFF) == 1 and st[0] == 0
    for a, b in zip(out["threads"], out["lanes"]):
        assert np.array_equal(a, b, equal_nan=True)
    ok = [i for i in range(B) if i != B - 1]
    Jo, _ = O.propagator_batch(A[ok], Bm[ok], Q[ok], Rinv[ok], z0[ok], QT[ok], T_use=N - 1)
    assert rel(out["threads"][0][ok], Jo) <= 1e-9


@pytest.mark.parametrize("name", CASE_NAMES)
def test_rollout_and_linearize_match_oracle(name):
    g = golden("case_" + name)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = cases.make_case(name, N=int(g["N"]))
    rng = np.random.default_rng(3)
    B = 5
    x0s = x0[None] + 0.05 * rng.standard_normal((B, x0.size))
    x0s[0] = x0
    U = g["U"]
    X = api.rollout_batched(F, _t(x0s), _t(U)).cpu().numpy()
    Xo = np.stack([O.rollout(F.hop_sys, F.hop_params, x, U) for x in x0s])
    assert np.abs(X - Xo).max() <= 1e-9 * max(1.0, np.abs(Xo).max())
    assert np.abs(X[0] - g["X"]).max() <= 1e-9 * max(1.0, np.abs(g["X"]).max())      # vs the reference itself
    for central, ka, kb in ((False, "A_fwd", "B_fwd"), (True, "A_cen", "B_cen")):
        A, Bm = api.linearize_batched(F, _t(Xo), _t(U), central=central)
        Ao, Bo = zip(*[O.linearize(F.hop_sys, F.hop_params, x, U, central=central) for x in Xo])
        # forward differences amplify a last-bit difference in sin/cos by 1/h = 1e5
        assert np.abs(A.cpu().numpy() - np.stack(Ao)).max() <= 2e-9 * max(1.0, np.abs(np.stack(Ao)).max())
        assert np.abs(Bm.cpu().numpy() - np.stack(Bo)).max() <= 2e-9 * max(1.0, np.abs(np.stack(Bo)).max())
        assert np.abs(A.cpu().numpy()[0] - g[ka]).max() <= 2e-9 * max(1.0, np.abs(g[ka]).max())
        assert np.abs(Bm.cpu().numpy()[0] - g[kb]).max() <= 2e-9 * max(1.0, np.abs(g[kb]).max())


def test_pipeline_linearisation_with_f0_from_rollout_is_bit_identical():
    """hop_select_from_x0 lets the quadrotor FD kernel read f0 = F(X_k, U_k) from X[k+1] (consistent rollout) and share
    the unperturbed sin/cos between its perturbed evaluations; the result must equal the stand-alone linearisation (which evaluates f0)
    bit for bit, NaN tails included (Euler-singularity instance: F returns NaN from step 1 on)."""
    case = cases.make_case("Quadrotor", N=128)
    F, u_ref, N = case[0], case[3], case[8]
    B = 48
    x0s = s1_x0(B)
    x0s[1, 7] = np.pi / 2
    x0s[2, 7] = 1.2                                         # large pitch: trajectory leaves the small-angle regime
    sel = api.HorizonSelector(case, B, mode=api.MODE_FAST)
    sel(_t(x0s))
    X, A, Bm = sel.views()
    A2, B2 = api.linearize_batched(F, X, _t(np.tile(u_ref, (N, 1))))
    assert np.isnan(X[1, 1:].cpu().numpy()).all() and np.isnan(A[1, 1:].cpu().numpy()).all()
    assert np.array_equal(A.cpu().numpy(), A2.cpu().numpy(), equal_nan=True)
    assert np.array_equal(Bm.cpu().numpy(), B2.cpu().numpy(), equal_nan=True)


def test_quadrotor_fd_kernels_agree_bit_for_bit():
    """The two implementations of linearize_forward_diff_traj and of linearize_central_diff_traj for the quadrotor
    (thread per step with compile-time sparsity, generic) must produce identical bits, on hover-like and on aggressive
    random states, guards included."""
    from hop import _cabi
    lib = _cabi.require_device()
    case = cases.make_case("Quadrotor", N=128)
    F, u_ref, N = case[0], case[3], case[8]
    rng = np.random.default_rng(11)
    B = 40
    x0s = s1_x0(B, seed=9)
    x0s[:, 3:] += rng.standard_normal((B, 9)) * np.array([1, 1, 1, .6, .6, 2.0, 3, 3, 3])   # velocities, large angles, rates
    x0s[3, 7] = np.pi / 2 - 1.0005e-3                    # |cos(pitch)| just above cos_pitch_min = 1e-3 (systems.py:166,187)
    x0s[4, 3:] = 0.0; x0s[4, 9] = 999.9995               # body rate just below omg_abs_max = 1e3: the perturbed point trips it
    x0s[5, 3:] = 0.0; x0s[5, :3] = [999999.4, 0.0, 0.0]  # norm just below state_norm_max = 1e6: h = 1 trips it for c = 0
    U = np.tile(u_ref, (N, 1))[None] + 0.5 * rng.standard_normal((B, N, 4))
    X = api.rollout_batched(F, _t(x0s), _t(U))
    out = {}
    try:
        for variant in (0, 2):
            lib.hop_test_set_linearize_variant(variant)
            A, Bm = api.linearize_batched(F, X, _t(U))
            Ac, Bc = api.linearize_batched(F, X, _t(U), central=True)
            out[variant] = (A.cpu().numpy(), Bm.cpu().numpy(), Ac.cpu().numpy(), Bc.cpu().numpy())
    finally:
        lib.hop_test_set_linearize_variant(0)
    assert np.isfinite(out[2][0]).mean() > 0.5 and np.isfinite(out[2][2]).mean() > 0.5
    for q in range(4):
        assert np.array_equal(out[0][q], out[2][q], equal_nan=True), q
    # a structurally independent entry is an exact zero, as in the reference ((F_i - F_i) / h)
    fin = np.isfinite(out[0][0][:, :, 0, 0])
    assert (out[0][0][:, :, 9, 0][fin] == 0.0).all()


def test_rollout_divergence_guard_nan_fills_like_the_reference():
    F = cases.make_case("Quadrotor", N=128)[0]
    x0 = np.zeros((2, 12)); x0[1, 7] = np.pi / 2          # Euler singularity -> F returns NaN (systems.py:179-181)
    U = np.tile(np.array([9.81, 0, 0, 0.0]), (16, 1))
    X = api.rollout_batched(F, _t(x0), _t(U)).cpu().numpy()
    assert np.isfinite(X[0]).all() and np.isfinite(X[1, 0]).all() and np.isnan(X[1, 1:]).all()


@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_GJ, api.MODE_FAST])
def test_s1_from_x0_device_and_host_paths_match_reference_and_oracle(mode):
    """Headline workload S1: quadrotor n=12, N=128, x0 ~ x0 + sigma xi, against (i) 4096 instances computed by the REAL
    reference (tests/golden/s1_quadrotor_ref4096.npz: T*, J at T* +- 2) and (ii) the oracle on every instance with the
    three-number census (oracle/census.py).  A T* mismatch is only accepted when the fp80 sweep shows the instance to be
    ill-posed (gap between the two candidates below 10 x the fp64 noise at those horizons); no count is waived."""
    from oracle import census
    g = golden("s1_quadrotor_ref4096")
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    B = int(g["T"].shape[0])
    x0s = s1_x0(B, seed=int(g["seed"]))
    sel = api.select_horizon_batched(case, _t(x0s), mode=mode)
    T = sel.T_star.cpu().numpy(); J = sel.J.cpu().numpy()
    assert not (sel.status.cpu().numpy() & 0xFF).any()
    # (i) the reference itself
    Tr, Jr5 = g["T"].astype(np.int64), g["J_pm2"]                      # J at T*-2 .. T*+2 (NaN outside [1, T_max])
    cols = Tr[:, None] + np.arange(-2, 3)[None, :]
    inside = (cols >= 1) & (cols <= T_max)
    Jg5 = np.where(inside, J[np.arange(B)[:, None], np.clip(cols, 1, T_max) - 1], np.nan)
    relr = np.abs(Jg5 - Jr5) / np.abs(Jr5)
    assert np.nanmax(relr) <= (2e-8 if mode == api.MODE_EXACT else 5e-8)        # at T* +- 2, vs the reference
    rep = census.census_from_x0(case, x0s, J, T, nthreads=8, fp80_stride=4)
    assert rep["T_star_mismatches_unexplained"] == 0, rep["mismatch_detail"]
    for b in np.nonzero(T != Tr)[0]:                                   # vs the reference: same rule, through the census list
        assert int(b) in rep["ill_posed"]["instances"] or any(int(b) == m["instance"] and m["ill_posed"] for m in rep["mismatch_detail"]) \
            or abs(Jr5[b, 2] - Jr5[b, 2 + int(T[b] - Tr[b])]) <= 1e-8 * abs(Jr5[b, 2]), (b, T[b], Tr[b])
    assert rep["rel_J_window"]["gpu_vs_oracle"]["max"] <= (2e-8 if mode == api.MODE_EXACT else 1e-6)
    # the checked implementation is as close to the fp80 truth as the fp64 oracle is (within 3 x)
    assert rep["rel_J_window"]["gpu_vs_fp80"]["p99"] <= 3.0 * rep["rel_J_window"]["oracle_vs_fp80"]["p99"]
    Jh, Th, Jsh, sth = api.select_horizon_host(case, x0s[:300], mode=mode)
    assert np.array_equal(Th, T[:300]) and np.array_equal(Jh, J[:300]) and np.array_equal(sth, sel.status.cpu().numpy()[:300])


def test_exact_mode_is_bit_identical_to_the_oracle_on_4096_device_linearisations():
    """HOP_MODE_EXACT issues the reference's operations one IEEE rounding at a time, so on IDENTICAL inputs its curve is the
    oracle's curve bit for bit.  Inputs: the rollout + forward-difference linearisation the DEVICE produced for 4096 S1
    instances (they differ from the host's only through CUDA's sin/cos/tan, <= 2 ulp), downloaded and fed to the oracle."""
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    B = 4096
    sel = api.HorizonSelector(case, B, device=DEV, mode=api.MODE_EXACT)
    r = sel(_t(s1_x0(B, seed=31)))
    X, A, Bm = (t.cpu().numpy() for t in sel.views())
    Jo, To, sto = O.select_fused_batch(A, Bm, X, np.tile(u_ref, (N, 1)), xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx,
                                       nthreads=8)
    assert not sto.any() and not (r.status.cpu().numpy() & 0xFF).any()
    assert np.array_equal(r.J.cpu().numpy(), Jo)
    assert np.array_equal(r.T_star.cpu().numpy(), To)


@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_GJ, api.MODE_FAST])
def test_nonzero_affine_residuals_in_every_selection_kernel(mode):
    """compute_affine_residuals (linearization.py:269-270) is exactly zero on a consistent rollout, so every other test feeds
    a_resid = 0.  Here X is perturbed AFTER the rollout (a_k = F(X_k, U_k) - X_{k+1} ~ 1e-3) and the residuals enter
    A_aug[:, n] = a_k - B_k du (augmented.py:50): fused kernels (TMA-staged a_k in the DMMA bodies) and the LQR-boundary
    kernels (through k_build_augmented) against the reference golden and the oracle."""
    g = golden("resid_Quadrotor")
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    X, U, A, Bm, ar = g["X"], g["U"], g["A"], g["B"], g["a_resid"]
    assert np.abs(ar).max() > 1e-4
    Bsz = X.shape[0]
    sel = api.select_fused_batched(_t(A), _t(Bm), _t(X), _t(U), xg, w, u_ref, Q, R, alpha, T_min, T_max, wrap_idx,
                                   a_resid=_t(ar), mode=mode)
    J = sel.J.cpu().numpy()
    Jo, To, sto = O.select_fused_batch(A, Bm, X, U, xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx, a_resid=ar, nthreads=4)
    assert not sto.any() and not (sel.status.cpu().numpy() & 0xFF).any()
    if mode == api.MODE_EXACT:
        assert np.array_equal(J, Jo)
    # compared on T in [T_min, 70]: beyond, the randomly perturbed controls make the tail of the curve noise-dominated (the
    # reference itself is 1e-4 away from the fp80 sweep there); on [40, 70] oracle and reference agree to 7e-8
    win = slice(T_min - 1, 70)
    assert rel(J[:, win], Jo[:, win]) <= 5e-7
    assert np.array_equal(sel.T_star.cpu().numpy(), To)
    assert np.array_equal(To, g["T"])                                          # the reference itself
    assert rel(J[:, win], g["J"][:, win]) <= 5e-7
    rows = np.arange(Bsz)
    assert rel(J[rows, g["T"] - 1], g["J"][rows, g["T"] - 1]) <= 5e-8
    # without the residuals the curve is a different one (2e-4 on instance 0): the input is live
    sel0 = api.select_fused_batched(_t(A), _t(Bm), _t(X), _t(U), xg, w, u_ref, Q, R, alpha, T_min, T_max, wrap_idx, mode=mode)
    assert rel(sel0.J.cpu().numpy()[:, win], Jo[:, win]) > 1e-5
    if mode != api.MODE_FAST:
        # LQR-boundary kernels on device-built blocks (hop_build_augmented_f64 carries a_k into A_aug)
        from hop import _cabi
        import ctypes as C
        lib = _cabi.require_device()
        d, m = 13, 4
        A_aug = torch.empty((Bsz, N, d, d), dtype=torch.float64, device=DEV); Q_aug = torch.empty_like(A_aug)
        QT = torch.empty_like(A_aug); B_aug = torch.empty((Bsz, N, d, m), dtype=torch.float64, device=DEV)
        xg_t = _t(np.broadcast_to(xg, (Bsz, 12)).copy()); w_t = _t(np.full(Bsz, float(w)))
        p_ = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        Xd, Ud, Ad, Bd, ard = _t(X), _t(U), _t(A), _t(Bm), _t(ar)
        ur_t, Q_t, Qf_t = _t(u_ref), _t(Q), _t(O.as_terminal_weight(alpha, 12))   # (kept alive: the launches are asynchronous)
        _cabi.check(lib.hop_build_augmented_f64(Bsz, N, 12, m, p_(Ad), p_(Bd), p_(ard), p_(Xd), p_(Ud), N * m, p_(xg_t), p_(w_t),
                                                p_(ur_t), p_(Q_t), O.wrap_mask(wrap_idx), 1e-9, 1e-12, p_(A_aug),
                                                p_(B_aug), p_(Q_aug), None), "hop_build_augmented_f64")
        _cabi.check(lib.hop_build_terminal_f64(Bsz, N, 12, p_(Xd), p_(xg_t), p_(Qf_t),
                                               O.wrap_mask(wrap_idx), 1e-12, p_(QT), None), "hop_build_terminal_f64")
        torch.cuda.synchronize()
        z0 = np.zeros(d); z0[-1] = 1.0
        s1 = api.propagator_all_Jt_aug_batched(A_aug, B_aug, Q_aug, _t(O.chol_inv(0.5 * (R + R.T))), _t(z0), QT, T_min, T_max,
                                               mode=mode)
        Ao, Bo, Qo, _, _ = O.build_augmented(A[0], Bm[0], ar[0], X[0], U[0], xg, u_ref, Q, R, w, wrap_idx)
        assert np.array_equal(A_aug[0].cpu().numpy(), Ao) and np.array_equal(B_aug[0].cpu().numpy(), Bo)
        assert np.array_equal(Q_aug[0].cpu().numpy(), Qo)
        assert np.array_equal(QT[0].cpu().numpy(), O.build_terminal(X[0], xg, alpha, wrap_idx))
        if mode == api.MODE_EXACT:
            assert np.array_equal(s1.J.cpu().numpy(), Jo)
        assert rel(s1.J.cpu().numpy()[:, win], Jo[:, win]) <= 5e-7
        assert np.array_equal(s1.T_star.cpu().numpy(), To)


def test_full_size_properties_without_oracle():
    """At a size the oracle would not finish quickly: size-independent properties.
    (1) determinism, (2) batch-permutation equivariance, (3) J(T) for T < T_min unaffected by window."""
    case = cases.make_case("Quadrotor", N=128)
    B = 4096
    x0s = s1_x0(B, seed=7)
    sel = api.HorizonSelector(case, B, device=DEV, mode=api.MODE_FAST)
    r1 = sel(_t(x0s)); T1 = r1.T_star.clone(); J1 = r1.J.clone()
    r2 = sel(_t(x0s))
    assert torch.equal(T1, r2.T_star) and torch.equal(J1, r2.J)
    perm = np.random.default_rng(0).permutation(B)
    r3 = sel(_t(x0s[perm]))
    assert torch.equal(r3.T_star.cpu(), T1.cpu()[perm]) and torch.equal(r3.J.cpu(), J1.cpu()[perm])
    assert int(T1.min()) >= 40 and int(T1.max()) <= 128 and torch.isfinite(J1).all()
    Jw = J1[:, 39:]
    assert torch.equal(Jw.argmin(dim=1).int() + 40, T1)


def test_chunked_host_path_equals_the_device_path_on_ragged_chunks():
    """hop_select_from_x0_host_f64 cuts large batches into chunks that alternate between two streams (uploads, kernels and
    the J(T) download of neighbouring chunks overlap).  Chunking must not change a bit: B = 40 003 gives three ragged
    chunks; per-instance xg / w and per-instance controls exercise every offset computation."""
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    B = 40003
    rng = np.random.default_rng(5)
    x0s = s1_x0(B, seed=3)
    xgs = xg[None] + 0.05 * rng.standard_normal((B, 12)) * np.r_[np.ones(3), np.zeros(9)]
    ws = w * (0.5 + rng.random(B))
    dev = api.select_horizon_batched(case, _t(x0s), xg=_t(xgs), w=_t(ws), mode=api.MODE_FAST)
    Jh, Th, Jsh, sth = api.select_horizon_host(case, x0s, xg=xgs, w=ws, mode=api.MODE_FAST)
    assert np.array_equal(Th, dev.T_star.cpu().numpy()) and np.array_equal(Jh, dev.J.cpu().numpy())
    assert np.array_equal(Jsh, dev.J_star.cpu().numpy()) and np.array_equal(sth, dev.status.cpu().numpy())
    assert len(np.unique(Th)) > 3


@pytest.mark.parametrize("mode", [api.MODE_FAST, api.MODE_GJ])
def test_fast_and_gj_modes_agree_with_exact_mode_on_4096_instances(mode):
    """FAST restructures the block inverses algebraically and GJ inverts by Gauss-Jordan with FMA: against HOP_MODE_EXACT on
    the same device inputs they must agree on J to the stated tolerance (include/hop_b200.h: 1e-6 on the window of the
    rank-deficient augmented problem, 5e-8 at T*) and select the same horizon except on near-ties: a T* mismatch is only
    accepted when the gap between the two candidates is below 10 x the distance between the two curves at those horizons."""
    case = cases.make_case("Quadrotor", N=128)
    x0s = _t(s1_x0(4096, seed=11))
    a = api.select_horizon_batched(case, x0s, mode=api.MODE_EXACT)
    Ta, Ja = a.T_star.cpu().numpy().astype(np.int64), a.J.cpu().numpy()
    b = api.select_horizon_batched(case, x0s, mode=mode)
    Tb, Jb = b.T_star.cpu().numpy().astype(np.int64), b.J.cpu().numpy()
    assert not (a.status.cpu().numpy() & 0xFF).any() and not (b.status.cpu().numpy() & 0xFF).any()
    assert rel(Jb[:, 39:], Ja[:, 39:]) <= 1e-6
    rows = np.arange(4096)
    assert rel(Jb[rows, Ta - 1], Ja[rows, Ta - 1]) <= 5e-8
    for i in np.nonzero(Ta != Tb)[0]:
        gap = abs(Ja[i, Ta[i] - 1] - Ja[i, Tb[i] - 1]) / abs(Ja[i, Ta[i] - 1])
        noise = max(abs(Jb[i, t - 1] - Ja[i, t - 1]) / abs(Ja[i, t - 1]) for t in (Ta[i], Tb[i]))
        assert gap < 10.0 * noise, (i, Ta[i], Tb[i], gap, noise)


def test_fp32_mode_reproduces_T_star_on_the_well_conditioned_family():
    """HOP_MODE_FP32 (hop_select_f64 only): the EXACT sweep in IEEE single precision.  Stated tolerance on S2 (include/hop_b200.h):
    J within 1e-4 relative, T* reproduced on >= 99 % of instances, every miss a gap below the fp32 noise."""
    for d, m, N in ((4, 2, 128), (12, 4, 64), (13, 4, 128)):
        B = 512
        A, Bm, Q, R, z0, w, QT = s2_batch(range(B), d, m, N)
        Rinv = np.stack([O.chol_inv(r) for r in R])
        args = (_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 1, N)
        ex = api.propagator_all_Jt_aug_batched(*args, w_explicit=_t(w), mode=api.MODE_EXACT)
        lo = api.propagator_all_Jt_aug_batched(*args, w_explicit=_t(w), mode=api.MODE_FP32)
        Je, Jl = ex.J.cpu().numpy(), lo.J.cpu().numpy()
        Te, Tl = ex.T_star.cpu().numpy().astype(np.int64), lo.T_star.cpu().numpy().astype(np.int64)
        assert not lo.status.cpu().numpy().any()
        assert rel(Jl, Je) <= 1e-4
        miss = np.nonzero(Te != Tl)[0]
        assert len(miss) <= B // 100, (d, N, len(miss))
        tot = Je + w[:, None] * np.arange(1, N + 1)
        for i in miss:
            assert abs(tot[i, Te[i] - 1] - tot[i, Tl[i] - 1]) <= 1e-4 * abs(tot[i, Te[i] - 1])


def test_fused_scan_mode_on_the_quadrotor_embedding():
    """HOP_MODE_SCAN through the fused entry point (blocks materialised by k_build_augmented / k_build_terminal, then the chunked
    parallel scan): same T* as the sequential sweep; chunk 0 of the curve within 1e-9, the rest within the re-association noise
    SURVEY.md s.9 measured on the quadrotor embedding (<= 1e-6 on the window)."""
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    B = 8
    sel = api.HorizonSelector(case, B, device=DEV, mode=api.MODE_EXACT)
    ex = sel(_t(s1_x0(B, seed=2)))
    X, A, Bm = sel.views()
    sc = api.select_fused_batched(A, Bm, X, _t(np.tile(u_ref, (N, 1))), xg, w, u_ref, Q, R, alpha, T_min, T_max, wrap_idx,
                                  mode=api.MODE_SCAN)
    assert not (sc.status.cpu().numpy() & 0xFF).any()
    Je, Js = ex.J.cpu().numpy(), sc.J.cpu().numpy()
    assert rel(Js[:, T_min - 1:], Je[:, T_min - 1:]) <= 1e-6
    Te, Ts = ex.T_star.cpu().numpy().astype(np.int64), sc.T_star.cpu().numpy().astype(np.int64)
    for i in np.nonzero(Te != Ts)[0]:
        assert abs(Je[i, Te[i] - 1] - Je[i, Ts[i] - 1]) <= 1e-7 * abs(Je[i, Te[i] - 1])


# ------------------------------------------------------------------ HOP-DDP iteration pieces + solver loop
@pytest.mark.parametrize("name", CASE_NAMES)
def test_backward_linesearch_and_cost_match_reference_golden(name):
    g = golden("case_" + name)
    case = cases.make_case(name, N=int(g["N"]))
    T0 = int(g["T0"])
    T = torch.tensor([T0, T0], dtype=torch.int32)
    A = _t(np.stack([g["A_fwd"]] * 2)); Bm = _t(np.stack([g["B_fwd"]] * 2))
    X = _t(np.stack([g["X"]] * 2)); U = _t(np.stack([g["U"]] * 2))
    J = api.cost_timeopt_true_batched(case, X, U, T).cpu().numpy()
    assert abs(J[0] - float(g["cost0"])) <= 1e-12 * abs(float(g["cost0"]))
    r = api.backward_linesearch_batched(case, A, Bm, X, U, T, 1e-3)
    assert r["ok"].cpu().numpy().all() and not r["err"].cpu().numpy().any()
    k = r["k"].cpu().numpy()[1, :T0]; K = r["K"].cpu().numpy()[1, :T0]
    assert np.abs(k - g["k_list"]).max() <= 1e-9 * np.abs(g["k_list"]).max()
    assert np.abs(K - g["K_list"]).max() <= 1e-9 * np.abs(g["K_list"]).max()
    assert bool(r["accepted"][0]) == bool(g["acc1"])
    assert abs(float(r["J_new"][0]) - float(g["J1"])) <= 1e-9 * abs(float(g["J1"]))
    assert np.abs(r["U_new"].cpu().numpy()[0] - g["U1"]).max() <= 1e-8 * max(1.0, np.abs(g["U1"]).max())
    assert np.abs(r["X_new"].cpu().numpy()[0, :T0 + 1] - g["X1"][:T0 + 1]).max() <= 1e-8


@pytest.mark.parametrize("name", ["DoubleIntegrator", "Quadrotor", "Segway_Balance"])
@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_FAST])
def test_batched_hop_ddp_solve_matches_reference_golden(name, mode):
    """solver.ilqr_timeopt_ourmethod with run_suite defaults (max_iter=12, forward differences): T_hist exact,
    J_hist to 1e-9 (north-star tolerance), final controls to 1e-6."""
    g = golden("case_" + name)
    case = cases.make_case(name, N=int(g["N"]))
    x0 = case[1]
    r = api.ilqr_timeopt_batched(case, _t(np.stack([x0, x0, x0])), max_iter=12, use_central_diff=False, mode=mode)
    nh = int(r["n_hist"][1])
    assert not (r["status"].cpu().numpy() & 0xFF).any()
    assert list(r["T_hist"].cpu().numpy()[1, :nh]) == list(g["sol_T_hist"])
    assert rel(r["J_hist"].cpu().numpy()[1, :nh], g["sol_J_hist"]) <= 1e-9
    assert int(r["T_star"][1]) == int(g["sol_T_star"])
    T = int(g["sol_T_star"])
    assert np.abs(r["U"].cpu().numpy()[1, :T] - g["sol_U"][:T]).max() <= 1e-6 * max(1.0, np.abs(g["sol_U"]).max())
    assert np.abs(r["X"].cpu().numpy()[1, :T + 1] - g["sol_X"][:T + 1]).max() <= 1e-6
    assert torch.equal(r["T_hist"][0], r["T_hist"][2]) and torch.equal(r["J_hist"][0, :nh], r["J_hist"][2, :nh])


@pytest.mark.parametrize("name", ["Segway_Balance", "Quadrotor"])
def test_one_pass_backward_gains_fall_back_to_the_reference_sequence(name):
    """The warp backward kernel forms the gains of a step in one pass (PD test and jittered factor in lockstep, all right-hand
    sides substituted together) and re-runs the reference sequence -- cholesky, chol_solve, chol_solve with their ladders and
    error codes -- whenever the straight-line path does not apply.  Instances: clean; an infinite entry in A_k (non-finite
    Qux: chol_solve's FloatingPointError); a negative regularisation (Quu_reg not PD: ok = False); an overflowing B_k.  The
    thread-per-problem kernel runs the reference sequence only: gains, flags and error codes must be identical."""
    from hop import _cabi
    lib = _cabi.require_device()
    g = golden("case_" + name)
    case = cases.make_case(name, N=int(g["N"]))
    Bsz = 4
    A = np.repeat(g["A_fwd"][None], Bsz, 0); Bm = np.repeat(g["B_fwd"][None], Bsz, 0)
    X = np.repeat(g["X"][None], Bsz, 0); U = np.repeat(g["U"][None], Bsz, 0)
    T = np.full(Bsz, min(40, int(g["N"])), np.int32)
    A[1, 17, 0, 1] = np.inf
    lm = np.array([1e-3, 1e-3, -1e9, 1e-3])
    Bm[3, 9] *= 1e200
    out = {}
    try:
        for variant in (2, 1):
            lib.hop_test_set_backward_variant(variant)
            r = api.backward_linesearch_batched(case, _t(A), _t(Bm), _t(X), _t(U), torch.as_tensor(T), lm)
            out[variant] = {k: v.cpu().numpy() for k, v in r.items()}
    finally:
        lib.hop_test_set_backward_variant(0)
    assert out[2]["ok"][0] == 1 and out[2]["ok"][2] == 0 and out[2]["ok"][1] == 0
    flat = lambda a: np.nan_to_num(a.astype(float), nan=-1.0, posinf=-2.0, neginf=-3.0)   # noqa: E731
    for key in ("ok", "err", "accepted"):
        assert np.array_equal(out[2][key], out[1][key]), key
    good = out[2]["ok"] == 1                         # the line search leaves X_new / U_new / J_new of a failed backward pass untouched
    assert np.array_equal(flat(out[2]["k"]), flat(out[1]["k"])) and np.array_equal(flat(out[2]["K"]), flat(out[1]["K"]))
    for key in ("X_new", "U_new", "J_new"):
        assert np.array_equal(flat(out[2][key][good]), flat(out[1][key][good])), key


@pytest.mark.parametrize("name", ["Quadrotor", "Segway_Balance", "DoubleIntegrator"])
def test_warp_and_thread_backward_kernels_agree_bit_for_bit(name):
    """backward_pass_truncated has two device mappings in the reference's summation order (one warp per problem, elements of
    every product spread over the lanes; one thread per problem).  Same operation order per element => identical gains, flags
    and solves."""
    from hop import _cabi
    lib = _cabi.require_device()
    case = cases.make_case(name, N=128) if name == "Quadrotor" else cases.make_case(name)
    n = case[1].size
    rng = np.random.default_rng(2)
    x0s = case[1][None] + 0.05 * rng.standard_normal((37, n))
    out = {}
    try:
        for variant in (2, 1):
            lib.hop_test_set_backward_variant(variant)
            out[variant] = api.ilqr_timeopt_batched(case, _t(x0s), max_iter=4, use_central_diff=False, mode=api.MODE_FAST)
    finally:
        lib.hop_test_set_backward_variant(0)
    for key in ("X", "U", "J_hist", "T_hist", "n_hist", "T_star", "status"):
        assert torch.equal(torch.nan_to_num(out[2][key].double(), nan=-1.0), torch.nan_to_num(out[1][key].double(), nan=-1.0)), key


def test_tensor_pipe_backward_kernel_against_the_ordered_kernel_and_the_reference():
    """The quadrotor backward pass of FAST / GJ solves runs its 12 x 12 products on the FP64 tensor pipe (hop_ddp_mma.cuh): FMA
    accumulation in k-blocks instead of the reference's unfused left-to-right sums.  Gains against the ordered kernel on the
    same inputs (<= 1e-12 relative) and against the reference golden (<= 1e-9); whole solves: same T_hist, J_hist <= 1e-9.
    HOP_MODE_EXACT solves and the stand-alone entry point keep the ordered kernel."""
    from hop import _cabi
    lib = _cabi.require_device()
    g = golden("case_Quadrotor")
    case = cases.make_case("Quadrotor", N=128)
    T0 = int(g["T0"])
    Bsz = 5
    A = _t(np.stack([g["A_fwd"]] * Bsz)); Bm = _t(np.stack([g["B_fwd"]] * Bsz))
    X = _t(np.stack([g["X"]] * Bsz)); U = _t(np.stack([g["U"]] * Bsz))
    T = torch.tensor([T0, T0 - 7, T0 + 9, 1, T0], dtype=torch.int32)
    res = {}
    try:
        for variant in (2, 3):
            lib.hop_test_set_backward_variant(variant)
            res[variant] = api.backward_linesearch_batched(case, A, Bm, X, U, T, 1e-3)
    finally:
        lib.hop_test_set_backward_variant(0)
    assert res[3]["ok"].cpu().numpy().all() and torch.equal(res[3]["ok"], res[2]["ok"]) and torch.equal(res[3]["accepted"], res[2]["accepted"])
    for key in ("k", "K"):
        a, b = res[3][key].cpu().numpy(), res[2][key].cpu().numpy()
        assert np.abs(a - b).max() <= 1e-12 * np.abs(b).max(), key
    K = res[3]["K"].cpu().numpy()[0, :T0]
    assert np.abs(K - g["K_list"]).max() <= 1e-9 * np.abs(g["K_list"]).max()                   # the reference itself
    assert abs(float(res[3]["J_new"][0]) - float(g["J1"])) <= 1e-9 * abs(float(g["J1"]))
    x0s = _t(s1_x0(48, seed=13))
    sol = {}
    try:
        for variant in (2, 3):
            lib.hop_test_set_backward_variant(variant)
            sol[variant] = api.ilqr_timeopt_batched(case, x0s, max_iter=8, use_central_diff=False, mode=api.MODE_FAST)
    finally:
        lib.hop_test_set_backward_variant(0)
    assert torch.equal(sol[3]["n_hist"], sol[2]["n_hist"]) and torch.equal(sol[3]["T_hist"], sol[2]["T_hist"])
    Ja, Jb = sol[3]["J_hist"].cpu().numpy(), sol[2]["J_hist"].cpu().numpy()
    m_ = np.isfinite(Jb)
    assert np.abs(Ja[m_] - Jb[m_]).max() <= 1e-9 * np.abs(Jb[m_]).max()
    assert not torch.equal(sol[3]["J_hist"], sol[2]["J_hist"])                              # (it IS a different kernel)


@pytest.mark.parametrize("d,m,N,T_max", [(12, 4, 48, 48), (13, 4, 64, 61), (13, 4, 8, 1)])
def test_pre_inverted_and_in_kernel_sweep_b_agree_bit_for_bit(d, m, N, T_max):
    """hop_select_f64, d in {12, 13}: the input-only inversions E_k = chol_inv(Q_k), X_t = chol_inv(QT_t) either run
    inside the sequential kernel (sweep B) or in a parallel pre-pass over every (problem, step) with the same interleaved
    sweep.  Same bits -- including instances that leave the pipelined path (ladder, LU fallback, NaN)."""
    from hop import _cabi
    lib = _cabi.require_device()
    B = 23
    A, Bm, Q, R, z0, w, QT = s2_batch(range(B), d, m, N)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    if T_max > 8:
        Q[1, 3] = np.diag(np.r_[np.ones(d - 1), -1e-4])       # ladder
        QT[2, 5] = -np.eye(d)                                  # LU fallback
        A[B - 1, 7, 1, 1] = np.nan
    args = (_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 1, T_max)
    out = {}
    try:
        for on in (0, 1):
            lib.hop_test_set_generic_pre(on)
            sel = api.propagator_all_Jt_aug_batched(*args, w_explicit=_t(w), mode=api.MODE_FAST)
            out[on] = tuple(x.cpu().numpy() for x in (sel.J, sel.T_star, sel.J_star, sel.status))
    finally:
        lib.hop_test_set_generic_pre(-1)
    for a, b in zip(out[1], out[0]):
        assert np.array_equal(a, b, equal_nan=True)
    if T_max > 8:
        st = out[1][3]
        assert st[1] == 0x300 or st[1] == 0x100
        assert st[2] == 0x300 and (st[B - 1] & 0xFF) == 1 and st[0] == 0


@pytest.mark.parametrize("d,m,N", [(12, 4, 40), (13, 4, 64)])
def test_diagonal_block_fast_path_and_sweep_agree_bit_for_bit(d, m, N):
    """hop_select_f64, d in {12, 13}: DIAGONAL input blocks Q_k / QT_t (the whole S2 family) are inverted element-wise instead
    of by two Gauss-Jordan sweeps; the sweep of a diagonal matrix computes exactly those reciprocals, so nothing may change by a
    bit -- with dense blocks mixed in (instance 1) and a non-PD diagonal block (instance 2: ladder, sequential cold path)."""
    from hop import _cabi
    lib = _cabi.require_device()
    B = 19
    A, Bm, Q, R, z0, w, QT = s2_batch(range(B), d, m, N)
    Rinv = np.stack([O.chol_inv(r) for r in R])
    rng = np.random.default_rng(8)
    Mx = rng.standard_normal((d, d)); Q[1, 3] = Mx @ Mx.T / d + np.eye(d)
    Mx = rng.standard_normal((d, d)); QT[1, 5] = Mx @ Mx.T + 50.0 * np.eye(d)
    Q[2, 4] = np.diag(np.r_[np.ones(d - 1), -1e-4])
    args = (_t(A), _t(Bm), _t(Q), _t(Rinv), _t(z0), _t(QT), 1, N)
    out = {}
    old = lib.hop_test_set_generic_diag(1)
    try:
        for on in (1, 0):
            lib.hop_test_set_generic_diag(on)
            sel = api.propagator_all_Jt_aug_batched(*args, w_explicit=_t(w), mode=api.MODE_FAST)
            out[on] = tuple(x.cpu().numpy() for x in (sel.J, sel.T_star, sel.J_star, sel.status))
    finally:
        lib.hop_test_set_generic_diag(old)
    for a, b in zip(out[1], out[0]):
        assert np.array_equal(a, b, equal_nan=True)
    Jo, sto = O.propagator_batch(A, Bm, Q, Rinv, z0, QT, nthreads=4)
    assert not sto.any() and out[1][3][0] == 0 and out[1][3][2] & 0x100
    assert rel(out[1][0], Jo) <= 1e-9


@pytest.mark.parametrize("name", ["DoubleIntegrator", "Segway_Balance", "Cartpole_SwingUp"])
def test_element_per_lane_and_lane_group_fused_kernels_agree_bit_for_bit(name):
    """The fused selection of the small systems has three device mappings: a lane group per problem (large batches), a warp
    per problem with one matrix element per lane, and -- for batches that leave the machine idle -- one problem per CTA as a
    warp-specialised pipeline (two stage warps, the prefix recursion on one warp, the queries J(t) on three, blocks handed
    over through shared-memory rings).  Same IEEE operations per element => the whole batched HOP-DDP solve (every selection
    of every iteration feeds the next one) is identical bit for bit, and so are T_max = 1, 2 and T_min = T_max."""
    from hop import _cabi
    lib = _cabi.require_device()
    case = cases.make_case(name)
    n = case[1].size
    rng = np.random.default_rng(6)
    x0s = case[1][None] + 0.2 * rng.standard_normal((41, n))
    out = {}
    try:
        for variant in (1, 2, 3):
            lib.hop_test_set_fused_small_variant(variant)
            out[variant] = api.ilqr_timeopt_batched(case, _t(x0s), max_iter=5, use_central_diff=False, mode=api.MODE_GJ)
    finally:
        lib.hop_test_set_fused_small_variant(0)
    for variant in (2, 3):
        for key in ("X", "U", "J_hist", "T_hist", "n_hist", "T_star", "J_curve", "status"):
            assert torch.equal(torch.nan_to_num(out[variant][key].double(), nan=-1.0),
                               torch.nan_to_num(out[1][key].double(), nan=-1.0)), (variant, key)
    assert torch.isfinite(out[1]["J_curve"]).any()
    # short sweeps: fewer steps than ring slots / query warps, a one-point window, a NaN in the inputs
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    g = golden("case_" + name)
    A = _t(np.repeat(g["A_fwd"][None], 3, 0)); Bm = _t(np.repeat(g["B_fwd"][None], 3, 0)); X = np.repeat(g["X"][None], 3, 0)
    X[2, 3, 0] = np.nan
    X = _t(X); U = _t(np.repeat(g["U"][None], 3, 0)); ar = _t(np.repeat(g["a_resid"][None], 3, 0))
    for (tmin, tmax) in ((1, 1), (1, 2), (2, 2), (3, 7), (int(T_min), min(int(T_max), int(g["N"])))):
        res = {}
        try:
            for variant in (1, 2, 3):
                lib.hop_test_set_fused_small_variant(variant)
                r = api.select_fused_batched(A, Bm, X, U, xg, w, u_ref, Q, R, alpha, tmin, tmax, wrap_idx=wrap_idx, a_resid=ar,
                                             mode=api.MODE_GJ)
                res[variant] = tuple(x.cpu().numpy() for x in (r.J, r.T_star, r.J_star, r.status))
        finally:
            lib.hop_test_set_fused_small_variant(0)
        for variant in (2, 3):
            for a, b in zip(res[variant], res[1]):
                assert np.array_equal(a, b, equal_nan=True), (variant, tmin, tmax)


@pytest.mark.parametrize("name", CASE_NAMES)
def test_parallel_and_serial_line_search_kernels_agree_bit_for_bit(name):
    """forward_linesearch_fixedT has two device mappings: the five step sizes side by side (six threads per problem, the
    cost evaluated while rolling) and one thread per problem trying them in turn.  Each candidate is the same
    instruction sequence, the first improving alpha wins in both => identical trajectories, histories and statuses.
    Perturbed initial states make iterations with alpha < 1 and fully rejected iterations both occur."""
    from hop import _cabi
    lib = _cabi.require_device()
    case = cases.make_case(name, N=128) if name == "Quadrotor" else cases.make_case(name)
    n = case[1].size
    rng = np.random.default_rng(4)
    x0s = case[1][None] + 0.3 * rng.standard_normal((45, n))
    out = {}
    try:
        for variant in (0, 1):
            lib.hop_test_set_linesearch_variant(variant)
            out[variant] = api.ilqr_timeopt_batched(case, _t(x0s), max_iter=6, use_central_diff=False, mode=api.MODE_FAST)
    finally:
        lib.hop_test_set_linesearch_variant(0)
    for key in ("X", "U", "J_hist", "T_hist", "n_hist", "T_star", "status"):
        assert torch.equal(torch.nan_to_num(out[0][key].double(), nan=-1.0), torch.nan_to_num(out[1][key].double(), nan=-1.0)), key
    assert int(out[0]["n_hist"].max()) >= 3


@pytest.mark.parametrize("name", CASE_NAMES)
def test_bruteforce_curve_matches_reference_golden_and_oracle(name):
    """solver.py:293-358 on the device (one warp per horizon) against the reference's own output (first 48 horizons in
    the goldens) and against the oracle over the whole window -- on the nominal trajectory (du = 0) and on the converged
    one, where du != 0 exercises the lu = R du terms (a shared-memory aliasing bug in exactly those terms for m = 1 went
    unnoticed while only the nominal trajectory was tested)."""
    g = golden("case_" + name)
    case = cases.make_case(name, N=int(g["N"]))
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    A, Bm, X, U = g["A_fwd"], g["B_fwd"], g["X"], g["U"]
    J, st = api.bruteforce_all_Jt_batched(case, _t(A[None]), _t(Bm[None]), _t(X[None]), _t(U[None]), T_max=T_max)
    J = J.cpu().numpy()[0]
    assert int(st[0]) == 0
    nb = len(g["J_bruteforce48"])
    assert rel(J[:nb], g["J_bruteforce48"]) <= 1e-10
    Jo = O.bruteforce_all_Jt(A, Bm, X, U, xg, u_ref, Q, R, alpha, w, T_max, 1e-6, wrap_idx)
    assert rel(J, Jo) <= 1e-10
    Xc, Uc = g["sol_X"], g["sol_U"]
    assert np.abs(Uc - u_ref[None]).max() > 1e-3
    Ac, Bc = O.linearize(F.hop_sys, F.hop_params, Xc, Uc)
    Jc, st = api.bruteforce_all_Jt_batched(case, _t(Ac[None]), _t(Bc[None]), _t(Xc[None]), _t(Uc[None]), T_max=T_max)
    assert int(st[0]) == 0
    Joc = O.bruteforce_all_Jt(Ac, Bc, Xc, Uc, xg, u_ref, Q, R, alpha, w, T_max, 1e-6, wrap_idx)
    assert rel(Jc.cpu().numpy()[0], Joc) <= 1e-9


def test_propagator_curve_agrees_with_the_bruteforce_curve_on_device():
    """Independent cross-check at scale, entirely on the device: the propagator's J(T) (O(T n^3)) against T separate Riccati
    sweeps (O(T^2 n^3)) for 256 sampled quadrotor instances.  The two formulations regularise differently (1e-9 jitter and
    q_reg in the propagator, lm_lambda = 1e-6 in the sweep): on the reference itself the curves differ by a smooth 1.3e-5
    relative offset that varies by < 1e-6 over the window, so the argmin must coincide except on near-ties."""
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    B = 256
    sel = api.HorizonSelector(case, B, mode=api.MODE_FAST)
    s = sel(_t(s1_x0(B, seed=21)))
    X, A, Bm = sel.views()
    Jb, st = api.bruteforce_all_Jt_batched(case, A, Bm, X, _t(np.tile(u_ref, (N, 1))), T_max=T_max)
    assert not st.cpu().numpy().any()
    Jp, Jb = s.J.cpu().numpy(), Jb.cpu().numpy()
    r = (Jp[:, T_min - 1:] - Jb[:, T_min - 1:]) / Jb[:, T_min - 1:]
    assert np.abs(r).max() <= 1e-4
    assert (r.max(axis=1) - r.min(axis=1)).max() <= 5e-6       # same SHAPE: the offset is almost constant in T
    Tb = np.argmin(Jb[:, T_min - 1:], axis=1) + T_min
    Tp = s.T_star.cpu().numpy()
    diff = np.nonzero(Tb != Tp)[0]
    for b in diff:                                       # only near-ties may differ
        assert abs(Jb[b, Tb[b] - 1] - Jb[b, Tp[b] - 1]) <= 5e-6 * abs(Jb[b, Tb[b] - 1])
    assert len(diff) <= B // 10


@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_FAST])
def test_batched_hop_ddp_matches_oracle_on_sampled_quadrotor_instances(mode):
    """Config 4 (scaled down): quadrotor N=128, sampled x0; every instance runs its own state machine.  T_hist must be the
    oracle's on every instance, with one documented exception: a near-tie in ONE selection may move that entry to the
    ADJACENT horizon (SURVEY.md s.9); such an instance must still converge to the same cost (1e-6)."""
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    Bsz = 24
    x0s = s1_x0(Bsz, seed=5)
    r = api.ilqr_timeopt_batched(case, _t(x0s), max_iter=12, use_central_diff=False, mode=mode)
    o = O.ilqr_timeopt_batch(F.hop_sys, F.hop_params, N, T_min, T_max, x0s, np.tile(u_ref, (N, 1)), xg, u_ref, Q, R, alpha, w,
                             wrap_idx, max_iter=12, use_central_diff=False, nthreads=8)
    nh = r["n_hist"].cpu().numpy()
    Th = r["T_hist"].cpu().numpy(); Jh = r["J_hist"].cpu().numpy()
    differing = []
    for b in range(Bsz):
        if nh[b] == o["n_hist"][b] and np.array_equal(Th[b, :nh[b]], o["T_hist"][b, :nh[b]]):
            assert rel(Jh[b, :nh[b]], o["J_hist"][b, :nh[b]]) <= 1e-8
            assert int(r["T_star"][b]) == int(o["T_star"][b])
            continue
        differing.append(b)
        k = min(nh[b], o["n_hist"][b])
        first = int(np.nonzero(Th[b, :k] != o["T_hist"][b, :k])[0][0]) if (Th[b, :k] != o["T_hist"][b, :k]).any() else k - 1
        assert abs(int(Th[b, first]) - int(o["T_hist"][b, first])) <= 1, (b, Th[b, :nh[b]], o["T_hist"][b, :o["n_hist"][b]])
        assert abs(Jh[b, nh[b] - 1] - o["J_hist"][b, o["n_hist"][b] - 1]) <= 1e-6 * abs(o["J_hist"][b, o["n_hist"][b] - 1])
    assert len(differing) <= (0 if mode == api.MODE_EXACT else 1), differing


def test_cartpole_batched_solve_against_the_oracle_on_identical_initial_states():
    """Config 3 flavour: cartpole from perturbed initial states (the reference's own sigma is zero), HOP_MODE_EXACT and
    HOP_MODE_FAST against the oracle on the SAME x0.  The cartpole embedding amplifies rounding (Q has a zero weight:
    |E_k| ~ 5e8): the reference computation itself flips T_hist on 12-19 % of the instances under ONE rounding-level
    perturbation (fp80 selection sweep, x0 +- 1e-15, ...; measured by tests/run_configs.py: ddp_census).  A device run is one
    more such perturbation (CUDA's sin/cos: <= 2 ulp from glibc's), so the bar is:
      (1) its T_hist mismatch rate against the oracle is not above the oracle's own worst single-perturbation flip rate
          (+ 3 instances of sampling slack);
      (2) on the instances that are stable under all six oracle perturbations it reproduces the oracle's T_hist on >= 95 %
          (a seventh perturbation still flips a few instances that six did not: the same holds between the oracle runs)
          with J_hist within 1e-6."""
    from run_configs import ddp_census
    g = golden("case_Cartpole_SwingUp")
    case = cases.make_case("Cartpole_SwingUp")
    rng = np.random.default_rng(0)
    Bsz = 256
    x0s = np.array([rng.normal(0, .1, Bsz), rng.normal(0, .1, Bsz), rng.normal(0, .2, Bsz), rng.normal(0, .2, Bsz)]).T
    x0s[0] = case[1]
    r = api.ilqr_timeopt_batched(case, _t(x0s), max_iter=12, use_central_diff=False, mode=api.MODE_FAST)
    assert torch.isfinite(r["J_hist"][:, 0]).all()
    rep = ddp_census(case, case[8], x0s, 12, {"fast": (r["n_hist"].cpu().numpy(), r["T_hist"].cpu().numpy(),
                                                         r["J_hist"].cpu().numpy(), r["T_star"].cpu().numpy())}, DEV)
    assert rep["well_posed"] >= Bsz // 2, rep
    worst_self = max(rep["oracle_self_flip_rate"].values())
    for label in ("exact", "fast"):
        assert rep[label]["mismatch_rate"] <= worst_self + 3.0 / Bsz, (label, rep)
        assert rep[label]["T_hist_identical_among_well_posed"] >= 0.95 * rep["well_posed"], (label, rep)
        assert rep[label]["max_rel_J_hist_where_T_identical"] <= 1e-6, (label, rep)
    # the reference's own run of the nominal instance (golden); the oracle itself is within |dT| <= 1 of it (tests/test_oracle.py)
    n0 = len(g["sol_T_hist"])
    assert int(r["n_hist"][0]) == n0 and np.abs(r["T_hist"].cpu().numpy()[0, :n0] - g["sol_T_hist"]).max() <= 1


@pytest.mark.parametrize("name", ["Segway_Balance", "Cartpole_SwingUp", "Quadrotor"])
@pytest.mark.parametrize("mode", [api.MODE_EXACT, api.MODE_FAST])
def test_batched_hop_ddp_against_reference_solves_on_sampled_initial_states(name, mode):
    """tests/golden/ddp_batch.npz (full solves of the REAL reference: Segway 25 trials, Cartpole 48, Quadrotor 16 instances) on
    the device.  Same bar as tests/test_oracle.py applies to the oracle: on every instance that is well-posed by the oracle's
    perturbation census T_hist is the reference's (Segway, Quadrotor; J_hist <= 1e-9); on the cartpole embedding the device's
    distance to the reference stays within the oracle's own self-flip band and >= 75 % of the well-posed instances agree."""
    from oracle import census
    g = golden("ddp_batch")
    case = cases.make_case(name, N=128) if name == "Quadrotor" else cases.make_case(name)
    x0s = g[name + "_x0"]
    B = len(x0s)
    r = api.ilqr_timeopt_batched(case, _t(x0s), max_iter=12, use_central_diff=False, mode=mode)
    dev = {"n_hist": r["n_hist"].cpu().numpy(), "T_hist": r["T_hist"].cpu().numpy()}
    Jh = r["J_hist"].cpu().numpy()
    ref = {"n_hist": g[name + "_n_hist"], "T_hist": g[name + "_T_hist"]}
    o, well, self_flip, _ = census.ddp_oracle_census(case, case[8], x0s, 12, nthreads=8)
    same = np.array([census.same_history(dev, ref, b) for b in range(B)])
    relJ = [rel(Jh[b, :dev["n_hist"][b]], g[name + "_J_hist"][b, :dev["n_hist"][b]]) for b in range(B) if same[b]]
    assert not (r["status"].cpu().numpy() & 0xFF).any()
    if name == "Cartpole_SwingUp":
        # (the device is TWO rounding-level perturbations away from the reference -- CUDA's sin/cos against glibc's, and the
        #  oracle's plain loops against OpenBLAS -- so the bar is a little below the oracle's own 28 of 31)
        assert 1.0 - same.mean() <= max(self_flip.values()) + 3.0 / B + 0.1, (same.sum(), self_flip)
        assert (same & well).sum() >= 0.75 * well.sum(), ((same & well).sum(), well.sum())
        assert max(relJ) <= 1e-6
    else:
        assert (same & well).sum() == well.sum(), (np.nonzero(well & ~same)[0], self_flip)
        assert max(relJ) <= 1e-9
