"""Shared helpers for the test-suite (synthetic generators of SURVEY.md s.8d, tolerances)."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASE_NAMES = ["DoubleIntegrator", "Cartpole_SwingUp", "Quadrotor", "Segway_Balance"]


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def s2_instance(seed, d, m, N):
    """Synthetic HOP-LQR instance S2: draw order all A, all B, all Q, R, z0, w."""
    r = np.random.default_rng(seed)
    A = np.eye(d)[None] + 0.05 * r.standard_normal((N, d, d)) / np.sqrt(d)
    B = 0.05 * r.standard_normal((N, d, m))
    Q = np.stack([np.diag(r.uniform(0.5, 2.0, d)) for _ in range(N)])
    R = np.diag(r.uniform(0.05, 0.5, m))
    z0 = r.standard_normal(d)
    w = r.uniform(0.01, 0.1)
    QT = np.tile(50.0 * np.eye(d), (N, 1, 1))
    return A, B, Q, R, z0, w, QT


def s2_batch(seeds, d, m, N):
    inst = [s2_instance(s, d, m, N) for s in seeds]
    A = np.stack([i[0] for i in inst]); B = np.stack([i[1] for i in inst]); Q = np.stack([i[2] for i in inst])
    R = np.stack([i[3] for i in inst]); z0 = np.stack([i[4] for i in inst]); w = np.array([i[5] for i in inst])
    QT = np.stack([i[6] for i in inst])
    return A, B, Q, R, z0, w, QT


def s1_x0(B, seed=0):
    """S1 workload: quadrotor x0_b = x0 + sigma * xi_b (run_suite.py:72 sigma)."""
    x0 = np.zeros(12); x0[:3] = 2.0
    sigma = np.array([0.4, 0.4, 0.4] + [0.0] * 9)
    xi = np.random.default_rng(seed).standard_normal((B, 12))
    return x0[None] + sigma[None] * xi


# Per-case tolerance of the selection curve J(T) against the reference's own output.
# The reference curve is reproducible only to this level across BLAS builds (SURVEY.md s.9):
# (window rel tol, rel tol at T*, allowed |T - T_ref|)
J_TOL = {
    "DoubleIntegrator": (1e-5, 1e-7, 0),
    "Quadrotor": (1e-6, 5e-8, 0),           # reference vs fp80 truth at T*: 3.5e-10 (nominal) .. 4.8e-9 (converged)
    "Segway_Balance": (None, 1e-6, 0),      # uncontrolled diverging tail beyond T*: window is O(0.1) noise
    "Cartpole_SwingUp": (None, 1e-3, 1),    # argmin gap 1.3e-5 < reference noise 3e-5: T* ill-posed
}


def perstep_R(seed, B, N, m):
    """R_k [B, N, m, m] that differ per instance AND per step and are not diagonal: diag(U(0.05, 0.5)) + 0.01 11^T (SPD), so
    that a wrong step or instance offset of a per-step R^-1 changes the result."""
    r = np.random.default_rng(seed)
    return np.stack([[np.diag(r.uniform(0.05, 0.5, m)) + 0.01 * np.ones((m, m)) for _ in range(N)] for _ in range(B)])


def fused_batch(seed, B, n, m, N):
    """Synthetic inputs of the fused selection (augmented.py:10-87) at any (n, m): A [B,N,n,n], Bm [B,N,n,m], a_resid
    [B,N,n], X [B,N+1,n], one shared U [N,m], xg [B,n], w [B], u_ref [m], Q [n,n], R [m,m] (both SPD, not diagonal),
    alpha [n] (terminal weight diag(alpha)), wrap_idx = {0, n-1}.  State 0 sits a turn or more away from its goal on part of
    the horizon, so the angle wrap changes the errors."""
    r = np.random.default_rng(seed)
    A = np.eye(n)[None, None] + 0.05 * r.standard_normal((B, N, n, n)) / np.sqrt(n)
    Bm = 0.1 * r.standard_normal((B, N, n, m))
    a = 0.01 * r.standard_normal((B, N, n))
    X = 0.5 * r.standard_normal((B, N + 1, n))
    X[:, ::3, 0] += 2.0 * np.pi + 1.0
    U = 0.3 * r.standard_normal((N, m))
    xg = 0.2 * r.standard_normal((B, n))
    w = r.uniform(0.01, 0.1, B)
    u_ref = 0.1 * r.standard_normal(m)
    M = r.standard_normal((n, n))
    Q = np.diag(r.uniform(0.5, 2.0, n)) + 0.02 * (M @ M.T)
    R = np.diag(r.uniform(0.05, 0.5, m)) + 0.01 * np.ones((m, m))
    alpha = r.uniform(5.0, 50.0, n)
    return dict(A=A, Bm=Bm, a=a, X=X, U=U, xg=xg, w=w, u_ref=u_ref, Q=Q, R=R, alpha=alpha, wrap_idx=sorted({0, n - 1}))


def _oracle():
    import oracle                         # (imported late: the helpers above do not need the compiled oracle)
    return oracle


def perstep_problem(d, m, N, B, seed=0):
    """S2 blocks with a per-step R^-1 [B, N, m, m] = chol_inv(perstep_R)."""
    A, Bm, Q, _, z0, w, QT = s2_batch(range(seed, seed + B), d, m, N)
    Rinv = np.array([[_oracle().chol_inv(r) for r in inst] for inst in perstep_R(100 + seed, B, N, m)])
    return A, Bm, Q, Rinv, z0, w, QT


def reference_b(A, Bm, Q, Rinv, z0, QT, T_use, f80=False):
    """J(t) of the per-step problem through the UNMODIFIED single-R^-1 oracle: B'_k = B_k L_k, R^-1 = I."""
    m = Bm.shape[-1]
    Bp = Bm @ np.linalg.cholesky(Rinv)
    return np.stack([_oracle().propagator_all_Jt(A[b], Bp[b], Q[b], np.eye(m), z0[b], QT[b], T_use=T_use, f80=f80)
                     for b in range(A.shape[0])])


# (n, m) corners of the fused EXACT form (1 <= n <= 15, m <= n + 1)
FUSED_NM = [(1, 1), (1, 2), (3, 4), (5, 2), (7, 8), (10, 3), (15, 1), (15, 9), (15, 16)]


def fused_oracle(g, T_min, T_max):
    """The oracle's fused selection of every instance of a fused_batch: (J [B, T_max], T* [B])."""
    O = _oracle()
    out = [O.select_fused(g["A"][b], g["Bm"][b], g["X"][b], g["U"], g["xg"][b], g["u_ref"], g["Q"], g["R"], g["alpha"],
                          g["w"][b], T_min, T_max, g["wrap_idx"], a_resid=g["a"][b]) for b in range(g["A"].shape[0])]
    return np.stack([o[0] for o in out]), np.array([o[1] for o in out])
