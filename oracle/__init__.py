"""CPU ORACLE for the HOP horizon-selection hot path -- TEST INFRASTRUCTURE ONLY.

ctypes front-end to ``oracle/libhop_oracle.so`` (plain-C restatement of the reference numpy
algorithm; see hop_oracle.h).  Only ``tests/``, ``__graft_entry__.smoke()`` and bench.py's CPU
baseline / ``--impl reference`` legs may import this package.  The product
(``time-opt-ilqr_b200/``) never imports it and has no CPU fallback.

Parity pin: ``tests/golden/*.npz`` are generated from the real reference by
``tests/golden/make_golden.py``; ``tests/test_oracle.py`` checks this oracle against them.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhop_oracle.so")

HOP_OK, HOP_ERR_NONFINITE, HOP_ERR_LINALG, HOP_ERR_ALLOC, HOP_ERR_ARG = 0, 1, 2, 3, 4
SYS_IDS = {"DoubleIntegrator": 0, "Cartpole_SwingUp": 1, "Quadrotor": 2, "Quadrotor_Hover": 2, "Segway_Balance": 3}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_lp = C.POINTER(C.c_long)


class IlqrOpts(C.Structure):
    _fields_ = [("max_iter", C.c_int), ("lm_init", C.c_double), ("use_central_diff", C.c_int),
                ("use_f80_select", C.c_int)]


def build(force: bool = False) -> str:
    """Compile the oracle with gcc (recipe: oracle/Makefile)."""
    srcs = [os.path.join(_HERE, f) for f in ("hop_oracle.c", "hop_la.inc", "hop_oracle.h")]
    stale = force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if stale:
        subprocess.check_call(["make", "-C", _HERE, "-B", "libhop_oracle.so"], stdout=subprocess.DEVNULL)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = C.CDLL(_SO)
        _lib.hopo_angle_normalize.restype = C.c_double
        _lib.hopo_cost_timeopt_true.restype = C.c_double
        _lib.hopo_version.restype = C.c_char_p
    return _lib


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(_dp)


def _pi(a):
    return a.ctypes.data_as(_ip)


def wrap_mask(wrap_idx) -> int:
    mask = 0
    for i in (wrap_idx or []):
        mask |= 1 << int(i)
    return mask


def _raise(rc, what):
    if rc == HOP_OK:
        return
    if rc == HOP_ERR_NONFINITE:
        raise FloatingPointError(f"Non-finite values in {what}")
    if rc == HOP_ERR_LINALG:
        raise np.linalg.LinAlgError(f"{what} failed")
    raise RuntimeError(f"{what}: oracle error code {rc}")


# ----------------------------------------------------------------------------- utils.py
def as_terminal_weight(alpha, n):
    """utils.py:49-62."""
    A = np.asarray(alpha, dtype=float)
    if A.ndim == 0:
        return float(A) * np.eye(n)
    if A.ndim == 1:
        if A.shape[0] != n:
            raise ValueError("terminal weight vector has wrong shape")
        return np.diag(A)
    if A.ndim == 2:
        if A.shape != (n, n):
            raise ValueError("terminal weight matrix has wrong shape")
        return 0.5 * (A + A.T)
    raise ValueError("unsupported terminal weight ndim")


def chol_inv(A, jitter=1e-9, max_tries=8, return_info=False):
    A = _d(A)
    d = A.shape[0]
    X = np.empty((d, d))
    info = C.c_int(0)
    rc = lib().hopo_chol_inv(d, _p(A), _p(X), C.c_double(jitter), int(max_tries), C.byref(info))
    _raise(rc, "chol_inv(A)")
    return (X, info.value) if return_info else X


def chol_solve(A, B, jitter=1e-9, max_tries=8):
    A = _d(A)
    B0 = np.asarray(B, dtype=float)
    Bm = _d(B0.reshape(A.shape[0], -1))
    X = np.empty_like(Bm)
    rc = lib().hopo_chol_solve(A.shape[0], Bm.shape[1], _p(A), _p(Bm), _p(X), C.c_double(jitter), int(max_tries))
    _raise(rc, "chol_solve")
    return X.reshape(B0.shape)


def angle_normalize(a):
    return float(lib().hopo_angle_normalize(C.c_double(float(a))))


def wrap_error(e, wrap_idx=None):
    e = _d(e).copy()
    lib().hopo_wrap_error(e.size, _p(e), C.c_uint(wrap_mask(wrap_idx)))
    return e


# ----------------------------------------------------------------------------- systems.py
def sys_dims(sys):
    n, m = C.c_int(0), C.c_int(0)
    if lib().hopo_sys_dims(int(sys), C.byref(n), C.byref(m)):
        raise ValueError("unknown system id")
    return n.value, m.value


def dynamics(sys, p, x, u):
    n, _ = sys_dims(sys)
    p, x, u = _d(p), _d(x), _d(u).reshape(-1)
    xn = np.empty(n)
    lib().hopo_dynamics(int(sys), _p(p), _p(x), _p(u), _p(xn))
    return xn


# ----------------------------------------------------------------------------- solver.py
def rollout(sys, p, x0, U, max_state_norm=1e6):
    n, m = sys_dims(sys)
    p, x0, U = _d(p), _d(x0), _d(U).reshape(-1, m)
    N = U.shape[0]
    X = np.empty((N + 1, n))
    lib().hopo_rollout(int(sys), _p(p), N, _p(x0), _p(U), _p(X), C.c_double(max_state_norm))
    return X


def cost_timeopt_true(X, U, xg, u_ref, Q, R, alpha, w, T_star, wrap_idx=None):
    X, U = _d(X), _d(U)
    n, m = X.shape[1], U.shape[1]
    Qf = _d(as_terminal_weight(alpha, n))
    xg, u_ref, Q, R = _d(xg), _d(u_ref), _d(Q), _d(R)
    return float(lib().hopo_cost_timeopt_true(n, m, _p(X), _p(U), _p(xg), _p(u_ref), _p(Q), _p(R), _p(Qf),
                                              C.c_double(w), int(T_star), C.c_uint(wrap_mask(wrap_idx))))


def backward_pass(A, B, X, U, xg, u_ref, Q, R, alpha, T_star, lm_lambda=1e-3, wrap_idx=None):
    A, B, X, U = _d(A), _d(B), _d(X), _d(U)
    n, m = X.shape[1], U.shape[1]
    Qf = _d(as_terminal_weight(alpha, n))
    xg, u_ref, Q, R = _d(xg), _d(u_ref), _d(Q), _d(R)
    T = int(T_star)
    k = np.zeros((max(T, 1), m))
    K = np.zeros((max(T, 1), m, n))
    ok = C.c_int(0)
    rc = lib().hopo_backward_pass(n, m, _p(A), _p(B), _p(X), _p(U), _p(xg), _p(u_ref), _p(Q), _p(R), _p(Qf), T,
                                  C.c_double(lm_lambda), C.c_uint(wrap_mask(wrap_idx)), _p(k), _p(K), C.byref(ok))
    _raise(rc, "chol_solve")
    if not ok.value:
        return None, None, False
    return k[:T], K[:T], True


def forward_linesearch(sys, p, X, U, xg, u_ref, Q, R, alpha, w, T_star, k_list, K_list, wrap_idx=None):
    n, m = sys_dims(sys)
    X, U, p = _d(X), _d(U), _d(p)
    N = U.shape[0]
    Qf = _d(as_terminal_weight(alpha, n))
    xg, u_ref, Q, R = _d(xg), _d(u_ref), _d(Q), _d(R)
    kl = np.zeros((N, m)); Kl = np.zeros((N, m, n))
    kl[:int(T_star)] = np.asarray(k_list).reshape(-1, m)[:int(T_star)]
    Kl[:int(T_star)] = np.asarray(K_list).reshape(-1, m, n)[:int(T_star)]
    Xn, Un = np.empty_like(X), np.empty_like(U)
    J, acc = C.c_double(0), C.c_int(0)
    rc = lib().hopo_forward_linesearch(int(sys), _p(p), N, _p(X), _p(U), _p(xg), _p(u_ref), _p(Q), _p(R), _p(Qf),
                                       C.c_double(w), int(T_star), _p(kl), _p(Kl), C.c_uint(wrap_mask(wrap_idx)),
                                       _p(Xn), _p(Un), C.byref(J), C.byref(acc))
    _raise(rc, "forward_linesearch")
    return Xn, Un, J.value, bool(acc.value)


def bruteforce_all_Jt(A, B, X, U, xg, u_ref, Q, R, alpha, w, T_max, lm_lambda=1e-6, wrap_idx=None):
    A, B, X, U = _d(A), _d(B), _d(X), _d(U)
    n, m = X.shape[1], U.shape[1]
    Qf = _d(as_terminal_weight(alpha, n))
    xg, u_ref, Q, R = _d(xg), _d(u_ref), _d(Q), _d(R)
    J = np.zeros(int(T_max))
    rc = lib().hopo_bruteforce_all_Jt(n, m, _p(A), _p(B), _p(X), _p(U), _p(xg), _p(u_ref), _p(Q), _p(R), _p(Qf),
                                      C.c_double(w), int(T_max), C.c_double(lm_lambda),
                                      C.c_uint(wrap_mask(wrap_idx)), _p(J))
    _raise(rc, "chol_solve")
    return J


# ----------------------------------------------------------------------------- linearization.py
def linearize(sys, p, X, U, central=False, epsx=1e-5, epsu=1e-5, relx=1e-6, relu=1e-6):
    n, m = sys_dims(sys)
    p, X, U = _d(p), _d(X), _d(U).reshape(-1, m)
    N = U.shape[0]
    A = np.empty((N, n, n)); B = np.empty((N, n, m))
    lib().hopo_linearize(int(sys), _p(p), N, _p(X), _p(U), int(bool(central)), C.c_double(epsx), C.c_double(epsu),
                         C.c_double(relx), C.c_double(relu), _p(A), _p(B))
    return A, B


def affine_residuals(sys, p, X, U):
    n, m = sys_dims(sys)
    p, X, U = _d(p), _d(X), _d(U).reshape(-1, m)
    N = U.shape[0]
    a = np.empty((N, n))
    lib().hopo_affine_residuals(int(sys), _p(p), N, _p(X), _p(U), _p(a))
    return a


# ----------------------------------------------------------------------------- augmented.py
def build_augmented(A, B, a, X, U, xg, u_ref, Q, R, w, wrap_idx=None, q_reg=1e-9, rho_reg=1e-12):
    A, B, X, U = _d(A), _d(B), _d(X), _d(U)
    N, n, m = A.shape[0], X.shape[1], U.shape[1]
    d = n + 1
    xg, u_ref, Q, R = _d(xg), _d(u_ref), _d(Q), _d(R)
    a_arr = None if a is None else _d(np.asarray(a).reshape(N, n))
    A_aug = np.empty((N, d, d)); B_aug = np.empty((N, d, m)); Q_aug = np.empty((N, d, d)); R_inv = np.empty((m, m))
    rc = lib().hopo_build_augmented(n, m, N, _p(A), _p(B), None if a_arr is None else _p(a_arr), _p(X), _p(U),
                                    _p(xg), _p(u_ref), _p(Q), _p(R), C.c_double(w), C.c_uint(wrap_mask(wrap_idx)),
                                    C.c_double(q_reg), C.c_double(rho_reg), _p(A_aug), _p(B_aug), _p(Q_aug), _p(R_inv))
    _raise(rc, "chol_inv(A)")
    z0 = np.zeros(d); z0[-1] = 1.0
    return A_aug, B_aug, Q_aug, z0, R_inv


def build_terminal(X, xg, alpha, wrap_idx=None, rho_reg=1e-12):
    X = _d(X)
    n = X.shape[1]
    N = X.shape[0] - 1
    Qf = _d(as_terminal_weight(alpha, n))
    xg = _d(xg)
    QT = np.empty((N, n + 1, n + 1))
    rc = lib().hopo_build_terminal(n, N, _p(X), _p(xg), _p(Qf), C.c_uint(wrap_mask(wrap_idx)), C.c_double(rho_reg),
                                   _p(QT))
    _raise(rc, "build_terminal")
    return QT


# ----------------------------------------------------------------------------- horizon_selection.py
def _rinv_stride(R_inv, per_step_ndim, N, m):
    """0 for one R^-1 ([m,m] / [B,m,m]), m*m for one per step ([N,m,m] / [B,N,m,m]: chol_inv(R_list[k]))."""
    if R_inv.ndim == per_step_ndim:
        if R_inv.shape[-3] != N:
            raise ValueError(f"per-step R_inv has {R_inv.shape[-3]} steps, expected N = {N}")
        return m * m
    return 0


def propagator_all_Jt(A_aug, B_aug, Q_aug, R_inv, z0, QT, T_use=None, f80=False, jitter=1e-9, max_tries=8,
                      return_retries=False):
    """R_inv: [m,m] (the R_inv_cached argument) or [N,m,m] (chol_inv(R_list[k]) per step)."""
    A_aug, B_aug, Q_aug, QT = _d(A_aug), _d(B_aug), _d(Q_aug), _d(QT)
    R_inv, z0 = _d(R_inv), _d(z0)
    N, d = A_aug.shape[0], A_aug.shape[1]
    m = B_aug.shape[2]
    stride = _rinv_stride(R_inv, 3, N, m)
    T = N if T_use is None else int(T_use)
    J = np.zeros(max(T, 0))
    retries = (C.c_long * 5)()
    fn = lib().hopo_propagator_all_Jt_f80 if f80 else lib().hopo_propagator_all_Jt_f64
    rc = fn(T, d, m, _p(A_aug), _p(B_aug), _p(Q_aug), _p(R_inv), C.c_long(stride), _p(z0), _p(QT), _p(J),
            C.c_double(jitter), int(max_tries), retries)
    _raise(rc, "chol_inv(A)")
    return (J, list(retries)) if return_retries else J


def argmin_window(J, T_min, T_max):
    J = _d(J)
    return int(lib().hopo_argmin_window(_p(J), int(T_min), int(T_max)))


def propagator_batch(A_aug, B_aug, Q_aug, R_inv, z0, QT, T_use=None, nthreads=1):
    """R_inv: [m,m] (shared), [B,m,m] (one per instance) or [B,N,m,m] (one per instance and step)."""
    A_aug, B_aug, Q_aug, QT, z0 = _d(A_aug), _d(B_aug), _d(Q_aug), _d(QT), _d(z0)
    Bsz, N, d = A_aug.shape[0], A_aug.shape[1], A_aug.shape[2]
    m = B_aug.shape[3]
    R_inv = np.asarray(R_inv, dtype=float)
    R_inv = _d(np.broadcast_to(R_inv, (Bsz, m, m)) if R_inv.ndim == 2 else R_inv)
    stride = _rinv_stride(R_inv, 4, N, m)
    T = N if T_use is None else int(T_use)
    J = np.zeros((Bsz, T)); status = np.zeros(Bsz, dtype=np.int32)
    rc = lib().hopo_propagator_batch(int(nthreads), Bsz, N, T, d, m, _p(A_aug), _p(B_aug), _p(Q_aug), _p(R_inv),
                                     C.c_long(stride), _p(z0), _p(QT), _p(J), _pi(status))
    _raise(rc, "propagator_batch")
    return J, status


# ----------------------------------------------------------------------------- composed paths
def select_fused(A, B, X, U, xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx=None, a_resid=None, sys=-1, p=None,
                 f80=False):
    A, B, X, U = _d(A), _d(B), _d(X), _d(U)
    N, n, m = A.shape[0], X.shape[1], U.shape[1]
    Qf = _d(as_terminal_weight(alpha, n))
    xg, u_ref, Q, R = _d(xg), _d(u_ref), _d(Q), _d(R)
    pp = _d(p) if p is not None else np.zeros(1)
    a_arr = None if a_resid is None else _d(np.asarray(a_resid).reshape(N, n))
    J = np.zeros(int(T_max)); T = C.c_int(0)
    rc = lib().hopo_select_fused(int(sys), _p(pp), n, m, N, int(T_min), int(T_max), _p(A), _p(B),
                                 None if a_arr is None else _p(a_arr), _p(X), _p(U), _p(xg), _p(u_ref), _p(Q), _p(R),
                                 _p(Qf), C.c_double(w), C.c_uint(wrap_mask(wrap_idx)), int(bool(f80)), _p(J), C.byref(T))
    _raise(rc, "chol_inv(A)")
    return J, T.value


def select_fused_batch(A, B, X, U, xg, u_ref, Q, R, alpha, w, T_min, T_max, wrap_idx=None, a_resid=None, f80=False,
                       nthreads=1):
    """select_fused over a batch of GIVEN linearisations: A [B,N,n,n], B [B,N,n,m], X [B,N+1,n], U [B,N,m] or [N,m],
    xg [B,n] or [n], w [B] or scalar -> (J [B,T_max], T [B], status [B])."""
    A, B, X = _d(A), _d(B), _d(X)
    Bsz, N, n = A.shape[0], A.shape[1], A.shape[2]
    m = B.shape[3]
    U = _d(np.broadcast_to(np.asarray(U, dtype=float), (Bsz, N, m)))
    xg = _d(np.broadcast_to(np.asarray(xg, dtype=float), (Bsz, n)))
    w = _d(np.broadcast_to(np.asarray(w, dtype=float), (Bsz,)))
    Qf = _d(as_terminal_weight(alpha, n))
    u_ref, Q, R = _d(u_ref), _d(Q), _d(R)
    ar = None if a_resid is None else _d(np.asarray(a_resid).reshape(Bsz, N, n))
    J = np.zeros((Bsz, int(T_max))); T = np.zeros(Bsz, dtype=np.int32); status = np.zeros(Bsz, dtype=np.int32)
    rc = lib().hopo_select_fused_batch(int(nthreads), Bsz, n, m, N, int(T_min), int(T_max), _p(A), _p(B),
                                       None if ar is None else _p(ar), _p(X), _p(U), _p(xg), _p(u_ref), _p(Q), _p(R),
                                       _p(Qf), _p(w), C.c_uint(wrap_mask(wrap_idx)), int(bool(f80)), _p(J), _pi(T),
                                       _pi(status))
    _raise(rc, "select_fused_batch")
    return J, T, status


def select_from_x0_batch(sys, p, N, T_min, T_max, x0, U, xg, u_ref, Q, R, alpha, w, wrap_idx=None, central=False,
                         nthreads=1, f80=False):
    n, m = sys_dims(sys)
    x0 = _d(np.asarray(x0).reshape(-1, n))
    Bsz = x0.shape[0]
    xg = _d(np.broadcast_to(np.asarray(xg, dtype=float), (Bsz, n)))
    w = _d(np.broadcast_to(np.asarray(w, dtype=float), (Bsz,)))
    p, U, u_ref, Q, R = _d(p), _d(U).reshape(N, m), _d(u_ref), _d(Q), _d(R)
    Qf = _d(as_terminal_weight(alpha, n))
    J = np.zeros((Bsz, int(T_max))); T = np.zeros(Bsz, dtype=np.int32); status = np.zeros(Bsz, dtype=np.int32)
    rc = lib().hopo_select_from_x0_batch_ex(int(nthreads), Bsz, int(sys), _p(p), int(N), int(T_min), int(T_max), _p(x0),
                                            _p(U), _p(xg), _p(u_ref), _p(Q), _p(R), _p(Qf), _p(w),
                                            C.c_uint(wrap_mask(wrap_idx)), int(bool(central)), int(bool(f80)), _p(J),
                                            _pi(T), _pi(status))
    _raise(rc, "select_from_x0_batch")
    return J, T, status


def ilqr_timeopt_batch(sys, p, N, T_min, T_max, x0, U_init, xg, u_ref, Q, R, alpha, w, wrap_idx=None, max_iter=15,
                       lm_init=1e-3, use_central_diff=True, f80_select=False, nthreads=1):
    """solver.py:449-765 (method='propagator') over a batch of (x0, xg, w)."""
    n, m = sys_dims(sys)
    x0 = _d(np.asarray(x0).reshape(-1, n))
    Bsz = x0.shape[0]
    xg = _d(np.broadcast_to(np.asarray(xg, dtype=float), (Bsz, n)))
    w = _d(np.broadcast_to(np.asarray(w, dtype=float), (Bsz,)))
    p, U_init, u_ref, Q, R = _d(p), _d(U_init).reshape(N, m), _d(u_ref), _d(Q), _d(R)
    Qf = _d(as_terminal_weight(alpha, n))
    opts = IlqrOpts(int(max_iter), float(lm_init), int(bool(use_central_diff)), int(bool(f80_select)))
    cap = int(max_iter) + 1
    X = np.zeros((Bsz, N + 1, n)); U = np.zeros((Bsz, N, m))
    J_hist = np.full((Bsz, cap), np.nan); T_hist = np.zeros((Bsz, cap), dtype=np.int32)
    n_hist = np.zeros(Bsz, dtype=np.int32); J_curve = np.zeros((Bsz, int(T_max)))
    T_star = np.zeros(Bsz, dtype=np.int32); status = np.zeros(Bsz, dtype=np.int32)
    rc = lib().hopo_ilqr_timeopt_batch(int(nthreads), Bsz, int(sys), _p(p), int(N), int(T_min), int(T_max), _p(x0),
                                       _p(U_init), _p(xg), _p(u_ref), _p(Q), _p(R), _p(Qf), _p(w),
                                       C.c_uint(wrap_mask(wrap_idx)), C.byref(opts), _p(X), _p(U), _p(J_hist),
                                       _pi(T_hist), _pi(n_hist), _p(J_curve), _pi(T_star), _pi(status))
    _raise(rc, "ilqr_timeopt_batch")
    return dict(X=X, U=U, J_hist=J_hist, T_hist=T_hist, n_hist=n_hist, J_curve=J_curve, T_star=T_star, status=status)
