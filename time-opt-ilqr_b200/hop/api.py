"""Batched entry points of the B200 HOP path (additive to the reference's single-instance API).

All tensors are fp64 CUDA tensors owned by the caller (PyTorch is only the allocator / stream
provider); the work is done by libhop_b200.so through the C ABI in include/hop_b200.h.

    propagator_all_Jt_aug_batched   horizon_selection.py:36-86 (+ solver.py:522 argmin) over a batch
    select_fused_batched            augmented.py:10-87 + the above, fused (no (n+1)^2 blocks in HBM)
    rollout_batched                 solver.py:42-62
    linearize_batched               linearization.py:177-262
    select_horizon_batched          x0 -> rollout -> linearise -> fused selection (device tensors)
    select_horizon_host             same through HOST buffers (numpy in / numpy out)
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _cabi
from .cases import NPARAMS, SYS_DIMS

# include/hop_b200.h HOP_MODE_*
MODE_EXACT = 0   # PARITY mode: the reference's operation order with individually rounded IEEE operations (Cholesky route,
                 # no FMA); J(T) bit-identical to the plain-C oracle on identical inputs; any d, m <= 16
MODE_FAST = 1    # throughput mode: closed-form block inverses + pivot-only J(t), pipelined Gauss-Jordan sweeps (same function)
MODE_SCAN = 2    # d in {12, 13}: chunked parallel scan over the horizon (small batches; re-association changes the rounding)
MODE_GJ = 3      # materialised blocks + in-place Gauss-Jordan inverse with FMA (the cold path of FAST; instantiated dims only)
MODE_FP32 = 4    # propagator_all_Jt_aug_batched only: the EXACT sweep in single precision (well-conditioned problems only)
MODE_VERIFIED = 5  # fused forms and the solver, quadrotor and DI: FAST, then instances whose two best horizons are within the
                   # measured tie tolerance (or with a non-finite window / non-zero status) recomputed in EXACT: T* and status low
                   # byte equal EXACT's (include/hop_b200.h); propagator_all_Jt_aug_batched with the caller's tie_tol
ST_FLAG_REEVALUATED = 0x400   # include/hop_b200.h status bit 10: MODE_VERIFIED recomputed this instance in EXACT


@dataclass
class Selection:
    """Result of a batched horizon selection."""
    J: Optional[torch.Tensor]     # [B, T_max] fp64, J[:, t-1] = optimal LQR cost-to-go with horizon t (incl. w t when implicit)
    T_star: torch.Tensor          # [B] int32
    J_star: torch.Tensor          # [B] fp64 (value of the minimised curve at T*)
    status: torch.Tensor          # [B] int32, see include/hop_b200.h

    def raise_for_status(self):
        """Mirror the reference's exceptions for the first failing instance (utils.py:40-42,93)."""
        st = self.status.cpu().numpy() & 0xFF
        bad = np.nonzero(st)[0]
        if bad.size:
            if st[bad[0]] == 1:
                raise FloatingPointError("Non-finite values in chol_inv(A)")
            raise np.linalg.LinAlgError("chol_inv failed even with jitter")


def wrap_mask(wrap_idx: Optional[Sequence[int]]) -> int:
    mask = 0
    for i in (wrap_idx or []):
        mask |= 1 << int(i)
    return mask


def as_terminal_weight(alpha, n: int) -> np.ndarray:
    """utils.py:49-62 (host-side constant preparation)."""
    A = np.asarray(alpha, dtype=float)
    if A.ndim == 0:
        return float(A) * np.eye(n)
    if A.ndim == 1:
        if A.shape[0] != n:
            raise ValueError(f"terminal weight vector has shape {A.shape}, expected ({n},)")
        return np.diag(A)
    if A.ndim == 2:
        if A.shape != (n, n):
            raise ValueError(f"terminal weight matrix has shape {A.shape}, expected ({n},{n})")
        return 0.5 * (A + A.T)
    raise ValueError(f"unsupported terminal weight ndim={A.ndim}")


def _dev(t, device=None) -> torch.Tensor:
    if isinstance(t, torch.Tensor):
        out = t.to(dtype=torch.float64)
        if device is not None:
            out = out.to(device)
    else:
        out = torch.as_tensor(np.asarray(t, dtype=np.float64), device=device)
    if not out.is_cuda:
        raise _cabi.HopError("expected a CUDA tensor: the HOP B200 path has no CPU fallback")
    return out.contiguous()


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _params(F) -> np.ndarray:
    p = np.zeros(NPARAMS, dtype=np.float64)
    src = np.asarray(F.hop_params, dtype=np.float64)
    p[: src.size] = src
    return p


def _outputs(B, T_max, device, want_J=True):
    J = torch.empty((B, T_max), dtype=torch.float64, device=device) if want_J else None
    T = torch.empty(B, dtype=torch.int32, device=device)
    Js = torch.empty(B, dtype=torch.float64, device=device)
    st = torch.empty(B, dtype=torch.int32, device=device)
    return J, T, Js, st


def propagator_all_Jt_aug_batched(A_aug, B_aug, Q_aug, R_inv, z0, QT, T_min: int = 1, T_max: Optional[int] = None,
                                  w_explicit=None, mode: int = MODE_EXACT, tie_tol: Optional[float] = None) -> Selection:
    """Batched horizon_selection.propagator_all_Jt_aug + argmin.  Shapes: A_aug/Q_aug/QT [B,N,d,d],
    B_aug [B,N,d,m], R_inv [B,m,m] or [m,m], z0 [B,d] or [d].
    mode=MODE_VERIFIED needs tie_tol (finite, > 0): the relative gap below which an instance's two best horizons count as
    tied and the instance is recomputed in EXACT (hop_select_verified_f64).  T* equals EXACT's when FAST stays within
    tie_tol / 2 of EXACT on the caller's inputs; include/hop_b200.h gives measured values per input family."""
    if mode == MODE_VERIFIED:
        if tie_tol is None or not math.isfinite(float(tie_tol)) or not float(tie_tol) > 0.0:
            raise ValueError("mode=MODE_VERIFIED needs a finite tie_tol > 0 (the caller's tie tolerance, include/hop_b200.h)")
    elif tie_tol is not None:
        raise ValueError("tie_tol is only used with mode=MODE_VERIFIED")
    lib = _cabi.require_device()
    A_aug = _dev(A_aug)
    dev = A_aug.device
    B_aug, Q_aug, QT = _dev(B_aug, dev), _dev(Q_aug, dev), _dev(QT, dev)
    Bsz, N, d, _ = A_aug.shape
    m = B_aug.shape[-1]
    R_inv = _dev(R_inv, dev)
    if R_inv.dim() == 2:
        R_inv = R_inv.expand(Bsz, m, m).contiguous()
    rstride = m * m if R_inv.dim() == 4 else 0      # [B,N,m,m]: a different R^-1 per step
    z0 = _dev(z0, dev)
    if z0.dim() == 1:
        z0 = z0.expand(Bsz, d).contiguous()
    T_max = N if T_max is None else int(T_max)
    wx = None if w_explicit is None else _dev(w_explicit, dev).reshape(Bsz)
    J, T, Js, st = _outputs(Bsz, T_max, dev)
    with torch.cuda.device(dev):
        if mode == MODE_VERIFIED:
            rc = lib.hop_select_verified_f64(Bsz, N, d, m, int(T_min), T_max, _ptr(A_aug), _ptr(B_aug), _ptr(Q_aug), _ptr(R_inv),
                                             rstride, _ptr(z0), _ptr(QT), _ptr(wx), float(tie_tol), _ptr(J), _ptr(T), _ptr(Js),
                                             _ptr(st), _stream(dev))
            _cabi.check(rc, "hop_select_verified_f64")
            return Selection(J, T, Js, st)
        rc = lib.hop_select_f64(Bsz, N, d, m, int(T_min), T_max, _ptr(A_aug), _ptr(B_aug), _ptr(Q_aug), _ptr(R_inv),
                                rstride, _ptr(z0), _ptr(QT), _ptr(wx), mode, _ptr(J), _ptr(T), _ptr(Js), _ptr(st), _stream(dev))
    _cabi.check(rc, "hop_select_f64")
    return Selection(J, T, Js, st)


def select_fused_batched(A, Bm, X, U, xg, w, u_ref, Q, R, alpha, T_min: int, T_max: int, wrap_idx=None, a_resid=None,
                         q_reg: float = 1e-9, rho_reg: float = 1e-12, mode: int = MODE_EXACT) -> Selection:
    """Fused augmented.build_augmented_sequence_QR + build_terminal_aug_list + propagator + argmin.
    A [B,N,n,n], Bm [B,N,n,m], X [B,N+1,n], U [B,N,m] or shared [N,m], xg [B,n] or [n], w [B] or scalar."""
    lib = _cabi.require_device()
    A = _dev(A)
    dev = A.device
    Bm, X, U = _dev(Bm, dev), _dev(X, dev), _dev(U, dev)
    Bsz, N, n, _ = A.shape
    m = Bm.shape[-1]
    ustride = 0 if U.dim() == 2 else N * m
    xg = _dev(xg, dev)
    if xg.dim() == 1:
        xg = xg.expand(Bsz, n).contiguous()
    w = _dev(np.broadcast_to(np.asarray(w, dtype=float), (Bsz,)).copy() if not isinstance(w, torch.Tensor) else w, dev)
    u_ref, Q, R = _dev(u_ref, dev), _dev(Q, dev), _dev(R, dev)
    Qf = _dev(as_terminal_weight(alpha, n), dev)
    ar = None if a_resid is None else _dev(a_resid, dev)
    J, T, Js, st = _outputs(Bsz, int(T_max), dev)
    with torch.cuda.device(dev):
        rc = lib.hop_select_fused_f64(Bsz, N, n, m, int(T_min), int(T_max), _ptr(A), _ptr(Bm), _ptr(ar), _ptr(X), _ptr(U),
                                      ustride, _ptr(xg), _ptr(w), _ptr(u_ref), _ptr(Q), _ptr(R), _ptr(Qf),
                                      wrap_mask(wrap_idx), q_reg, rho_reg, mode, _ptr(J), _ptr(T), _ptr(Js), _ptr(st),
                                      _stream(dev))
    _cabi.check(rc, "hop_select_fused_f64")
    return Selection(J, T, Js, st)


def rollout_batched(F, x0, U, max_state_norm: float = 1e6) -> torch.Tensor:
    """solver.rollout over a batch: x0 [B,n], U [B,N,m] or shared [N,m] -> X [B,N+1,n]."""
    lib = _cabi.require_device()
    x0 = _dev(x0)
    dev = x0.device
    U = _dev(U, dev)
    n, m = SYS_DIMS[F.hop_sys]
    Bsz = x0.shape[0]
    N = U.shape[-2]
    ustride = 0 if U.dim() == 2 else N * m
    X = torch.empty((Bsz, N + 1, n), dtype=torch.float64, device=dev)
    p = _params(F)
    with torch.cuda.device(dev):
        rc = lib.hop_rollout_f64(Bsz, F.hop_sys, p.ctypes.data_as(C.c_void_p), N, _ptr(x0), _ptr(U), ustride,
                                 float(max_state_norm), _ptr(X), _stream(dev))
    _cabi.check(rc, "hop_rollout_f64")
    return X


def linearize_batched(F, X, U, central: bool = False, epsx=1e-5, epsu=1e-5, relx=1e-6, relu=1e-6):
    """linearization.linearize_{forward,central}_diff_traj over a batch -> A [B,N,n,n], Bm [B,N,n,m]."""
    lib = _cabi.require_device()
    X = _dev(X)
    dev = X.device
    U = _dev(U, dev)
    n, m = SYS_DIMS[F.hop_sys]
    Bsz = X.shape[0]
    N = U.shape[-2]
    ustride = 0 if U.dim() == 2 else N * m
    A = torch.empty((Bsz, N, n, n), dtype=torch.float64, device=dev)
    Bm = torch.empty((Bsz, N, n, m), dtype=torch.float64, device=dev)
    p = _params(F)
    with torch.cuda.device(dev):
        rc = lib.hop_linearize_f64(Bsz, F.hop_sys, p.ctypes.data_as(C.c_void_p), N, _ptr(X), _ptr(U), ustride,
                                   int(bool(central)), epsx, epsu, relx, relu, _ptr(A), _ptr(Bm), _stream(dev))
    _cabi.check(rc, "hop_linearize_f64")
    return A, Bm


class HorizonSelector:
    """Reusable x0 -> T* pipeline for one case (keeps the device workspace and constants alive).

    ``case`` is the reference's 13-tuple (hop.cases.make_*); U defaults to tile(u_ref) as in
    solver.py:480-481."""

    def __init__(self, case, B: int, device="cuda", central: bool = False, mode: int = MODE_EXACT, U=None):
        self.lib = _cabi.require_device()
        (self.F, _x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, extra) = case
        if extra is not None:
            raise NotImplementedError("extra_stage_cost is not supported on the B200 path")
        self.device = torch.device(device)
        self.B, self.N, self.T_min, self.T_max = int(B), int(N), int(T_min), int(min(T_max, N))
        self.n, self.m = SYS_DIMS[self.F.hop_sys]
        self.central, self.mode = bool(central), int(mode)
        self.wrap = wrap_mask(wrap_idx)
        self.params = _params(self.F)
        dev = self.device
        self.u_ref, self.Q, self.R = _dev(u_ref, dev), _dev(Q, dev), _dev(R, dev)
        self.Qf = _dev(as_terminal_weight(alpha, self.n), dev)
        self.xg_default = np.asarray(xg, dtype=float)
        self.w_default = float(w)
        if U is None:
            U = np.tile(np.asarray(u_ref, dtype=float).reshape(1, -1), (self.N, 1))
        self.U = _dev(U, dev)
        self.ustride = 0 if self.U.dim() == 2 else self.N * self.m
        nbytes = int(self.lib.hop_select_from_x0_workspace_bytes(self.B, self.N, self.n, self.m))
        self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self.J, self.T, self.Js, self.st = _outputs(self.B, self.T_max, dev)

    def views(self):
        """(X, A, Bm) views into the workspace after a call (for inspection / the solver loop)."""
        B, N, n, m = self.B, self.N, self.n, self.m
        al = lambda x: (x + 255) & ~255  # noqa: E731
        oX, sX = 0, al(8 * B * (N + 1) * n)
        sA = al(8 * B * N * n * n)
        X = self.workspace[oX:oX + 8 * B * (N + 1) * n].view(torch.float64).view(B, N + 1, n)
        A = self.workspace[sX:sX + 8 * B * N * n * n].view(torch.float64).view(B, N, n, n)
        Bm = self.workspace[sX + sA:sX + sA + 8 * B * N * n * m].view(torch.float64).view(B, N, n, m)
        return X, A, Bm

    def _goal_and_weight(self, xg, w):
        """xg -> [B, n], w -> [B] fp64 CUDA tensors (scalars / single goals are broadcast; shapes are checked: the kernel
        indexes xg[b*n + r] and w[b])."""
        dev = self.device
        if xg is None:
            xg = np.broadcast_to(self.xg_default, (self.B, self.n)).copy()
        xg = _dev(xg, dev)
        if xg.dim() == 1:
            xg = xg.expand(self.B, self.n).contiguous()
        if w is None:
            w = torch.full((self.B,), self.w_default, dtype=torch.float64, device=dev)
        elif not isinstance(w, torch.Tensor):
            w = np.broadcast_to(np.asarray(w, dtype=float), (self.B,)).copy()
        w = _dev(w, dev)
        if w.dim() == 0:
            w = w.expand(self.B).contiguous()
        if tuple(xg.shape) != (self.B, self.n) or tuple(w.shape) != (self.B,):
            raise ValueError(f"xg must be [{self.n}] or [{self.B},{self.n}] and w a scalar or [{self.B}]; "
                             f"got {tuple(xg.shape)} and {tuple(w.shape)}")
        return xg, w

    def select_resident(self, xg=None, w=None) -> Selection:
        """Fused selection on the (X, A, Bm) already resident in the workspace (no allocation, no copies):
        the kernel-only step bench.py times.  The returned Selection ALIASES the selector's output buffers (J, T_star,
        J_star, status are overwritten by the next call on this selector); clone what must outlive it."""
        X, A, Bm = self.views()
        dev = self.device
        xg, w = self._goal_and_weight(xg, w)
        with torch.cuda.device(dev):
            rc = self.lib.hop_select_fused_f64(
                self.B, self.N, self.n, self.m, self.T_min, self.T_max, _ptr(A), _ptr(Bm), None, _ptr(X), _ptr(self.U),
                self.ustride, _ptr(xg), _ptr(w), _ptr(self.u_ref), _ptr(self.Q), _ptr(self.R), _ptr(self.Qf), self.wrap,
                1e-9, 1e-12, self.mode, _ptr(self.J), _ptr(self.T), _ptr(self.Js), _ptr(self.st), _stream(dev))
        _cabi.check(rc, "hop_select_fused_f64")
        return Selection(self.J, self.T, self.Js, self.st)

    def __call__(self, x0: torch.Tensor, xg=None, w=None) -> Selection:
        """x0 [B, n] -> Selection.  The result aliases the selector's reused output buffers (see select_resident)."""
        dev = self.device
        x0 = _dev(x0, dev)
        if tuple(x0.shape) != (self.B, self.n):
            raise ValueError(f"x0 must be [{self.B},{self.n}], got {tuple(x0.shape)}")
        xg, w = self._goal_and_weight(xg, w)
        with torch.cuda.device(dev):
            rc = self.lib.hop_select_from_x0_f64(
                self.B, self.F.hop_sys, self.params.ctypes.data_as(C.c_void_p), self.N, self.T_min, self.T_max,
                _ptr(x0), _ptr(self.U), self.ustride, _ptr(xg), _ptr(w), _ptr(self.u_ref), _ptr(self.Q), _ptr(self.R),
                _ptr(self.Qf), self.wrap, int(self.central), self.mode, _ptr(self.workspace),
                self.workspace.numel(), _ptr(self.J), _ptr(self.T), _ptr(self.Js), _ptr(self.st), _stream(dev))
        _cabi.check(rc, "hop_select_from_x0_f64")
        return Selection(self.J, self.T, self.Js, self.st)


def select_horizon_batched(case, x0, xg=None, w=None, central: bool = False, mode: int = MODE_EXACT) -> Selection:
    """One-shot x0 [B,n] (CUDA tensor) -> Selection (owns its outputs: the selector is dropped)."""
    x0 = _dev(x0)
    sel = HorizonSelector(case, x0.shape[0], device=x0.device, central=central, mode=mode)
    return sel(x0, xg, w)


_HOST_BCAST = {}   # (kind, value bytes, B) -> pinned, already broadcast host array (case defaults are re-used across calls)


def _pinned_broadcast(kind: str, value, shape):
    """Broadcast a case default (goal state / weight) to the batch ONCE into pinned host memory: a fresh pageable
    array per call costs an allocation, a fill and a staged (synchronous) host-to-device copy of 6.8 MB at B = 65 536."""
    v = np.ascontiguousarray(value, dtype=np.float64)
    key = (kind, v.tobytes(), tuple(shape))
    buf = _HOST_BCAST.get(key)
    if buf is None:
        if len(_HOST_BCAST) > 16:
            _HOST_BCAST.clear()
        t = torch.empty(tuple(shape), dtype=torch.float64)
        if torch.cuda.is_available():
            t = t.pin_memory()
        buf = t.numpy()
        buf[...] = np.broadcast_to(v, shape)
        _HOST_BCAST[key] = buf
    return buf


def select_horizon_host(case, x0: np.ndarray, xg: Optional[np.ndarray] = None, w: Optional[np.ndarray] = None,
                        central: bool = False, mode: int = MODE_EXACT, want_curve: bool = True, out=None):
    """HOST-buffer entry (numpy in, numpy out): the library copies x0/xg/w to the device, runs
    rollout + linearisation + fused selection and copies T*, J*, status (and J) back.  Pass pinned
    arrays (``torch.empty(..., pin_memory=True).numpy()``) for asynchronous copies.
    Returns (J or None, T_star, J_star, status)."""
    lib = _cabi.require_device()
    F, _x0, xg0, u_ref, Q, R, alpha, w0, N, T_min, T_max, wrap_idx, extra = case
    if extra is not None:
        raise NotImplementedError("extra_stage_cost is not supported on the B200 path")
    n, m = SYS_DIMS[F.hop_sys]
    T_max = int(min(T_max, N))
    x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(-1, n)
    Bsz = x0.shape[0]
    xg = _pinned_broadcast("xg", xg0, (Bsz, n)) if xg is None else \
        np.ascontiguousarray(np.broadcast_to(np.asarray(xg, dtype=np.float64), (Bsz, n)))
    w = _pinned_broadcast("w", w0, (Bsz,)) if w is None else \
        np.ascontiguousarray(np.broadcast_to(np.asarray(w, dtype=np.float64), (Bsz,)))
    U = np.ascontiguousarray(np.tile(np.asarray(u_ref, dtype=np.float64).reshape(1, -1), (N, 1)))
    u_ref = np.ascontiguousarray(u_ref, dtype=np.float64)
    Q = np.ascontiguousarray(Q, dtype=np.float64)
    R = np.ascontiguousarray(R, dtype=np.float64)
    Qf = np.ascontiguousarray(as_terminal_weight(alpha, n))
    if out is None:
        J = np.empty((Bsz, T_max)) if want_curve else None
        T = np.empty(Bsz, dtype=np.int32); Js = np.empty(Bsz); st = np.empty(Bsz, dtype=np.int32)
    else:
        J, T, Js, st = out
    p = _params(F)
    vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = lib.hop_select_from_x0_host_f64(Bsz, F.hop_sys, vp(p), int(N), int(T_min), T_max, vp(x0), vp(U), 0, vp(xg), vp(w),
                                         vp(u_ref), vp(Q), vp(R), vp(Qf), wrap_mask(wrap_idx), int(bool(central)), mode,
                                         vp(J), vp(T), vp(Js), vp(st))
    _cabi.check(rc, "hop_select_from_x0_host_f64")
    return J, T, Js, st


# ------------------------------------------------------------------------------------------------
# HOP-DDP pieces and the batched solver (solver.py:449-765, method="propagator")
# ------------------------------------------------------------------------------------------------
def _case_consts(case, Bsz, dev, xg=None, w=None):
    F, _x0, xg0, u_ref, Q, R, alpha, w0, N, T_min, T_max, wrap_idx, extra = case
    if extra is not None:
        raise NotImplementedError("extra_stage_cost is not supported on the B200 path")
    n, m = SYS_DIMS[F.hop_sys]
    xg_t = _dev(np.broadcast_to(np.asarray(xg0, dtype=float), (Bsz, n)).copy(), dev) if xg is None else _dev(xg, dev)
    if xg_t.dim() == 1:
        xg_t = xg_t.expand(Bsz, n).contiguous()
    if w is None:
        w_t = torch.full((Bsz,), float(w0), dtype=torch.float64, device=dev)
    else:
        w_t = _dev(np.broadcast_to(np.asarray(w, dtype=float), (Bsz,)).copy() if not isinstance(w, torch.Tensor) else w, dev)
    return dict(F=F, n=n, m=m, N=int(N), T_min=int(T_min), T_max=int(min(T_max, N)), wrap=wrap_mask(wrap_idx), xg=xg_t, w=w_t,
                u_ref=_dev(u_ref, dev), Q=_dev(Q, dev), R=_dev(R, dev), Qf=_dev(as_terminal_weight(alpha, n), dev),
                params=_params(F))


def cost_timeopt_true_batched(case, X, U, T_star, xg=None, w=None) -> torch.Tensor:
    """solver.cost_timeopt_true over a batch, at per-instance horizons T_star [B] (int32)."""
    lib = _cabi.require_device()
    X = _dev(X)
    dev = X.device
    U = _dev(U, dev)
    Bsz = X.shape[0]
    c = _case_consts(case, Bsz, dev, xg, w)
    T = T_star.to(device=dev, dtype=torch.int32).contiguous()
    J = torch.empty(Bsz, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        rc = lib.hop_cost_f64(Bsz, c["N"], c["n"], c["m"], _ptr(X), _ptr(U), _ptr(c["xg"]), _ptr(c["w"]), _ptr(c["u_ref"]),
                              _ptr(c["Q"]), _ptr(c["R"]), _ptr(c["Qf"]), c["wrap"], _ptr(T), _ptr(J), _stream(dev))
    _cabi.check(rc, "hop_cost_f64")
    return J


def bruteforce_all_Jt_batched(case, A, Bm, X, U, T_max: Optional[int] = None, lm_lambda: float = 1e-6, xg=None, w=None):
    """solver.bruteforce_all_Jt_backward_expansion over a batch: (J [B, T_max] with J[b, T-1] = V0[0] of a Riccati sweep
    T -> 0, status [B]).  O(T_max^2 n^3) per instance: a comparator / cross-check, not the selection path."""
    lib = _cabi.require_device()
    X = _dev(X)
    dev = X.device
    A, Bm, U = _dev(A, dev), _dev(Bm, dev), _dev(U, dev)
    Bsz = X.shape[0]
    c = _case_consts(case, Bsz, dev, xg, w)
    N = A.shape[1]
    T_max = N if T_max is None else int(T_max)
    ustride = 0 if U.dim() == 2 else N * c["m"]
    J = torch.empty((Bsz, T_max), dtype=torch.float64, device=dev)
    st = torch.empty(Bsz, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.hop_bruteforce_jt_f64(Bsz, N, c["n"], c["m"], T_max, _ptr(A), _ptr(Bm), _ptr(X), _ptr(U), ustride, _ptr(c["xg"]),
                                       _ptr(c["w"]), _ptr(c["u_ref"]), _ptr(c["Q"]), _ptr(c["R"]), _ptr(c["Qf"]), c["wrap"],
                                       float(lm_lambda), _ptr(J), _ptr(st), _stream(dev))
    _cabi.check(rc, "hop_bruteforce_jt_f64")
    return J, st


def backward_linesearch_batched(case, A, Bm, X, U, T_star, lm, xg=None, w=None):
    """solver.backward_pass_truncated + forward_linesearch_fixedT over a batch.
    Returns dict(k, K, ok, err, X_new, U_new, J_new, accepted)."""
    lib = _cabi.require_device()
    A = _dev(A)
    dev = A.device
    Bm, X, U = _dev(Bm, dev), _dev(X, dev), _dev(U, dev)
    Bsz = A.shape[0]
    c = _case_consts(case, Bsz, dev, xg, w)
    N, n, m = c["N"], c["n"], c["m"]
    T = T_star.to(device=dev, dtype=torch.int32).contiguous()
    lm_t = _dev(np.broadcast_to(np.asarray(lm, dtype=float), (Bsz,)).copy() if not isinstance(lm, torch.Tensor) else lm, dev)
    k = torch.zeros((Bsz, N, m), dtype=torch.float64, device=dev)
    K = torch.zeros((Bsz, N, m, n), dtype=torch.float64, device=dev)
    ok = torch.zeros(Bsz, dtype=torch.int32, device=dev)
    err = torch.zeros(Bsz, dtype=torch.int32, device=dev)
    Xn = torch.empty_like(X)
    Un = torch.empty_like(U)
    Jn = torch.zeros(Bsz, dtype=torch.float64, device=dev)
    acc = torch.zeros(Bsz, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.hop_backward_linesearch_f64(Bsz, c["F"].hop_sys, c["params"].ctypes.data_as(C.c_void_p), N, _ptr(A), _ptr(Bm),
                                             _ptr(X), _ptr(U), _ptr(c["xg"]), _ptr(c["w"]), _ptr(c["u_ref"]), _ptr(c["Q"]),
                                             _ptr(c["R"]), _ptr(c["Qf"]), c["wrap"], _ptr(T), _ptr(lm_t), _ptr(k), _ptr(K),
                                             _ptr(ok), _ptr(err), _ptr(Xn), _ptr(Un), _ptr(Jn), _ptr(acc), _stream(dev))
    _cabi.check(rc, "hop_backward_linesearch_f64")
    return dict(k=k, K=K, ok=ok, err=err, X_new=Xn, U_new=Un, J_new=Jn, accepted=acc)


def ilqr_timeopt_batched(case, x0, xg=None, w=None, U_init=None, max_iter: int = 15, lm_init: float = 1e-3,
                         use_central_diff: bool = True, mode: int = MODE_EXACT):
    """Batched HOP-DDP solve (solver.ilqr_timeopt, method="propagator") for B instances (x0 [B,n], optional
    per-instance xg [B,n] and w [B]).  Returns a dict of CUDA tensors: X [B,N+1,n], U [B,N,m],
    J_hist / T_hist [B,max_iter+1] with n_hist [B] valid entries, J_curve [B,T_max], T_star [B], status [B],
    plus ``iters`` (outer iterations actually run)."""
    lib = _cabi.require_device()
    x0 = _dev(x0)
    dev = x0.device
    Bsz = x0.shape[0]
    c = _case_consts(case, Bsz, dev, xg, w)
    N, n, m, T_max = c["N"], c["n"], c["m"], c["T_max"]
    Ui = None
    if U_init is not None:
        Ui = _dev(U_init, dev)
        if Ui.dim() == 2:
            Ui = Ui.expand(Bsz, N, m).contiguous()
    cap = int(max_iter) + 1
    X = torch.empty((Bsz, N + 1, n), dtype=torch.float64, device=dev)
    U = torch.empty((Bsz, N, m), dtype=torch.float64, device=dev)
    J_hist = torch.full((Bsz, cap), float("nan"), dtype=torch.float64, device=dev)
    T_hist = torch.zeros((Bsz, cap), dtype=torch.int32, device=dev)
    n_hist = torch.zeros(Bsz, dtype=torch.int32, device=dev)
    J_curve = torch.zeros((Bsz, T_max), dtype=torch.float64, device=dev)
    T_star = torch.zeros(Bsz, dtype=torch.int32, device=dev)
    status = torch.zeros(Bsz, dtype=torch.int32, device=dev)
    nbytes = int(lib.hop_ilqr_workspace_bytes(Bsz, N, n, m))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    iters = C.c_int(0)
    timers = (C.c_double * 4)()
    with torch.cuda.device(dev):
        rc = lib.hop_ilqr_timeopt_f64(Bsz, c["F"].hop_sys, c["params"].ctypes.data_as(C.c_void_p), N, c["T_min"], T_max,
                                      _ptr(x0), _ptr(Ui), _ptr(c["xg"]), _ptr(c["w"]), _ptr(c["u_ref"]), _ptr(c["Q"]),
                                      _ptr(c["R"]), _ptr(c["Qf"]), c["wrap"], int(max_iter), float(lm_init),
                                      int(bool(use_central_diff)), int(mode), _ptr(ws), nbytes, _ptr(X), _ptr(U),
                                      _ptr(J_hist), _ptr(T_hist), _ptr(n_hist), _ptr(J_curve), _ptr(T_star), _ptr(status),
                                      C.cast(C.byref(iters), C.c_void_p), C.cast(timers, C.c_void_p), _stream(dev))
    _cabi.check(rc, "hop_ilqr_timeopt_f64")
    return dict(X=X, U=U, J_hist=J_hist, T_hist=T_hist, n_hist=n_hist, J_curve=J_curve, T_star=T_star, status=status,
                iters=iters.value,
                timers=dict(zip(("linearize", "select", "backward", "forward"), (float(v) for v in timers))))
