"""The selection kernels over the argument space include/hop_b200.h documents, beyond the shapes of the four cases: a
different R^-1 per step (R_inv [B][N][m][m], rinv_step_stride = m*m) in every kernel body that reads it, and the fused
EXACT body at odd (n, m).  The kernel sources run on the host SIMT emulator (tests/emul); CPU only.  The GPU run of the
same arguments through the C-ABI is tests/test_argspace_gpu.py.

Per-step R^-1 has two references:
  - the oracle's per-step path (oracle/hop_la.inc reloads R^-1 at every step), and
  - an independent one built on the single-R^-1 path only: R^-1 enters the sweep through B_k R_k^-1 B_k^T alone, so with
    R_k^-1 = L_k L_k^T the problem equals the one with B'_k = B_k L_k and R^-1 = I (up to rounding).  A step or instance
    offset the kernels and the oracle's per-step path got wrong in the same way would not survive this one.
R_k differ per step AND per instance and are not diagonal (_common.perstep_R): with a constant or diagonal R_k a wrong
offset would read the right numbers."""
import numpy as np
import pytest

import emul
import oracle as O
from _common import FUSED_NM, fused_batch, fused_oracle, perstep_problem, reference_b, rel


def check_against_references(J, T, st, A, Bm, Q, Rinv, z0, w, QT, T_min, T_max, tol):
    Jo, sto = O.propagator_batch(A, Bm, Q, Rinv, z0, QT, T_use=T_max)
    Jb = reference_b(A, Bm, Q, Rinv, z0, QT, T_max)
    Jb80 = reference_b(A, Bm, Q, Rinv, z0, QT, T_max, f80=True)
    assert not st.any() and not sto.any()
    assert rel(Jo, Jb80) <= 1e-12 and rel(Jb, Jb80) <= 1e-12     # the two references agree
    assert rel(J, Jo) <= tol and rel(J, Jb80) <= tol
    tot = Jo + w[:, None] * np.arange(1, T_max + 1)
    assert np.array_equal(T, np.argmin(tot[:, T_min - 1:], axis=1) + T_min)
    return Jo


def test_per_step_rinv_changes_the_curve():
    """The test problem is sensitive to the R^-1 of each step: R^-1 of step 0 everywhere, or the next instance's R^-1, moves
    the curve far beyond every tolerance below."""
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(5, 2, 12, 3)
    Jo, _ = O.propagator_batch(A, Bm, Q, Rinv, z0, QT)
    J0, _ = O.propagator_batch(A, Bm, Q, np.repeat(Rinv[:, :1], 12, 1), z0, QT)
    J1, _ = O.propagator_batch(A, Bm, Q, np.roll(Rinv, 1, axis=0), z0, QT)
    assert rel(J0, Jo) > 1e-3 and rel(J1, Jo) > 1e-3


# (body, emulator switch, instantiated (d, m)).  lanes: G-lane groups (hop_select_body.cuh); dmma: one warp per problem in
# DMMA fragments (hop_select_mma_body.cuh); pipe: the software-pipelined sweep (hop_select_gpipe_body.cuh), which stages
# R^-1 of step k + 1 while step k computes; scan: HOP_MODE_SCAN (hop_select_scan_body.cuh)
BODIES = [("lanes", {}, (3, 1)), ("lanes", {}, (4, 2)), ("lanes", {}, (5, 1)), ("lanes", {}, (12, 4)), ("lanes", {}, (13, 4)),
          ("dmma", {"mma": True}, (12, 4)), ("dmma", {"mma": True}, (13, 4)),
          ("pipe", {"pipe": True}, (12, 4)), ("pipe", {"pipe": True}, (13, 4))]


@pytest.mark.parametrize("body,kw,dm", BODIES, ids=[f"{b}-{d}x{m}" for b, _, (d, m) in BODIES])
def test_emulated_per_step_rinv(body, kw, dm):
    d, m = dm
    N, B, T_min, T_max = 12, 5, 2, 11                  # 5 instances: a ragged last warp for every lane-group width
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, B)
    J, T, Js, st = emul.select_generic(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w_explicit=w, **kw)
    check_against_references(J, T, st, A, Bm, Q, Rinv, z0, w, QT, T_min, T_max, 1e-12)


@pytest.mark.parametrize("d,m", [(12, 4), (13, 4)])
def test_emulated_scan_mode_per_step_rinv(d, m):
    """HOP_MODE_SCAN re-associates the prefix composition after chunk 0: chunk 0 is bit-identical to the sequential DMMA body,
    the rest within the scan's stated 1e-9 (hop_b200.h), both with per-step R^-1."""
    N, B, T_max = 19, 2, 19
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, B)
    Js, Ts, _, sts = emul.select_generic(A, Bm, Q, Rinv, z0, QT, 1, T_max, w_explicit=w, mma=True)
    Jp, Tp, _, stp = emul.select_generic(A, Bm, Q, Rinv, z0, QT, 1, T_max, w_explicit=w, scan=True)
    Lc = -(-T_max // 8)
    assert np.array_equal(Jp[:, :Lc], Js[:, :Lc])
    check_against_references(Jp, Tp, stp, A, Bm, Q, Rinv, z0, w, QT, 1, T_max, 1e-9)
    assert np.array_equal(Tp, Ts)


@pytest.mark.parametrize("d,m", [(1, 1), (3, 1), (4, 7), (5, 2), (13, 4), (16, 16)])
def test_emulated_exact_and_fp32_per_step_rinv(d, m):
    """EXACT: bit-identical to the oracle's per-step path.  FP32: within its stated 1e-4 of it."""
    N, B, T_min, T_max = 9, 2, 2, 8
    A, Bm, Q, Rinv, z0, w, QT = perstep_problem(d, m, N, B)
    J, T, Js, st = emul.select_generic(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w_explicit=w, ref=True)
    Jo = check_against_references(J, T, st, A, Bm, Q, Rinv, z0, w, QT, T_min, T_max, 1e-12)
    assert np.array_equal(J, Jo)
    J32, _, _, st32 = emul.select_generic(A, Bm, Q, Rinv, z0, QT, T_min, T_max, w_explicit=w, fp32=True)
    assert not st32.any() and rel(J32, Jo) <= 1e-4


@pytest.mark.parametrize("n,m", FUSED_NM)
def test_emulated_fused_exact_at_odd_dimensions(n, m):
    """Fused EXACT (hop_select_ref_body.cuh) at every documented corner of 1 <= n <= 15, m <= n + 1: bit-identical to the
    oracle, with affine residuals, one shared U, wrapped angles and a window 1 < T_min <= T_max < N."""
    N, B, T_min, T_max = 7, 2, 2, 6
    g = fused_batch(10 * n + m, B, n, m, N)
    J, T, Js, st = emul.select_fused(g["A"], g["Bm"], g["a"], g["X"], g["U"], g["xg"], g["w"], g["u_ref"], g["Q"], g["R"],
                                     O.as_terminal_weight(g["alpha"], n), O.wrap_mask(g["wrap_idx"]), T_min, T_max, ref=True)
    Jo, To = fused_oracle(g, T_min, T_max)
    assert not (st & 0xFF).any() and np.isfinite(Jo).all()
    assert np.array_equal(J, Jo) and np.array_equal(T, To)
    assert np.array_equal(Js, Jo[np.arange(B), To - 1])
