// hop_select_ref_body.cuh -- HOP_MODE_EXACT: horizon selection in the REFERENCE'S OPERATION ORDER.
//
// Replaces (reference file:line, dmmsjtu-umich/time-opt-ilqr):
//   utils.py:35-37,69-93          _sym, chol_inv: Cholesky (LAPACK dpotf2 order, column scaled by the reciprocal of the
//                                 pivot) -> solve(L, I) -> solve(L^T, Y) as two substitutions; jitter 1e-9 on the first
//                                 try, x10 per failure, 8 tries, then LU with partial pivoting of A + eps I
//   augmented.py:10-87            homogeneous embedding (fused entry point)
//   horizon_selection.py:36-86    stage / prefix / query, products evaluated left to right as numpy does
//   solver.py:522,590             argmin over [T_min, T_max]
//
// This is the PARITY mode.  Every floating-point operation is an individually rounded IEEE multiply, add, divide or
// square root (no FMA contraction, no reciprocal approximations, no re-association), issued in the order a plain scalar
// loop restatement of the reference issues them.  On identical inputs the curve J(T) is therefore reproducible bit for bit
// by any IEEE-754 scalar implementation of the same loops -- which is what tests/ assert against the CPU oracle --, and
// T* agrees by construction.  The faster modes (HOP_MODE_FAST, HOP_MODE_GJ) are checked against this one.
//
// Mapping: one warp per problem; every block lives in the warp's shared-memory slab (row-major, row stride d); the lanes
// share the elements of a product (element idx = lane, lane + 32, ...), the rows of a Cholesky column and the columns of a
// substitution.  d and m are run-time values (<= 16): one instantiation serves every problem size.  R is the arithmetic
// type: double, or float for HOP_MODE_FP32 (hop_select_f64 only; inputs are converted on load, J is written as double).
#pragma once
#include "hop_select_body.cuh"
#include "../../include/hop_b200.h"

namespace hop { namespace ref {

constexpr int kMaxD = 16;

// ---- individually rounded arithmetic ------------------------------------------------------------------------------
#ifdef HOP_HOST_EMUL
HOP_DEVICE double mul(double a, double b) { return a * b; }
HOP_DEVICE double add(double a, double b) { return a + b; }
HOP_DEVICE double quo(double a, double b) { return a / b; }
HOP_DEVICE double root(double a) { return std::sqrt(a); }
HOP_DEVICE float mul(float a, float b) { volatile float r = a * b; return r; }
HOP_DEVICE float add(float a, float b) { volatile float r = a + b; return r; }
HOP_DEVICE float quo(float a, float b) { volatile float r = a / b; return r; }
HOP_DEVICE float root(float a) { return std::sqrt(a); }
#else
HOP_DEVICE double mul(double a, double b) { return __dmul_rn(a, b); }
HOP_DEVICE double add(double a, double b) { return __dadd_rn(a, b); }
HOP_DEVICE double quo(double a, double b) { return __ddiv_rn(a, b); }
HOP_DEVICE double root(double a) { return __dsqrt_rn(a); }
HOP_DEVICE float mul(float a, float b) { return __fmul_rn(a, b); }
HOP_DEVICE float add(float a, float b) { return __fadd_rn(a, b); }
HOP_DEVICE float quo(float a, float b) { return __fdiv_rn(a, b); }
HOP_DEVICE float root(float a) { return __fsqrt_rn(a); }
#endif
template <typename R>
HOP_DEVICE R sub(R a, R b) { return add(a, -b); }   // a - b and a + (-b) round identically

// ---- slab layout (units of R) -------------------------------------------------------------------------------------
struct Layout {
    int mat;                                                                      // doubles per d x d buffer (even)
    int A, Q, E, F, G, EB, FB, GB, W, T1, T2, T3, XT, MB, LB;                      // d x d (T3 shares Q's buffer, XT shares F's)
    int BM, T4;                                                                   // d x m
    int RI;                                                                       // m x m
    int Z0, V0, V1, V2, V3;                                                       // vectors (kMaxD)
    int size;
    HOP_HD static Layout make(int d, int m) {
        Layout l;
        l.mat = (d * d + 1) & ~1;
        int o = 0;
        l.A = o; o += l.mat; l.Q = o; o += l.mat; l.E = o; o += l.mat; l.F = o; o += l.mat; l.G = o; o += l.mat;
        l.EB = o; o += l.mat; l.FB = o; o += l.mat; l.GB = o; o += l.mat; l.W = o; o += l.mat;
        l.T1 = o; o += l.mat; l.T2 = o; o += l.mat;
        l.T3 = l.Q;     // Q_k is dead once E_k = chol_inv(Q_k) exists; T3 is first written after that
        l.XT = l.F;     // F_k is dead after the prefix update; the terminal block is staged there just before the query
        l.MB = o; o += l.mat; l.LB = o; o += l.mat;
        const int dm = (d * m + 1) & ~1;
        l.BM = o; o += dm; l.T4 = o; o += dm;
        l.RI = o; o += (m * m + 1) & ~1;
        l.Z0 = o; o += kMaxD; l.V0 = o; o += kMaxD; l.V1 = o; o += kMaxD; l.V2 = o; o += kMaxD; l.V3 = o; o += kMaxD;
        l.size = o;
        return l;
    }
};

// ---- products (numpy `@`: plain left-to-right accumulation from zero).  C must not alias A or B; callers sync. ------
template <typename R>   // C[r x c] = A[r x k] B[k x c]
HOP_DEVICE void mm(int lane, int r, int k, int c, const R* A, const R* B, R* C) {
    for (int idx = lane; idx < r * c; idx += 32) {
        const int i = idx / c, j = idx - i * c;
        R s = 0;
        for (int l = 0; l < k; ++l) s = add(s, mul(A[i * k + l], B[l * c + j]));
        C[idx] = s;
    }
}
template <typename R>   // C[r x c] = A[r x k] B^T, B is [c x k]
HOP_DEVICE void mmt(int lane, int r, int k, int c, const R* A, const R* B, R* C) {
    for (int idx = lane; idx < r * c; idx += 32) {
        const int i = idx / c, j = idx - i * c;
        R s = 0;
        for (int l = 0; l < k; ++l) s = add(s, mul(A[i * k + l], B[j * k + l]));
        C[idx] = s;
    }
}
template <typename R>   // C[r x c] = A^T B, A is [k x r], B is [k x c]
HOP_DEVICE void mtm(int lane, int r, int k, int c, const R* A, const R* B, R* C) {
    for (int idx = lane; idx < r * c; idx += 32) {
        const int i = idx / c, j = idx - i * c;
        R s = 0;
        for (int l = 0; l < k; ++l) s = add(s, mul(A[l * r + i], B[l * c + j]));
        C[idx] = s;
    }
}
template <typename R>   // utils.py:35-37: S = 0.5 (A + A^T); S must not alias A
HOP_DEVICE void sym(int lane, int d, const R* A, R* S) {
    for (int idx = lane; idx < d * d; idx += 32) {
        const int i = idx / d, j = idx - i * d;
        S[idx] = mul((R)0.5, add(A[idx], A[j * d + i]));
    }
}
template <typename R>   // C = A + sgn B, element-wise (C may alias A or B)
HOP_DEVICE void axpy(int lane, int len, const R* A, const R* B, bool minus, R* C) {
    for (int idx = lane; idx < len; idx += 32) C[idx] = minus ? sub(A[idx], B[idx]) : add(A[idx], B[idx]);
}
template <typename R>
HOP_DEVICE void copy(int lane, int len, const R* A, R* C) {
    for (int idx = lane; idx < len; idx += 32) C[idx] = A[idx];
}

// ---- np.linalg.cholesky = LAPACK dpotf2 ('L'): a_jj - sum_p l_jp^2 (p ascending), fail on a pivot <= 0 or NaN,
// column scaled by the reciprocal of the pivot's root.  Lane i owns row i; the pivot is computed by every lane.
template <typename R>
HOP_DEVICE bool cholesky(int lane, int d, const R* M, R* L) {
    for (int j = 0; j < d; ++j) {
        R ajj = M[j * d + j];
        for (int p = 0; p < j; ++p) ajj = sub(ajj, mul(L[j * d + p], L[j * d + p]));
        if (!(ajj > (R)0)) return false;                                          // warp-uniform
        ajj = root(ajj);
        const R rinv = quo((R)1, ajj);
        if (lane == j) L[j * d + j] = ajj;
        if (lane > j && lane < d) {
            R s = M[lane * d + j];
            for (int p = 0; p < j; ++p) s = sub(s, mul(L[lane * d + p], L[j * d + p]));
            L[lane * d + j] = mul(s, rinv);
        }
        simt::sync();
    }
    return true;
}

// utils.py:84-85: Y = solve(L, I), X = solve(L^T, Y) by substitution; lane c owns column c.  Y must not alias L or X.
template <typename R>
HOP_DEVICE void solve_factored_identity(int lane, int d, const R* L, R* Y, R* X) {
    if (lane < d) {
        const int c = lane;
        // column c of the identity: Y[i][c] = +0 for i < c, and the terms p < c of the later rows subtract L[i][p] * (+0)
        // = +-0 from s, which leaves every s (zero or not) unchanged bit for bit -- so those rows and terms are skipped
        for (int i = 0; i < c; ++i) Y[i * d + c] = (R)0;
        for (int i = c; i < d; ++i) {
            R s = (i == c) ? (R)1 : (R)0;
            for (int p = c; p < i; ++p) s = sub(s, mul(L[i * d + p], Y[p * d + c]));
            Y[i * d + c] = quo(s, L[i * d + i]);
        }
        for (int i = d - 1; i >= 0; --i) {
            R s = Y[i * d + c];
            for (int p = i + 1; p < d; ++p) s = sub(s, mul(L[p * d + i], X[p * d + c]));
            X[i * d + c] = quo(s, L[i * d + i]);
        }
    }
    simt::sync();
}

// utils.py:90-93: solve(A + eps I, I) = LAPACK dgesv (LU with partial pivoting), on one lane.  A (d x d, destroyed), X holds
// the identity on entry and the inverse on return.  Returns false on an exactly zero pivot (LinAlgError).
template <typename R>
HOP_DEVICE_NOINLINE bool lu_inverse_serial(int d, R* A, R* X) {
    for (int j = 0; j < d; ++j) {
        int piv = j;
        R best = A[j * d + j] < 0 ? -A[j * d + j] : A[j * d + j];
        for (int i = j + 1; i < d; ++i) {
            const R v = A[i * d + j] < 0 ? -A[i * d + j] : A[i * d + j];
            if (v > best) { best = v; piv = i; }
        }
        if (A[piv * d + j] == (R)0) return false;
        if (piv != j)
            for (int q = 0; q < d; ++q) {
                R t = A[j * d + q]; A[j * d + q] = A[piv * d + q]; A[piv * d + q] = t;
                t = X[j * d + q]; X[j * d + q] = X[piv * d + q]; X[piv * d + q] = t;
            }
        const R rinv = quo((R)1, A[j * d + j]);
        for (int i = j + 1; i < d; ++i) {
            const R f = mul(A[i * d + j], rinv);
            A[i * d + j] = f;
            for (int q = j + 1; q < d; ++q) A[i * d + q] = sub(A[i * d + q], mul(f, A[j * d + q]));
            for (int q = 0; q < d; ++q) X[i * d + q] = sub(X[i * d + q], mul(f, X[j * d + q]));
        }
    }
    for (int c = 0; c < d; ++c)
        for (int i = d - 1; i >= 0; --i) {
            R s = X[i * d + c];
            for (int p = i + 1; p < d; ++p) s = sub(s, mul(A[i * d + p], X[p * d + c]));
            X[i * d + c] = quo(s, A[i * d + i]);
        }
    return true;
}

// utils.py:69-93 chol_inv.  Ain (d x d, any), Xout (d x d) must be distinct from the work buffers Mb, Lb.  Returns
// ST_OK / ST_NONFINITE / ST_LINALG (warp-uniform); ST_FLAG_* are or-ed into `flags`.
template <typename R>
HOP_DEVICE int chol_inv(int lane, int d, const R* Ain, R* Xout, R* Mb, R* Lb, R jitter, int max_tries, int& flags) {
    bool fin = true;
    for (int idx = lane; idx < d * d; idx += 32) {
        const int i = idx / d, j = idx - i * d;
        fin = fin && isfinite((double)mul((R)0.5, add(Ain[idx], Ain[j * d + i])));
    }
    if (!simt::all(fin)) return ST_NONFINITE;                                     // utils.py:75
    R eps = jitter;
    for (int t = 0; t <= max_tries; ++t) {
        const bool lu = (t == max_tries);
        for (int idx = lane; idx < d * d; idx += 32) {
            const int i = idx / d, j = idx - i * d;
            const R s = mul((R)0.5, add(Ain[idx], Ain[j * d + i]));
            Mb[idx] = (i == j) ? add(s, eps) : s;
            if (lu) Xout[idx] = (i == j) ? (R)1 : (R)0;
        }
        simt::sync();
        if (lu) break;
        if (cholesky(lane, d, Mb, Lb)) {
            solve_factored_identity(lane, d, Lb, Mb, Xout);
            return ST_OK;
        }
        simt::sync();
        eps = mul(eps, (R)10);
        flags |= ST_FLAG_RETRY;
    }
    flags |= ST_FLAG_LU;
    bool ok = true;
    if (lane == 0) ok = lu_inverse_serial(d, Mb, Xout);
    ok = simt::all(ok);
    simt::sync();                                     // lane 0's stores to Xout are ordered before the warp reads them
    return ok ? ST_OK : ST_LINALG;
}

// ---- one step of the sweep on blocks already in the slab, in two halves (the terminal block of the query is staged in a
// buffer that is only free after the prefix update):
//   stage_prefix_step: stage k (horizon_selection.py:57-64) + prefix k (:66-75); on entry s+L.A = A_k, s+L.BM = B_k,
//                      s+L.Q = Q_k, s+L.RI = R^-1
//   query_step       : query t = k + 1 (:77-86); on entry s+L.XT = QT_t (raw), s+L.Z0 = z0; J(t) in *J_out
// Both return the error code of the first failing chol_inv (the reference raises there).
template <typename R>
HOP_DEVICE int stage_prefix_step(int lane, int d, int m, int k, const Layout& L, R* s, R jitter, int max_tries, int& flags) {
    const int dd = d * d;
    R *A = s + L.A, *Q = s + L.Q, *E = s + L.E, *F = s + L.F, *G = s + L.G, *EB = s + L.EB, *FB = s + L.FB, *GB = s + L.GB;
    R *W = s + L.W, *T1 = s + L.T1, *T2 = s + L.T2, *T3 = s + L.T3, *MB = s + L.MB, *LB = s + L.LB;
    R *BM = s + L.BM, *T4 = s + L.T4, *RI = s + L.RI;
    // stage: E_k = chol_inv(Q_k); F_k = E_k A_k^T; G_k = sym((A_k E_k) A_k^T + (B_k R^-1) B_k^T)
    if (int rc = chol_inv(lane, d, Q, E, MB, LB, jitter, max_tries, flags)) return rc;
    mmt(lane, d, d, d, E, A, F);
    mm(lane, d, d, d, A, E, T1);
    mm(lane, d, m, m, BM, RI, T4);
    simt::sync();
    mmt(lane, d, d, d, T1, A, T2);
    mmt(lane, d, m, d, T4, BM, T3);                   // (T3 = Q's buffer: Q_k is dead)
    simt::sync();
    axpy(lane, dd, T2, T3, false, T2);
    simt::sync();
    sym(lane, d, T2, G);
    simt::sync();
    if (k == 0) {
        copy(lane, dd, E, EB); copy(lane, dd, F, FB); copy(lane, dd, G, GB);
        simt::sync();
        return ST_OK;
    }
    // prefix: W = chol_inv(E_k + Gbar); Ebar <- sym(Ebar - (Fbar W) Fbar^T); Fbar <- (Fbar W) F_k;
    //         Gbar <- sym(G_k - (F_k^T W) F_k); every right-hand side uses the OLD Ebar, Fbar, Gbar
    axpy(lane, dd, E, GB, false, T1);
    simt::sync();
    if (int rc = chol_inv(lane, d, T1, W, MB, LB, jitter, max_tries, flags)) return rc;
    mm(lane, d, d, d, FB, W, T1);
    mtm(lane, d, d, d, F, W, T3);
    simt::sync();
    mmt(lane, d, d, d, T1, FB, T2);
    simt::sync();
    axpy(lane, dd, EB, T2, true, T2);
    mm(lane, d, d, d, T1, F, FB);                     // old Fbar is no longer read
    simt::sync();
    sym(lane, d, T2, EB);
    mm(lane, d, d, d, T3, F, T1);
    simt::sync();
    axpy(lane, dd, G, T1, true, T1);
    simt::sync();
    sym(lane, d, T1, GB);
    simt::sync();
    return ST_OK;
}

template <typename R>
HOP_DEVICE int query_step(int lane, int d, const Layout& L, R* s, R jitter, int max_tries, int& flags, R* J_out) {
    const int dd = d * d;
    R *EB = s + L.EB, *FB = s + L.FB, *GB = s + L.GB, *W = s + L.W, *T1 = s + L.T1, *T2 = s + L.T2, *T3 = s + L.T3;
    R *XT = s + L.XT, *MB = s + L.MB, *LB = s + L.LB, *Z0 = s + L.Z0, *V0 = s + L.V0;
    // query: X_t = chol_inv(QT_t); W_t = chol_inv(X_t + Gbar); X0 = sym(Ebar - (Fbar W_t) Fbar^T); P0 = chol_inv(X0)
    if (int rc = chol_inv(lane, d, XT, T1, MB, LB, jitter, max_tries, flags)) return rc;
    axpy(lane, dd, T1, GB, false, T1);
    simt::sync();
    if (int rc = chol_inv(lane, d, T1, W, MB, LB, jitter, max_tries, flags)) return rc;
    mm(lane, d, d, d, FB, W, T1);
    simt::sync();
    mmt(lane, d, d, d, T1, FB, T2);
    simt::sync();
    axpy(lane, dd, EB, T2, true, T2);
    simt::sync();
    sym(lane, d, T2, T3);
    simt::sync();
    if (int rc = chol_inv(lane, d, T3, T1, MB, LB, jitter, max_tries, flags)) return rc;
    // J = 0.5 z0^T P0 z0 evaluated as (z0^T P0) z0
    if (lane < d) {
        R v = 0;
        for (int i = 0; i < d; ++i) v = add(v, mul(Z0[i], T1[i * d + lane]));
        V0[lane] = v;
    }
    simt::sync();
    R acc = 0;
    for (int j = 0; j < d; ++j) acc = add(acc, mul(V0[j], Z0[j]));
    *J_out = mul((R)0.5, acc);
    simt::sync();
    return ST_OK;
}

// ---- LQR-boundary form: horizon_selection.py:36-86 on caller-provided augmented blocks ------------------------------
template <typename R>
HOP_DEVICE void select_generic_body(const SelectArgs& p, int d, int m, int b, R* s) {
    const int lane = simt::lane_id();
    const Layout L = Layout::make(d, m);
    const int dd = d * d, dm = d * m, mm_ = m * m;
    const size_t rinv_inst = (size_t)(p.rinv_step_stride ? p.N : 1) * mm_;
    for (int i = lane; i < mm_; i += 32) s[L.RI + i] = (R)p.R_inv[(size_t)b * rinv_inst + i];
    if (lane < d) s[L.Z0 + lane] = (R)p.z0[(size_t)b * d + lane];
    const double wexp = p.w_explicit ? p.w_explicit[b] : 0.0;
    const size_t base = (size_t)b * p.N;
    ArgMin am;
    am.init();
    int flags = 0, err = 0;
    for (int k = 0; k < p.T_max; ++k) {
        const double* Ak = p.A_aug + (base + k) * dd;
        const double* Qk = p.Q_aug + (base + k) * dd;
        const double* Tk = p.QT + (base + k) * dd;
        const double* Bk = p.B_aug + (base + k) * dm;
        simt::sync();
        for (int i = lane; i < dd; i += 32) { s[L.A + i] = (R)Ak[i]; s[L.Q + i] = (R)Qk[i]; }
        for (int i = lane; i < dm; i += 32) s[L.BM + i] = (R)Bk[i];
        if (p.rinv_step_stride)
            for (int i = lane; i < mm_; i += 32) s[L.RI + i] = (R)p.R_inv[(size_t)b * rinv_inst + (size_t)k * p.rinv_step_stride + i];
        simt::sync();
        R J = 0;
        err = stage_prefix_step<R>(lane, d, m, k, L, s, (R)p.jitter, p.max_tries, flags);
        if (!err) {
            for (int i = lane; i < dd; i += 32) s[L.XT + i] = (R)Tk[i];
            simt::sync();
            err = query_step<R>(lane, d, L, s, (R)p.jitter, p.max_tries, flags, &J);
        }
        if (err) {                                    // the reference raises: the rest of the curve is undefined
            if (lane == 0)
                for (int q = k; q < p.T_max; ++q) p.J_out[(size_t)b * p.T_max + q] = nan("");
            am.push(nan(""), k + 1 < p.T_min ? p.T_min : k + 1);
            break;
        }
        if (lane == 0) p.J_out[(size_t)b * p.T_max + k] = (double)J;
        const int t = k + 1;
        if (t >= p.T_min) am.push(simt::add_rn((double)J, simt::mul_rn(wexp, (double)t)), t);   // J + w t: two roundings
    }
    if (lane == 0) {
        p.T_out[b] = am.idx;
        p.Jstar_out[b] = am.best;
        p.status[b] = flags | err;
    }
}

// List mode of the LQR-boundary form (HOP_MODE_VERIFIED re-evaluation, fp64 only): this warp computes the instances
// list[first], list[first + stride], ... below count, each exactly as select_generic_body computes it, and then sets
// HOP_ST_FLAG_REEVALUATED in its status.  k_select_ref_generic passes its grid stride, the host emulation (0, 1).
HOP_DEVICE void select_generic_list(const SelectArgs& p, int d, int m, const int* list, int count, int first, int stride,
                                    double* s) {
    for (int i = first; i < count; i += stride) {
        const int b = list[i];
        simt::sync();                                                             // the previous instance's slab reads are done
        select_generic_body<double>(p, d, m, b, s);
        if (simt::lane_id() == 0) p.status[b] |= HOP_ST_FLAG_REEVALUATED;
    }
}

// ---- fused form: augmented.py:10-87 built in the slab, then the same sweep ------------------------------------------
// CTA-wide constants (doubles): Qs = sym(Q) [n x n], Qraw [n x n], P = sym(Qf) [n x n], u_ref [m], Rs = sym(R) [m x m]
struct FusedCst {
    int QS, QRAW, PF, UREF, RS, size;
    HOP_HD static FusedCst make(int n, int m) {
        FusedCst c;
        c.QS = 0; c.QRAW = n * n; c.PF = 2 * n * n; c.UREF = 3 * n * n; c.RS = c.UREF + ((m + 1) & ~1);
        c.size = c.RS + ((m * m + 1) & ~1);
        return c;
    }
};
HOP_DEVICE void fused_cst_fill(const FusedArgs& p, int n, int m, double* cst, int tid, int nthr) {
    const FusedCst C = FusedCst::make(n, m);
    for (int i = tid; i < n * n; i += nthr) {
        const int a = i / n, c = i % n;
        cst[C.QS + i] = mul(0.5, add(p.Q[a * n + c], p.Q[c * n + a]));            // augmented.py:32 sym(Q)
        cst[C.QRAW + i] = p.Q[i];
        cst[C.PF + i] = mul(0.5, add(p.Qf[a * n + c], p.Qf[c * n + a]));          // augmented.py:76
    }
    for (int i = tid; i < m; i += nthr) cst[C.UREF + i] = p.u_ref[i];
    for (int i = tid; i < m * m; i += nthr) {
        const int a = i / m, c = i % m;
        cst[C.RS + i] = mul(0.5, add(p.R[a * m + c], p.R[c * m + a]));            // augmented.py:23
    }
}

HOP_DEVICE void select_fused_body(const FusedArgs& p, int n, int m, int b, double* s, const double* cst) {
    typedef double R;
    const int lane = simt::lane_id();
    const int d = n + 1;
    const Layout L = Layout::make(d, m);
    const FusedCst C = FusedCst::make(n, m);
    const int dd = d * d, dm = d * m;
    R *A = s + L.A, *Q = s + L.Q, *XT = s + L.XT, *BM = s + L.BM, *RI = s + L.RI, *Z0 = s + L.Z0;
    R *V0 = s + L.V0, *V1 = s + L.V1, *V2 = s + L.V2, *V3 = s + L.V3;
    int flags = 0, err = 0;
    // R_inv = chol_inv(sym(R))  (augmented.py:23)
    for (int i = lane; i < m * m; i += 32) s[L.T1 + i] = cst[C.RS + i];
    simt::sync();
    err = chol_inv<R>(lane, m, s + L.T1, RI, s + L.MB, s + L.LB, p.jitter, p.max_tries, flags);
    if (lane < d) Z0[lane] = (lane == n) ? 1.0 : 0.0;                             // augmented.py:59
    const double w = p.w[b];
    const size_t baseN = (size_t)b * p.N, baseX = (size_t)b * (p.N + 1);
    const bool isx = lane < n;
    const double xg_l = isx ? p.xg[(size_t)b * n + lane] : 0.0;
    const bool wrap_l = isx && ((p.wrap_mask >> lane) & 1u);
    ArgMin am;
    am.init();
    int k = 0;
    for (; k < p.T_max && !err; ++k) {
        const double* Ak = p.A + (baseN + k) * n * n;
        const double* Bk = p.Bm + (baseN + k) * n * m;
        simt::sync();
        // e = wrap(X_k - xg), du = U_k - u_ref (augmented.py:27-29); the terminal error of t = k + 1 goes to V3
        if (isx) {
            double e = sub(p.X[(baseX + k) * n + lane], xg_l);
            if (wrap_l) e = wrap_pi(e);
            V0[lane] = e;
            double et = sub(p.X[(baseX + k + 1) * n + lane], xg_l);
            if (wrap_l) et = wrap_pi(et);
            V3[lane] = et;
        }
        if (lane < m) V1[lane] = sub(p.U[(size_t)b * p.u_stride + (size_t)k * m + lane], cst[C.UREF + lane]);
        for (int i = lane; i < dd; i += 32) { A[i] = 0.0; }
        for (int i = lane; i < dm; i += 32) BM[i] = 0.0;
        simt::sync();
        // A_aug = [[A_k, a_k - B_k du], [0, 1]], B_aug = [[B_k], [0]]  (augmented.py:50-56)
        for (int i = lane; i < n * n; i += 32) A[(i / n) * d + (i % n)] = Ak[i];
        for (int i = lane; i < n * m; i += 32) BM[i] = Bk[i];
        if (isx) {
            double bdu = 0.0;
            for (int j = 0; j < m; ++j) bdu = add(bdu, mul(Bk[lane * m + j], V1[j]));
            const double ak = p.a_resid ? p.a_resid[(baseN + k) * n + lane] : 0.0;
            A[lane * d + n] = sub(ak, bdu);
            // Q e and the column sums e^T Q (augmented.py:35-37)
            double qe = 0.0, qc = 0.0;
            for (int j = 0; j < n; ++j) qe = add(qe, mul(cst[C.QRAW + lane * n + j], V0[j]));
            for (int i = 0; i < n; ++i) qc = add(qc, mul(V0[i], cst[C.QRAW + i * n + lane]));
            Q[lane * d + n] = qe;
            Q[n * d + lane] = qe;
            V2[lane] = mul(qc, V0[lane]);
        }
        if (lane == n) A[n * d + n] = 1.0;
        for (int i = lane; i < n * n; i += 32) {
            const int a = i / n, c = i % n;
            Q[a * d + c] = add(cst[C.QS + i], a == c ? p.q_reg : 0.0);           // augmented.py:32
        }
        simt::sync();
        if (lane == 0) {
            double eQe = 0.0;
            for (int j = 0; j < n; ++j) eQe = add(eQe, V2[j]);
            Q[n * d + n] = add(add(eQe, mul(2.0, w)), p.rho_reg);                // augmented.py:37
        }
        simt::sync();
        double J = 0.0;
        err = stage_prefix_step<R>(lane, d, m, k, L, s, p.jitter, p.max_tries, flags);
        if (err) break;
        // terminal block of horizon t = k + 1 from X[k + 1] (augmented.py:78-86), staged in F_k's buffer (dead by now)
        for (int i = lane; i < n * n; i += 32) XT[(i / n) * d + (i % n)] = cst[C.PF + i];
        if (isx) {
            double px = 0.0;
            for (int j = 0; j < n; ++j) px = add(px, mul(cst[C.PF + lane * n + j], V3[j]));
            XT[lane * d + n] = px;
            XT[n * d + lane] = px;
            V1[lane] = mul(V3[lane], px);
        }
        simt::sync();
        if (lane == 0) {
            double ePe = 0.0;
            for (int i = 0; i < n; ++i) ePe = add(ePe, V1[i]);
            XT[n * d + n] = add(mul(2.0, mul(0.5, ePe)), p.rho_reg);
        }
        simt::sync();
        err = query_step<R>(lane, d, L, s, p.jitter, p.max_tries, flags, &J);
        if (err) break;
        if (lane == 0) p.J_out[(size_t)b * p.T_max + k] = J;
        if (k + 1 >= p.T_min) am.push(J, k + 1);
    }
    if (err) {
        if (lane == 0)
            for (int q = k; q < p.T_max; ++q) p.J_out[(size_t)b * p.T_max + q] = nan("");
        am.push(nan(""), k + 1 < p.T_min ? p.T_min : (k + 1 > p.T_max ? p.T_max : k + 1));   // NaN wins, as in np.argmin
    }
    if (lane == 0) {
        p.T_out[b] = am.idx;
        p.Jstar_out[b] = am.best;
        p.status[b] = flags | err;
    }
}

}}  // namespace hop::ref
