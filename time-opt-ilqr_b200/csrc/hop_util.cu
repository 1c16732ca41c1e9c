// hop_util.cu -- small batched utilities behind the drop-in module functions that are not on the
// fused fast path but belong to the reference API of the hot path:
//   k_chol_inv / k_chol_solve   utils.py:69-120            (one thread per matrix, Cholesky route exactly as
//                                                            the reference: L, L^-1, L^-T L^-1; ladder; LU fallback)
//   k_affine_residuals          linearization.py:269-270
//   k_build_augmented           augmented.py:10-60          (materialises A_aug, B_aug, Q_aug in HBM)
//   k_build_terminal            augmented.py:63-87
#include "hop_common.cuh"
#include "hop_ddp_core.cuh"
#include "../../include/hop_b200.h"

namespace hop {

constexpr int kMaxD = 16;

__device__ bool chol_lower_dyn(int d, const double* M, double* Lo) {
    for (int i = 0; i < d * d; ++i) Lo[i] = 0.0;
    for (int j = 0; j < d; ++j) {
        double ajj = M[j * d + j];
        for (int p = 0; p < j; ++p) ajj = sub(ajj, mul(Lo[j * d + p], Lo[j * d + p]));
        if (!(ajj > 0.0)) return false;
        ajj = sqrt(ajj);
        Lo[j * d + j] = ajj;
        const double rinv = 1.0 / ajj;
        for (int i = j + 1; i < d; ++i) {
            double s = M[i * d + j];
            for (int p = 0; p < j; ++p) s = sub(s, mul(Lo[i * d + p], Lo[j * d + p]));
            Lo[i * d + j] = mul(s, rinv);
        }
    }
    return true;
}
__device__ void chol_subst_dyn(int d, int c, const double* Lo, const double* Bm, double* X) {
    double Y[kMaxD];
    for (int col = 0; col < c; ++col) {
        for (int i = 0; i < d; ++i) {
            double s = Bm ? Bm[i * c + col] : (i == col ? 1.0 : 0.0);
            for (int p = 0; p < i; ++p) s = sub(s, mul(Lo[i * d + p], Y[p]));
            Y[i] = s / Lo[i * d + i];
        }
        for (int i = d - 1; i >= 0; --i) {
            double s = Y[i];
            for (int p = i + 1; p < d; ++p) s = sub(s, mul(Lo[p * d + i], X[p * c + col]));
            X[i * c + col] = s / Lo[i * d + i];
        }
    }
}
__device__ bool lu_inverse_dyn(int d, double* A, double* X) {
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) X[i * d + j] = (i == j) ? 1.0 : 0.0;
    for (int j = 0; j < d; ++j) {
        int piv = j;
        double best = fabs(A[j * d + j]);
        for (int i = j + 1; i < d; ++i) { const double v = fabs(A[i * d + j]); if (v > best) { best = v; piv = i; } }
        if (A[piv * d + j] == 0.0) return false;
        if (piv != j)
            for (int q = 0; q < d; ++q) {
                double t = A[j * d + q]; A[j * d + q] = A[piv * d + q]; A[piv * d + q] = t;
                t = X[j * d + q]; X[j * d + q] = X[piv * d + q]; X[piv * d + q] = t;
            }
        const double rinv = 1.0 / A[j * d + j];
        for (int i = j + 1; i < d; ++i) {
            const double f = A[i * d + j] * rinv;
            for (int q = j + 1; q < d; ++q) A[i * d + q] -= f * A[j * d + q];
            for (int q = 0; q < d; ++q) X[i * d + q] -= f * X[j * d + q];
        }
    }
    for (int c = 0; c < d; ++c)
        for (int i = d - 1; i >= 0; --i) {
            double s = X[i * d + c];
            for (int p = i + 1; p < d; ++p) s -= A[i * d + p] * X[p * d + c];
            X[i * d + c] = s / A[i * d + i];
        }
    return true;
}

// utils.py:69-93 (c == 0: inverse) and utils.py:96-120 (c > 0: solve, no fallback)
__global__ void k_chol(int B, int d, int c, const double* A, const double* Bm, double* X, double jitter, int max_tries,
                       int* status) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double S[kMaxD * kMaxD], M[kMaxD * kMaxD], Lo[kMaxD * kMaxD];
    const double* Ab = A + (size_t)b * d * d;
    const double* Bb = c ? Bm + (size_t)b * d * c : nullptr;
    double* Xb = X + (size_t)b * d * (c ? c : d);
    bool fin = true;
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) { S[i * d + j] = 0.5 * add(Ab[i * d + j], Ab[j * d + i]); fin = fin && isfinite(S[i * d + j]); }
    if (c) for (int i = 0; i < d * c; ++i) fin = fin && isfinite(Bb[i]);
    int st = 0;
    if (!fin) { status[b] = HOP_ST_NONFINITE; return; }
    double eps = jitter;
    for (int t = 0; t < max_tries; ++t) {
        for (int i = 0; i < d * d; ++i) M[i] = S[i];
        for (int i = 0; i < d; ++i) M[i * d + i] = add(S[i * d + i], eps);
        if (chol_lower_dyn(d, M, Lo)) {
            chol_subst_dyn(d, c ? c : d, Lo, Bb, Xb);
            bool xfin = true;
            if (c) for (int i = 0; i < d * c; ++i) xfin = xfin && isfinite(Xb[i]);
            if (xfin) { status[b] = st; return; }
        }
        st |= HOP_ST_FLAG_RETRY;
        eps *= 10.0;
    }
    if (c) { status[b] = st | HOP_ST_LINALG; return; }           // chol_solve raises
    for (int i = 0; i < d * d; ++i) M[i] = S[i];
    for (int i = 0; i < d; ++i) M[i * d + i] = add(S[i * d + i], eps);
    st |= HOP_ST_FLAG_LU;
    if (!lu_inverse_dyn(d, M, Xb)) st |= HOP_ST_LINALG;
    status[b] = st;
}

template <int SYS>
__global__ void k_affine_residuals(int B, DynParams prm, int N, const double* X, const double* U, long ustride, double* a) {
    constexpr int n = SysDims<SYS>::n, m = SysDims<SYS>::m;
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)B * N) return;
    const size_t b = gid / N;
    const int k = (int)(gid % N);
    double x[n], u[m], f[n];
    for (int i = 0; i < n; ++i) x[i] = X[(b * (N + 1) + k) * n + i];
    for (int i = 0; i < m; ++i) u[i] = U[b * ustride + (size_t)k * m + i];
    dynamics<SYS>(prm.p, x, u, f);
    for (int i = 0; i < n; ++i) a[gid * n + i] = sub(f[i], X[(b * (N + 1) + k + 1) * n + i]);
}

// augmented.py:31-56 for one (instance, step); generic n <= 15, m <= 8
__global__ void k_build_augmented(int B, int N, int n, int m, const double* A, const double* Bm, const double* a,
                                  const double* X, const double* U, long ustride, const double* xg, const double* w,
                                  const double* u_ref, const double* Q, unsigned wrap_mask, double q_reg, double rho_reg,
                                  double* A_aug, double* B_aug, double* Q_aug) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)B * N) return;
    const size_t b = gid / N;
    const int k = (int)(gid % N);
    const int d = n + 1;
    double e[kMaxD], du[8], Qe[kMaxD];
    for (int i = 0; i < n; ++i) {
        double v = sub(X[(b * (N + 1) + k) * n + i], xg[b * n + i]);
        if ((wrap_mask >> i) & 1u) v = wrap_pi(v);
        e[i] = v;
    }
    for (int i = 0; i < m; ++i) du[i] = sub(U[b * ustride + (size_t)k * m + i], u_ref[i]);
    double eQe = 0.0;
    for (int i = 0; i < n; ++i) { double s = 0.0; for (int j = 0; j < n; ++j) s = add(s, mul(Q[i * n + j], e[j])); Qe[i] = s; }
    for (int j = 0; j < n; ++j) { double s = 0.0; for (int i = 0; i < n; ++i) s = add(s, mul(e[i], Q[i * n + j])); eQe = add(eQe, mul(s, e[j])); }
    double* Qk = Q_aug + gid * d * d;
    double* Ak = A_aug + gid * d * d;
    double* Bk = B_aug + gid * d * m;
    const double* As = A + gid * n * n;
    const double* Bs = Bm + gid * n * m;
    for (int i = 0; i < n; ++i) {
        for (int j = 0; j < n; ++j) {
            Qk[i * d + j] = add(0.5 * add(Q[i * n + j], Q[j * n + i]), (i == j) ? q_reg : 0.0);
            Ak[i * d + j] = As[i * n + j];
        }
        Qk[i * d + n] = Qe[i];
        Qk[n * d + i] = Qe[i];
        double Bdu = 0.0;
        for (int j = 0; j < m; ++j) { Bdu = add(Bdu, mul(Bs[i * m + j], du[j])); Bk[i * m + j] = Bs[i * m + j]; }
        Ak[i * d + n] = sub(a ? a[gid * n + i] : 0.0, Bdu);
        Ak[n * d + i] = 0.0;
    }
    Qk[n * d + n] = add(add(eQe, mul(2.0, w[b])), rho_reg);
    Ak[n * d + n] = 1.0;
    for (int j = 0; j < m; ++j) Bk[n * m + j] = 0.0;
}

// augmented.py:78-86: QT[t-1] from X[t]
__global__ void k_build_terminal(int B, int N, int n, const double* X, const double* xg, const double* Qf,
                                 unsigned wrap_mask, double rho_reg, double* QT) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)B * N) return;
    const size_t b = gid / N;
    const int t = (int)(gid % N) + 1;
    const int d = n + 1;
    double e[kMaxD], px[kMaxD];
    for (int i = 0; i < n; ++i) {
        double v = sub(X[(b * (N + 1) + t) * n + i], xg[b * n + i]);
        if ((wrap_mask >> i) & 1u) v = wrap_pi(v);
        e[i] = v;
    }
    double ePe = 0.0;
    for (int i = 0; i < n; ++i) {
        double s = 0.0;
        for (int j = 0; j < n; ++j) s = add(s, mul(0.5 * add(Qf[i * n + j], Qf[j * n + i]), e[j]));
        px[i] = s;
    }
    for (int i = 0; i < n; ++i) ePe = add(ePe, mul(e[i], px[i]));
    double* Qt = QT + gid * d * d;
    for (int i = 0; i < n; ++i) {
        for (int j = 0; j < n; ++j) Qt[i * d + j] = 0.5 * add(Qf[i * n + j], Qf[j * n + i]);
        Qt[i * d + n] = px[i];
        Qt[n * d + i] = px[i];
    }
    Qt[n * d + n] = add(mul(2.0, mul(0.5, ePe)), rho_reg);
}

// fused HOP_MODE_SCAN: per-instance copies of the shared R^-1 and z0 = e_d (augmented.py:23,59) for the LQR-boundary kernel
__global__ void k_scan_consts(int B, int d, int m, const double* R_inv1, double* R_inv, double* z0) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nr = (size_t)B * m * m, nz = (size_t)B * d;
    if (gid < nr) R_inv[gid] = R_inv1[gid % (m * m)];
    if (gid < nz) z0[gid] = ((int)(gid % d) == d - 1) ? 1.0 : 0.0;
}

int launch_chol(int B, int d, int c, const double* A, const double* Bm, double* X, double jitter, int max_tries, int* status,
                cudaStream_t st) {
    k_chol<<<grid1(B, 64), 64, 0, st>>>(B, d, c, A, Bm, X, jitter, max_tries, status);
    return check_launch("k_chol");
}
int launch_scan_consts(int B, int d, int m, const double* R_inv1, double* R_inv, double* z0, cudaStream_t st) {
    const size_t total = (size_t)B * (m * m > d ? m * m : d);
    k_scan_consts<<<grid1(total, 128), 128, 0, st>>>(B, d, m, R_inv1, R_inv, z0);
    return check_launch("k_scan_consts");
}
int launch_affine_residuals(int B, int sys, const double* params_host, int N, const double* X, const double* U, long ustride,
                            double* a, cudaStream_t st) {
    const DynParams prm = dyn_params(params_host);
    const int g = grid1((size_t)B * N, 128);
    return with_system(sys, "hop_affine_residuals_f64", [&](auto s) {
        k_affine_residuals<decltype(s)::value><<<g, 128, 0, st>>>(B, prm, N, X, U, ustride, a);
        return check_launch("k_affine_residuals");
    });
}
int launch_build_augmented(int B, int N, int n, int m, const double* A, const double* Bm, const double* a, const double* X,
                           const double* U, long ustride, const double* xg, const double* w, const double* u_ref,
                           const double* Q, unsigned wrap_mask, double q_reg, double rho_reg, double* A_aug, double* B_aug,
                           double* Q_aug, cudaStream_t st) {
    k_build_augmented<<<grid1((size_t)B * N, 128), 128, 0, st>>>(B, N, n, m, A, Bm, a, X, U, ustride, xg, w, u_ref, Q, wrap_mask,
                                                                 q_reg, rho_reg, A_aug, B_aug, Q_aug);
    return check_launch("k_build_augmented");
}
int launch_build_terminal(int B, int N, int n, const double* X, const double* xg, const double* Qf, unsigned wrap_mask,
                          double rho_reg, double* QT, cudaStream_t st) {
    k_build_terminal<<<grid1((size_t)B * N, 128), 128, 0, st>>>(B, N, n, X, xg, Qf, wrap_mask, rho_reg, QT);
    return check_launch("k_build_terminal");
}

}  // namespace hop
