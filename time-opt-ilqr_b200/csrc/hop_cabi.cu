// hop_cabi.cu -- extern "C" surface of libhop_b200.so (see include/hop_b200.h for the contract).
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "hop_common.cuh"
#include "hop_select_body.cuh"
#include "../../include/hop_b200.h"

namespace hop {
static thread_local std::string g_err;
void set_last_error(const char* msg) { g_err = msg ? msg : ""; }
int report_cuda(cudaError_t e, const char* where) {
    if (e == cudaSuccess) return 0;
    g_err = std::string(where) + ": " + cudaGetErrorString(e);
    return (int)e;
}
static int need_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        set_last_error("no CUDA device visible: libhop_b200 has no CPU fallback");
        return HOP_E_NO_DEVICE;
    }
    return 0;
}
static const double kJitter = 1e-9;   // utils.py:69 defaults
static const int kMaxTries = 8;

namespace {
// 1 <= T_min <= T_max <= N for a batch of B >= 0 instances, and R^-1 given per instance (stride 0) or per step (m * m)
bool window_ok(int B, int N, int T_min, int T_max, long rinv_step_stride = 0, int m = 0) {
    return B >= 0 && N >= 1 && T_min >= 1 && T_min <= T_max && T_max <= N &&
           (rinv_step_stride == 0 || rinv_step_stride == (long)m * m);
}

// consecutive 256-byte-aligned regions of a caller's buffer; a null base only measures (the *_workspace_bytes queries)
struct Carve {
    char* base;
    size_t off = 0;
    template <typename T>
    T* take(size_t count) {
        char* q = base ? base + off : nullptr;
        off += (sizeof(T) * count + 255) & ~(size_t)255;
        return (T*)q;
    }
};

// workspace of the x0 pipeline: X | A | Bm
struct X0Ws {
    double *X, *A, *Bm;
    size_t total;
};
X0Ws x0_layout(char* base, int B, int N, int n, int m) {
    Carve c{base};
    X0Ws w;
    w.X = c.take<double>((size_t)B * (N + 1) * n);
    w.A = c.take<double>((size_t)B * N * n * n);
    w.Bm = c.take<double>((size_t)B * N * n * m);
    w.total = c.off;
    return w;
}

// x0 -> T* on stream st: rollout (solver.py:42), forward-difference linearisation (linearization.py:177,216), fused selection
int select_from_x0(int B, int sys, const double* params_host, int N, int n, int m, int T_min, int T_max, const double* x0,
                   const double* U, long u_batch_stride, const double* xg, const double* w, const double* u_ref, const double* Q,
                   const double* R, const double* Qf, unsigned wrap_mask, int central, int mode, const X0Ws& ws, double* J_out,
                   int* Tstar_out, double* Jstar_out, int* status, cudaStream_t st) {
    if (int rc = dispatch_rollout(B, sys, params_host, N, x0, U, u_batch_stride, 1e6, ws.X, st)) return rc;
    // X comes from the rollout above, so F(X_k, U_k) = X[k+1] bit for bit: the linearisation may read f0 from it
    if (int rc = dispatch_linearize(B, sys, params_host, N, ws.X, U, u_batch_stride, central, 1e-5, 1e-5, 1e-6, 1e-6, 1, nullptr,
                                    ws.A, ws.Bm, st))
        return rc;
    // a_resid = NULL: on a trajectory produced by the rollout above F(X_k,U_k) - X_{k+1} is exactly 0
    return hop_select_fused_f64(B, N, n, m, T_min, T_max, ws.A, ws.Bm, nullptr, ws.X, U, u_batch_stride, xg, w, u_ref, Q, R, Qf,
                                wrap_mask, 1e-9, 1e-12, mode, J_out, Tstar_out, Jstar_out, status, st);
}
}  // namespace
}  // namespace hop

using namespace hop;

extern "C" {

int hop_abi_version(void) { return HOP_ABI_VERSION; }
const char* hop_version(void) { return "hop_b200 0.1 (sm_100a, fp64)"; }
const char* hop_last_error_string(void) { return g_err.c_str(); }
int hop_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return n;
}
int hop_select_supported(int d, int m) {
    return (d == 3 && m == 1) || (d == 4 && m == 2) || (d == 5 && m == 1) || (d == 12 && m == 4) || (d == 13 && m == 4);
}
int hop_select_supported_mode(int d, int m, int mode) {
    if (mode == HOP_MODE_EXACT || mode == HOP_MODE_FP32) return d >= 1 && d <= 16 && m >= 1 && m <= 16;
    if (mode == HOP_MODE_SCAN) return (d == 12 || d == 13) && m == 4;
    if (mode == HOP_MODE_FAST || mode == HOP_MODE_GJ) return hop_select_supported(d, m);
    if (mode == HOP_MODE_VERIFIED) return hop_select_supported(d, m) && verify_tie_tol(d - 1) > 0.0;   // fused forms only
    return 0;
}

int hop_select_f64(int B, int N, int d, int m, int T_min, int T_max, const double* A_aug, const double* B_aug,
                   const double* Q_aug, const double* R_inv, long rinv_step_stride, const double* z0, const double* QT,
                   const double* w_explicit, int mode, double* J_out, int* Tstar_out, double* Jstar_out, int* status,
                   void* stream) {
    if (!window_ok(B, N, T_min, T_max, rinv_step_stride, m) || mode < HOP_MODE_EXACT || mode > HOP_MODE_FP32) {
        set_last_error("hop_select_f64: bad argument (need 1 <= T_min <= T_max <= N, rinv_step_stride in {0, m*m})");
        return HOP_E_BADARG;
    }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    SelectArgs p{B, N, T_min, T_max, kJitter, kMaxTries, A_aug, B_aug, Q_aug, R_inv, z0, QT, rinv_step_stride, w_explicit,
                 J_out, Tstar_out, Jstar_out, status, nullptr, nullptr, nullptr, g_generic_nodiag};
    return dispatch_select_generic(d, m, mode, p, (cudaStream_t)stream);
}

int hop_select_verified_f64(int B, int N, int d, int m, int T_min, int T_max, const double* A_aug, const double* B_aug,
                            const double* Q_aug, const double* R_inv, long rinv_step_stride, const double* z0, const double* QT,
                            const double* w_explicit, double tie_tol, double* J_out, int* Tstar_out, double* Jstar_out,
                            int* status, void* stream) {
    if (!window_ok(B, N, T_min, T_max, rinv_step_stride, m) || !(std::isfinite(tie_tol) && tie_tol > 0.0)) {
        set_last_error("hop_select_verified_f64: bad argument (need 1 <= T_min <= T_max <= N, rinv_step_stride in {0, m*m}, "
                       "finite tie_tol > 0)");
        return HOP_E_BADARG;
    }
    if (!hop_select_supported(d, m)) {
        set_last_error("hop_select_verified_f64: (d, m) has no FAST kernel; supported: (3,1) (4,2) (5,1) (12,4) (13,4)");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    SelectArgs p{B, N, T_min, T_max, kJitter, kMaxTries, A_aug, B_aug, Q_aug, R_inv, z0, QT, rinv_step_stride, w_explicit,
                 J_out, Tstar_out, Jstar_out, status, nullptr, nullptr, nullptr, g_generic_nodiag};
    return dispatch_select_generic_verified(d, m, tie_tol, p, (cudaStream_t)stream);
}

int hop_select_fused_f64(int B, int N, int n, int m, int T_min, int T_max, const double* A, const double* Bm,
                         const double* a_resid, const double* X, const double* U, long u_batch_stride,
                         const double* xg, const double* w,
                         const double* u_ref, const double* Q, const double* R, const double* Qf, unsigned wrap_mask,
                         double q_reg, double rho_reg, int mode, double* J_out, int* Tstar_out, double* Jstar_out,
                         int* status, void* stream) {
    if (!window_ok(B, N, T_min, T_max) || (mode != HOP_MODE_EXACT && mode != HOP_MODE_FAST && mode != HOP_MODE_GJ &&
                                          mode != HOP_MODE_SCAN && mode != HOP_MODE_VERIFIED)) {
        set_last_error("hop_select_fused_f64: bad argument (need 1 <= T_min <= T_max <= N, mode in {EXACT, FAST, GJ, SCAN, VERIFIED})");
        return HOP_E_BADARG;
    }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    FusedArgs p{B, N, T_min, T_max, kJitter, kMaxTries, A, Bm, a_resid, X, U, u_batch_stride, xg, w, u_ref, Q, R, Qf,
                wrap_mask, q_reg, rho_reg, mode, nullptr, J_out, Tstar_out, Jstar_out, status};
    return dispatch_select_fused(n, m, p, (cudaStream_t)stream);
}

int hop_rollout_f64(int B, int sys, const double* params_host, int N, const double* x0, const double* U,
                    long u_batch_stride, double max_state_norm, double* X, void* stream) {
    if (B < 0 || N < 1 || !params_host) { set_last_error("hop_rollout_f64: bad argument"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    return dispatch_rollout(B, sys, params_host, N, x0, U, u_batch_stride, max_state_norm, X, (cudaStream_t)stream);
}

int hop_linearize_f64(int B, int sys, const double* params_host, int N, const double* X, const double* U,
                      long u_batch_stride, int central, double epsx, double epsu, double relx, double relu, double* A,
                      double* Bm, void* stream) {
    if (B < 0 || N < 1 || !params_host) { set_last_error("hop_linearize_f64: bad argument"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    return dispatch_linearize(B, sys, params_host, N, X, U, u_batch_stride, central, epsx, epsu, relx, relu, 0, nullptr, A, Bm,
                              (cudaStream_t)stream);
}

unsigned long long hop_select_from_x0_workspace_bytes(int B, int N, int n, int m) {
    return (unsigned long long)x0_layout(nullptr, B, N, n, m).total;
}

int hop_select_from_x0_f64(int B, int sys, const double* params_host, int N, int T_min, int T_max, const double* x0,
                           const double* U, long u_batch_stride, const double* xg, const double* w,
                           const double* u_ref, const double* Q, const double* R, const double* Qf, unsigned wrap_mask,
                           int central, int mode, void* workspace, unsigned long long workspace_bytes, double* J_out,
                           int* Tstar_out, double* Jstar_out, int* status, void* stream) {
    int n = 0, m = 0;
    if (int rc = sys_dims(sys, "hop_select_from_x0_f64", &n, &m)) return rc;
    if (workspace_bytes < hop_select_from_x0_workspace_bytes(B, N, n, m) || (!workspace && B > 0)) {
        set_last_error("hop_select_from_x0_f64: workspace too small");
        return HOP_E_WORKSPACE;
    }
    if (B == 0) return 0;
    if (B < 0 || N < 1 || !params_host) { set_last_error("hop_select_from_x0_f64: bad argument"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    return select_from_x0(B, sys, params_host, N, n, m, T_min, T_max, x0, U, u_batch_stride, xg, w, u_ref, Q, R, Qf, wrap_mask,
                          central, mode, x0_layout((char*)workspace, B, N, n, m), J_out, Tstar_out, Jstar_out, status,
                          (cudaStream_t)stream);
}

// ---- utilities of the reference API (utils.py, linearization.py:269, augmented.py) -----------------------
int hop_chol_inv_f64(int B, int d, const double* A, double* X, double jitter, int max_tries, int* status, void* stream) {
    if (d < 1 || d > 16 || B < 0) { set_last_error("hop_chol_inv_f64: need 1 <= d <= 16"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    return launch_chol(B, d, 0, A, nullptr, X, jitter, max_tries, status, (cudaStream_t)stream);
}
int hop_chol_solve_f64(int B, int d, int c, const double* A, const double* Bm, double* X, double jitter, int max_tries,
                       int* status, void* stream) {
    if (d < 1 || d > 16 || c < 1 || B < 0) { set_last_error("hop_chol_solve_f64: need 1 <= d <= 16, c >= 1"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    return launch_chol(B, d, c, A, Bm, X, jitter, max_tries, status, (cudaStream_t)stream);
}
int hop_affine_residuals_f64(int B, int sys, const double* params_host, int N, const double* X, const double* U,
                             long u_batch_stride, double* a_out, void* stream) {
    if (int rc = need_device()) return rc;
    if (B <= 0) return B == 0 ? 0 : HOP_E_BADARG;
    return launch_affine_residuals(B, sys, params_host, N, X, U, u_batch_stride, a_out, (cudaStream_t)stream);
}
int hop_build_augmented_f64(int B, int N, int n, int m, const double* A, const double* Bm, const double* a_resid,
                            const double* X, const double* U, long u_batch_stride, const double* xg, const double* w,
                            const double* u_ref, const double* Q, unsigned wrap_mask, double q_reg, double rho_reg,
                            double* A_aug, double* B_aug, double* Q_aug, void* stream) {
    if (n < 1 || n > 15 || m < 1 || m > 8) { set_last_error("hop_build_augmented_f64: need n <= 15, m <= 8"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    if (B <= 0) return B == 0 ? 0 : HOP_E_BADARG;
    return launch_build_augmented(B, N, n, m, A, Bm, a_resid, X, U, u_batch_stride, xg, w, u_ref, Q, wrap_mask, q_reg, rho_reg,
                                  A_aug, B_aug, Q_aug, (cudaStream_t)stream);
}
int hop_build_terminal_f64(int B, int N, int n, const double* X, const double* xg, const double* Qf, unsigned wrap_mask,
                           double rho_reg, double* QT, void* stream) {
    if (n < 1 || n > 15) { set_last_error("hop_build_terminal_f64: need n <= 15"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    if (B <= 0) return B == 0 ? 0 : HOP_E_BADARG;
    return launch_build_terminal(B, N, n, X, xg, Qf, wrap_mask, rho_reg, QT, (cudaStream_t)stream);
}

// ---- HOP-DDP pieces and the batched solver loop --------------------------------------------------------
int hop_cost_f64(int B, int N, int n, int m, const double* X, const double* U, const double* xg, const double* w,
                 const double* u_ref, const double* Q, const double* R, const double* Qf, unsigned wrap_mask,
                 const int* T_star, double* J_out, void* stream) {
    if (int rc = need_device()) return rc;
    if (B <= 0) return B == 0 ? 0 : HOP_E_BADARG;
    if (N < 1 || !X || !U || !xg || !w || !u_ref || !Q || !R || !Qf || !T_star || !J_out) {
        set_last_error("hop_cost_f64: null pointer or N < 1");
        return HOP_E_BADARG;
    }
    DdpConst c{xg, w, u_ref, Q, R, Qf, wrap_mask};
    return dispatch_cost(n, m, B, N, X, U, c, T_star, J_out, (cudaStream_t)stream);
}

int hop_bruteforce_jt_f64(int B, int N, int n, int m, int T_max, const double* A, const double* Bm, const double* X,
                          const double* U, long u_batch_stride, const double* xg, const double* w, const double* u_ref,
                          const double* Q, const double* R, const double* Qf, unsigned wrap_mask, double lm_lambda,
                          double* J_out, int* status, void* stream) {
    if (!window_ok(B, N, 1, T_max)) { set_last_error("hop_bruteforce_jt_f64: need 1 <= T_max <= N"); return HOP_E_BADARG; }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    DdpConst c{xg, w, u_ref, Q, R, Qf, wrap_mask};
    return dispatch_bruteforce(n, m, B, N, T_max, A, Bm, X, U, u_batch_stride, c, lm_lambda, J_out, status, (cudaStream_t)stream);
}

int hop_backward_linesearch_f64(int B, int sys, const double* params_host, int N, const double* A, const double* Bm,
                                const double* X, const double* U, const double* xg, const double* w, const double* u_ref,
                                const double* Q, const double* R, const double* Qf, unsigned wrap_mask, const int* T_star,
                                const double* lm, double* k_out, double* K_out, int* ok_out, int* err_out, double* X_new,
                                double* U_new, double* J_new, int* accepted, void* stream) {
    if (int rc = need_device()) return rc;
    if (B <= 0) return B == 0 ? 0 : HOP_E_BADARG;
    if (N < 1 || !params_host || !A || !Bm || !X || !U || !xg || !w || !u_ref || !Q || !R || !Qf || !T_star || !lm || !k_out ||
        !K_out || !ok_out || !err_out || !X_new || !U_new || !J_new || !accepted) {
        set_last_error("hop_backward_linesearch_f64: null pointer or N < 1");
        return HOP_E_BADARG;
    }
    DdpConst c{xg, w, u_ref, Q, R, Qf, wrap_mask};
    // the stand-alone entry point is the API-parity path: the reference's summation order
    return dispatch_backward_linesearch(sys, B, params_host, N, A, Bm, X, U, c, T_star, lm, nullptr, k_out, K_out, ok_out,
                                        err_out, X_new, U_new, J_new, accepted, true, nullptr, (cudaStream_t)stream);
}

int hop_linesearch_f64(int B, int sys, const double* params_host, int N, const double* X, const double* U, const double* xg,
                       const double* w, const double* u_ref, const double* Q, const double* R, const double* Qf,
                       unsigned wrap_mask, const int* T_star, const double* k_list, const double* K_list, const int* ok,
                       double* X_new, double* U_new, double* J_new, int* accepted, void* stream) {
    if (int rc = need_device()) return rc;
    if (B <= 0) return B == 0 ? 0 : HOP_E_BADARG;
    if (N < 1 || !params_host || !X || !U || !xg || !w || !u_ref || !Q || !R || !Qf || !T_star || !k_list || !K_list || !X_new ||
        !U_new || !J_new || !accepted) {
        set_last_error("hop_linesearch_f64: null pointer or N < 1");
        return HOP_E_BADARG;
    }
    DdpConst c{xg, w, u_ref, Q, R, Qf, wrap_mask};
    return dispatch_linesearch(sys, B, params_host, N, X, U, c, T_star, k_list, K_list, ok, X_new, U_new, J_new, accepted,
                               (cudaStream_t)stream);
}

namespace {
struct IlqrWs {
    double *A, *Bm, *Xn, *Un, *kl, *Kl, *lm, *Jn, *Jstar;
    int *T_bar, *T_sel, *ok, *acc, *bw_err, *done, *copy, *sel_status, *n_active;
    size_t total;
};
IlqrWs ilqr_layout(char* base, int B, int N, int n, int m) {
    Carve c{base};
    IlqrWs w;
    w.A = c.take<double>((size_t)B * N * n * n);
    w.Bm = c.take<double>((size_t)B * N * n * m);
    w.Xn = c.take<double>((size_t)B * (N + 1) * n);
    w.Un = c.take<double>((size_t)B * N * m);
    w.kl = c.take<double>((size_t)B * N * m);
    w.Kl = c.take<double>((size_t)B * N * m * n);
    w.lm = c.take<double>(B);
    w.Jn = c.take<double>(B);
    w.Jstar = c.take<double>(B);
    w.T_bar = c.take<int>(B);
    w.T_sel = c.take<int>(B);
    w.ok = c.take<int>(B);
    w.acc = c.take<int>(B);
    w.bw_err = c.take<int>(B);
    w.done = c.take<int>(B);
    w.copy = c.take<int>(B);
    w.sel_status = c.take<int>(B);
    w.n_active = c.take<int>(4);
    w.total = c.off;
    return w;
}
}  // namespace

unsigned long long hop_ilqr_workspace_bytes(int B, int N, int n, int m) {
    return (unsigned long long)ilqr_layout(nullptr, B, N, n, m).total;
}

int hop_ilqr_timeopt_f64(int B, int sys, const double* params_host, int N, int T_min, int T_max, const double* x0,
                         const double* U_init, const double* xg, const double* w, const double* u_ref, const double* Q,
                         const double* R, const double* Qf, unsigned wrap_mask, int max_iter, double lm_init, int central,
                         int mode, void* workspace, unsigned long long workspace_bytes, double* X, double* U,
                         double* J_hist, int* T_hist, int* n_hist, double* J_curve, int* T_star, int* status,
                         int* iters_run_host, double* timers_host, void* stream) {
    int n = 0, m = 0;
    if (int rc = sys_dims(sys, "hop_ilqr_timeopt_f64", &n, &m)) return rc;
    if (!window_ok(B, N, T_min, T_max) || max_iter < 0 ||
        (mode != HOP_MODE_EXACT && mode != HOP_MODE_FAST && mode != HOP_MODE_GJ && mode != HOP_MODE_VERIFIED)) {
        set_last_error("hop_ilqr_timeopt_f64: bad argument (need 1 <= T_min <= T_max <= N, max_iter >= 0, mode in {EXACT, FAST, GJ, "
                       "VERIFIED})");
        return HOP_E_BADARG;
    }
    if (mode == HOP_MODE_VERIFIED && !hop_select_supported_mode(n + 1, m, mode)) {
        set_last_error("hop_ilqr_timeopt_f64: HOP_MODE_VERIFIED has no calibrated tie tolerance for this system (include/hop_b200.h)");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    if (int rc = need_device()) return rc;
    if (B == 0) return 0;
    if (!workspace || workspace_bytes < hop_ilqr_workspace_bytes(B, N, n, m)) {
        set_last_error("hop_ilqr_timeopt_f64: workspace too small");
        return HOP_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    IlqrWs ws = ilqr_layout((char*)workspace, B, N, n, m);
    const int cap = max_iter + 1;
    const long ustride = (long)N * m;
    DdpConst c{xg, w, u_ref, Q, R, Qf, wrap_mask};
    // VERIFIED selects with FAST + EXACT re-evaluation (same T* and status low byte as EXACT); everything after the selection
    // runs as in an EXACT solve, so that the whole solve reproduces EXACT's
    const bool ordered = (mode == HOP_MODE_EXACT || mode == HOP_MODE_VERIFIED);
    int rc;
#define HOP_TRY(x) do { rc = (x); if (rc) return rc; } while (0)
    auto select = [&](const int* skip) -> int {
        FusedArgs p{B, N, T_min, T_max, kJitter, kMaxTries, ws.A, ws.Bm, nullptr, X, U, ustride, xg, w, u_ref, Q, R, Qf,
                    wrap_mask, 1e-9, 1e-12, mode, skip, J_curve, ws.T_sel, ws.Jstar, ws.sel_status};
        return dispatch_select_fused(n, m, p, st);
    };
    // optional per-phase device timing (the reference's timers dict: linearize / select / backward / forward): five events per
    // outer iteration, all read after the loop -- nothing here makes the host wait for the device
    const int n_sets = max_iter + 1;
    struct Events {   // destroyed on every exit path
        std::vector<cudaEvent_t> e;
        cudaEvent_t done[2] = {nullptr, nullptr};
        ~Events() {
            for (auto& x : e) if (x) cudaEventDestroy(x);
            for (auto& x : done) if (x) cudaEventDestroy(x);
        }
    } evs;
    double tsum[4] = {0.0, 0.0, 0.0, 0.0};
    if (timers_host) {
        evs.e.assign((size_t)5 * n_sets, nullptr);
        for (auto& e : evs.e) HOP_TRY(report_cuda(cudaEventCreate(&e), "cudaEventCreate"));
    }
    for (auto& e : evs.done) HOP_TRY(report_cuda(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate"));
    int set = 0;                                                                     // event set of the current iteration
    auto ev = [&](int i) { return evs.e[(size_t)5 * set + i]; };
    auto mark = [&](int i) { if (timers_host) cudaEventRecord(ev(i), st); };
    // pinned landing zone of the per-iteration "instances still active" counter (one per host thread, kept for the process)
    static thread_local int* h_active = nullptr;
    if (!h_active) HOP_TRY(report_cuda(cudaHostAlloc((void**)&h_active, 2 * sizeof(int), cudaHostAllocDefault), "cudaHostAlloc"));
    HOP_TRY(launch_init_state(B, lm_init, ws.lm, ws.done, n_hist, status, st));
    if (U_init) HOP_TRY(report_cuda(cudaMemcpyAsync(U, U_init, sizeof(double) * (size_t)B * N * m, cudaMemcpyDeviceToDevice, st), "copy U_init"));
    else HOP_TRY(launch_tile_u(B, N, m, u_ref, U, st));                                                  // solver.py:480-481
    HOP_TRY(dispatch_rollout(B, sys, params_host, N, x0, U, ustride, 1e6, X, st));                       // :492
    mark(0);
    HOP_TRY(dispatch_linearize(B, sys, params_host, N, X, U, ustride, central, 1e-5, 1e-5, 1e-6, 1e-6, 1, nullptr, ws.A, ws.Bm, st));
    mark(1);
    HOP_TRY(select(nullptr));                                                                            // :516-522
    HOP_TRY(launch_after_select(B, ws.sel_status, ws.done, status, st));
    mark(2);
    HOP_TRY(dispatch_backward_linesearch(sys, B, params_host, N, ws.A, ws.Bm, X, U, c, ws.T_sel, ws.lm, ws.done, ws.kl, ws.Kl,
                                         ws.ok, ws.bw_err, ws.Xn, ws.Un, ws.Jn, ws.acc, ordered, timers_host ? ev(3) : nullptr, st));   // :541-551
    HOP_TRY(launch_warm_update(B, cap, ws.T_sel, ws.ok, ws.acc, ws.Jn, ws.bw_err, ws.done, ws.T_bar, J_hist, T_hist, n_hist,
                               ws.copy, status, st));
    HOP_TRY(launch_copy_accepted(B, (size_t)(N + 1) * n, (size_t)N * m, ws.copy, ws.Xn, ws.Un, X, U, st));
    mark(4);
    // Outer loop (:564).  The early exit ("every instance has stopped") is decided ONE ITERATION LATE: iteration `it` is
    // enqueued before the host looks at the counter of iteration it - 1, so the stream never drains while the host waits.
    // When that counter is zero the already enqueued iteration finds every instance done and changes nothing.
    int iters = 0, enqueued = 0;
    for (int it = 0; it < max_iter; ++it) {                                                              // :564
        const int slot = it & 1;
        set = it + 1;
        ++enqueued;
        mark(0);
        HOP_TRY(dispatch_linearize(B, sys, params_host, N, X, U, ustride, central, 1e-5, 1e-5, 1e-6, 1e-6, 1, ws.done, ws.A, ws.Bm, st));
        mark(1);
        HOP_TRY(select(ws.done));                                                                        // :581-590
        HOP_TRY(launch_after_select(B, ws.sel_status, ws.done, status, st));
        mark(2);
        HOP_TRY(dispatch_backward_linesearch(sys, B, params_host, N, ws.A, ws.Bm, X, U, c, ws.T_sel, ws.lm, ws.done, ws.kl,
                                             ws.Kl, ws.ok, ws.bw_err, ws.Xn, ws.Un, ws.Jn, ws.acc, ordered, timers_host ? ev(3) : nullptr, st)); // :594-604
        HOP_TRY(report_cuda(cudaMemsetAsync(ws.n_active + slot, 0, sizeof(int), st), "memset n_active"));
        HOP_TRY(launch_ddp_update(B, cap, ws.T_sel, ws.ok, ws.acc, ws.Jn, ws.bw_err, ws.done, ws.T_bar, ws.lm, J_hist, T_hist,
                                  n_hist, ws.copy, status, ws.n_active + slot, st));                      // :735-748
        HOP_TRY(launch_copy_accepted(B, (size_t)(N + 1) * n, (size_t)N * m, ws.copy, ws.Xn, ws.Un, X, U, st));
        mark(4);
        HOP_TRY(report_cuda(cudaMemcpyAsync(h_active + slot, ws.n_active + slot, sizeof(int), cudaMemcpyDeviceToHost, st), "read n_active"));
        HOP_TRY(report_cuda(cudaEventRecord(evs.done[slot], st), "cudaEventRecord"));
        iters = it + 1;
        if (it >= 1) {                                                                                   // look at iteration it - 1
            HOP_TRY(report_cuda(cudaEventSynchronize(evs.done[slot ^ 1]), "hop_ilqr_timeopt_f64"));
            if (h_active[slot ^ 1] == 0) { iters = it; break; }
        }
    }
    HOP_TRY(report_cuda(cudaStreamSynchronize(st), "hop_ilqr_timeopt_f64"));
    if (timers_host)
        for (int q = 0; q <= enqueued; ++q)
            for (int i = 0; i < 4; ++i) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, evs.e[(size_t)5 * q + i], evs.e[(size_t)5 * q + i + 1]);
                tsum[i] += 1e-3 * ms;
            }
    HOP_TRY(launch_finalize(B, cap, n_hist, T_hist, ws.T_bar, T_star, st));
#undef HOP_TRY
    if (iters_run_host) *iters_run_host = iters;
    if (timers_host)
        for (int i = 0; i < 4; ++i) timers_host[i] = tsum[i];
    return 0;
}

// ---- FP64 pipe probe (roofline denominator; MEASURED_PEAKS.json has no FP64 figure) ---------------
__global__ void k_probe_dfma(int iters, double seed, double* sink) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0 - 1e-9, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 12345.678) sink[0] = r;   // never true; keeps the chain alive
}

int hop_test_set_backward_variant(int variant) {
    const int old = g_backward_variant;
    if (variant >= 0 && variant <= 3) g_backward_variant = variant;
    return old;
}

int hop_test_set_linesearch_variant(int variant) {
    const int old = g_linesearch_variant;
    if (variant == 0 || variant == 1) g_linesearch_variant = variant;
    return old;
}

int hop_test_set_fused_small_variant(int variant) {
    const int old = g_fused_small_variant;
    if (variant >= 0 && variant <= 3) g_fused_small_variant = variant;
    return old;
}

int hop_test_set_generic_diag(int on) {
    const int old = g_generic_nodiag ? 0 : 1;
    if (on == 0 || on == 1) g_generic_nodiag = on ? 0 : 1;
    return old;
}

int hop_test_set_generic_pre(int on) {
    const int old = g_generic_pre;
    if (on >= -1 && on <= 1) g_generic_pre = on;
    return old;
}

long hop_test_set_tpp_min_batch(long min_batch) { return hop::tpp_min_batch(min_batch); }

int hop_test_set_linearize_variant(int variant) {
    const int old = g_linearize_variant;
    if (variant == 0 || variant == 2) g_linearize_variant = variant;
    return old;
}

int hop_probe_fp64_tflops(int iters, double* tflops_out, double* ms_out) {
    if (int rc = need_device()) return rc;
    if (iters < 1 || !tflops_out) { set_last_error("hop_probe_fp64_tflops: bad argument"); return HOP_E_BADARG; }
    cudaDeviceProp prop;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaGetDeviceProperties(&prop, dev);
    const int threads = 512, blocks = prop.multiProcessorCount * 4;
    double* sink = nullptr;
    if (int rc = report_cuda(cudaMalloc(&sink, sizeof(double)), "cudaMalloc(probe)")) return rc;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    k_probe_dfma<<<blocks, threads>>>(iters / 8 + 1, 0.5, sink);   // warm-up
    cudaEventRecord(e0);
    k_probe_dfma<<<blocks, threads>>>(iters, 0.5, sink);
    cudaEventRecord(e1);
    cudaError_t e = cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(sink);
    if (e != cudaSuccess) return report_cuda(e, "hop_probe_fp64_tflops");
    const double flops = 2.0 * 8.0 * 16.0 * (double)iters * (double)threads * (double)blocks;
    *tflops_out = flops / (ms * 1e-3) / 1e12;
    if (ms_out) *ms_out = ms;
    return 0;
}

// ---- host-buffer variant ------------------------------------------------------------------------
// The batch is cut into up to four chunks that alternate between two streams: while chunk c runs its three kernels,
// the J(T) block of chunk c-1 (the bulk of the device -> host traffic, 8 T_max bytes per instance) drains over PCIe
// and the inputs of chunk c+1 arrive, so only the first upload and the last download are exposed.  It also bounds
// the linearisation workspace (A, B: 1.7 KB per instance and step) to two chunks instead of the whole batch.
// Measured (profiles/r2_experiments.txt): one step = 44.3 ms against 43.7 ms of kernels (selection 39.4 + linearisation 3.6 +
// rollout 0.74).  Running the rollout / linearisation of every chunk on a high-priority stream, under the selection of the
// previous chunk, bought nothing (B200: 44.52 against 44.34 ms per step, profiles/r2_experiments.txt item 1).
namespace {
struct HostCtx {
    std::mutex mu;
    cudaStream_t stream[2] = {nullptr, nullptr};
    cudaEvent_t consts_ready = nullptr;
    void* buf = nullptr;
    size_t cap = 0;
    int device = -1;
    void reset() {
        if (buf) cudaFree(buf);
        for (auto& st : stream) { if (st) cudaStreamDestroy(st); st = nullptr; }
        if (consts_ready) cudaEventDestroy(consts_ready);
        buf = nullptr; cap = 0; consts_ready = nullptr;
    }
};
HostCtx g_host;
constexpr int kHostChunkMin = 16384;   // instances: below this a chunk no longer fills the machine for several waves
constexpr int kHostChunksMax = 4;
}  // namespace

int hop_select_from_x0_host_f64(int B, int sys, const double* params_host, int N, int T_min, int T_max,
                                const double* x0, const double* U, long u_batch_stride, const double* xg,
                                const double* w, const double* u_ref, const double* Q, const double* R,
                                const double* Qf, unsigned wrap_mask, int central, int mode, double* J_out,
                                int* Tstar_out, double* Jstar_out, int* status) {
    int n = 0, m = 0;
    if (int rc = sys_dims(sys, "hop_select_from_x0_host_f64", &n, &m)) return rc;
    if (int rc = need_device()) return rc;
    if (B <= 0) return B == 0 ? 0 : HOP_E_BADARG;
    std::lock_guard<std::mutex> lock(g_host.mu);
    int dev = 0;
    cudaGetDevice(&dev);
    if (g_host.device != dev) {   // one cached context per process; re-created when the current device changes
        g_host.reset();
        g_host.device = dev;
    }
    for (auto& st : g_host.stream)
        if (!st) { if (int rc = report_cuda(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "cudaStreamCreate")) return rc; }
    if (!g_host.consts_ready) {
        if (int rc = report_cuda(cudaEventCreateWithFlags(&g_host.consts_ready, cudaEventDisableTiming), "cudaEventCreate")) return rc;
    }
    int chunks = (B + kHostChunkMin - 1) / kHostChunkMin;
    chunks = chunks < 1 ? 1 : (chunks > kHostChunksMax ? kHostChunksMax : chunks);
    const int per = (((B + chunks - 1) / chunks) + 3) & ~3;       // whole CTAs of the selection kernel
    const int lanes = chunks > 1 ? 2 : 1;                         // workspaces (= streams) in use
    const bool shared_U = (u_batch_stride == 0);
    const size_t nU = shared_U ? (size_t)N * m : (size_t)B * N * m;
    // arena: x0 | xg | w | U | case constants | J | T* | status | J* | one x0-pipeline workspace per lane
    const size_t s_ws = x0_layout(nullptr, per, N, n, m).total;
    double *d_x0, *d_xg, *d_w, *d_U, *d_c, *d_J, *d_Js;
    int *d_T, *d_st;
    char* d_ws;
    auto carve = [&](char* base) {
        Carve a{base};
        d_x0 = a.take<double>((size_t)B * n);
        d_xg = a.take<double>((size_t)B * n);
        d_w = a.take<double>(B);
        d_U = a.take<double>(nU);
        d_c = a.take<double>((size_t)(m + 2 * n * n + m * m));
        d_J = a.take<double>((size_t)B * T_max);
        d_T = a.take<int>(B);
        d_st = a.take<int>(B);
        d_Js = a.take<double>(B);
        d_ws = a.take<char>(lanes * s_ws);
        return a.off;
    };
    const size_t total = carve(nullptr);
    if (total > g_host.cap) {
        if (g_host.buf) cudaFree(g_host.buf);
        g_host.buf = nullptr; g_host.cap = 0;
        if (int rc = report_cuda(cudaMalloc(&g_host.buf, total), "cudaMalloc(host-variant arena)")) return rc;
        g_host.cap = total;
    }
    carve((char*)g_host.buf);
    double* d_uref = d_c; double* d_Q = d_uref + m; double* d_R = d_Q + n * n; double* d_Qf = d_R + m * m;
    cudaStream_t s0 = g_host.stream[0];
    int rc = 0;
    auto copy = [&](void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t st, const char* what) {
        if (rc == 0) rc = report_cuda(cudaMemcpyAsync(dst, src, bytes, kind, st), what);
    };
    copy(d_uref, u_ref, sizeof(double) * m, cudaMemcpyHostToDevice, s0, "H2D u_ref");
    copy(d_Q, Q, sizeof(double) * n * n, cudaMemcpyHostToDevice, s0, "H2D Q");
    copy(d_R, R, sizeof(double) * m * m, cudaMemcpyHostToDevice, s0, "H2D R");
    copy(d_Qf, Qf, sizeof(double) * n * n, cudaMemcpyHostToDevice, s0, "H2D Qf");
    if (shared_U) copy(d_U, U, sizeof(double) * nU, cudaMemcpyHostToDevice, s0, "H2D U");
    if (rc == 0) rc = report_cuda(cudaEventRecord(g_host.consts_ready, s0), "cudaEventRecord");
    if (rc == 0 && lanes > 1) rc = report_cuda(cudaStreamWaitEvent(g_host.stream[1], g_host.consts_ready, 0), "cudaStreamWaitEvent");
    for (int c = 0; c < chunks && rc == 0; ++c) {
        const int b0 = c * per, cb = (B - b0) < per ? (B - b0) : per;
        if (cb <= 0) break;
        const int lane = c % lanes;
        cudaStream_t st = g_host.stream[lane];
        const size_t o = (size_t)b0;
        copy(d_x0 + o * n, x0 + o * n, sizeof(double) * (size_t)cb * n, cudaMemcpyHostToDevice, st, "H2D x0");
        copy(d_xg + o * n, xg + o * n, sizeof(double) * (size_t)cb * n, cudaMemcpyHostToDevice, st, "H2D xg");
        copy(d_w + o, w + o, sizeof(double) * (size_t)cb, cudaMemcpyHostToDevice, st, "H2D w");
        const double* dU = d_U;
        if (!shared_U) {
            copy(d_U + o * N * m, U + o * N * m, sizeof(double) * (size_t)cb * N * m, cudaMemcpyHostToDevice, st, "H2D U");
            dU = d_U + o * N * m;
        }
        if (rc) break;
        rc = select_from_x0(cb, sys, params_host, N, n, m, T_min, T_max, d_x0 + o * n, dU, u_batch_stride, d_xg + o * n, d_w + o,
                            d_uref, d_Q, d_R, d_Qf, wrap_mask, central, mode, x0_layout(d_ws + lane * s_ws, per, N, n, m),
                            d_J + o * T_max, d_T + o, d_Js + o, d_st + o, st);
        if (rc) break;
        if (J_out) copy(J_out + o * T_max, d_J + o * T_max, sizeof(double) * (size_t)cb * T_max, cudaMemcpyDeviceToHost, st, "D2H J");
        copy(Tstar_out + o, d_T + o, sizeof(int) * (size_t)cb, cudaMemcpyDeviceToHost, st, "D2H T*");
        if (Jstar_out) copy(Jstar_out + o, d_Js + o, sizeof(double) * (size_t)cb, cudaMemcpyDeviceToHost, st, "D2H J*");
        if (status) copy(status + o, d_st + o, sizeof(int) * (size_t)cb, cudaMemcpyDeviceToHost, st, "D2H status");
    }
    cudaError_t e0 = cudaStreamSynchronize(g_host.stream[0]);
    cudaError_t e1 = lanes > 1 ? cudaStreamSynchronize(g_host.stream[1]) : cudaSuccess;
    if (rc) return rc;
    return report_cuda(e0 != cudaSuccess ? e0 : e1, "hop_select_from_x0_host_f64");
}

}  // extern "C"
