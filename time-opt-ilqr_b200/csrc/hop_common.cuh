// hop_common.cuh -- the host interface between the .cu translation units of libhop_b200.so.  Every function, hook global
// and struct that one of them uses from another is declared here, and every defining file includes this header, so the
// compiler checks each declaration against its definition.  Host-side only: no *_body.cuh includes it.
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <string>
#include <type_traits>

#include "../../include/hop_b200.h"

namespace hop {

struct SelectArgs;   // hop_select_body.cuh
struct FusedArgs;

// the HOP_NPARAMS parameters of a system (include/hop_b200.h), passed to its kernels by value
struct DynParams { double p[HOP_NPARAMS]; };
inline DynParams dyn_params(const double* params_host) {
    DynParams prm;
    for (int i = 0; i < HOP_NPARAMS; ++i) prm.p[i] = params_host[i];
    return prm;
}

// device pointers to the shared case constants + per-instance xg / w of the HOP-DDP kernels (passed to them by value)
struct DdpConst {
    const double *xg, *w, *u_ref, *Q, *R, *Qf;
    unsigned wrap_mask;
};

// ---- hop_cabi.cu
void set_last_error(const char* msg);
int report_cuda(cudaError_t e, const char* where);
inline int check_launch(const char* where) { return report_cuda(cudaGetLastError(), where); }
inline int grid1(size_t total, int threads) { return (int)((total + threads - 1) / threads); }

// f(std::integral_constant<int, SYS>{}) for the systems HOP_SYS_* (include/hop_b200.h); any other id is refused with
// "<where>: unknown system id"
template <typename F>
int with_system(int sys, const char* where, F&& f) {
    switch (sys) {
        case 0: return f(std::integral_constant<int, 0>{});
        case 1: return f(std::integral_constant<int, 1>{});
        case 2: return f(std::integral_constant<int, 2>{});
        case 3: return f(std::integral_constant<int, 3>{});
    }
    set_last_error((std::string(where) + ": unknown system id").c_str());
    return HOP_E_BADARG;
}

// ---- hop_select.cu
int dispatch_select_generic(int d, int m, int mode, const SelectArgs& p, cudaStream_t st);
int dispatch_select_fused(int n, int m, const FusedArgs& p, cudaStream_t st);
int stream_alloc(void** ptr, size_t bytes, cudaStream_t st, const char* what);
void stream_free(void* ptr, cudaStream_t st);
extern int g_generic_pre;
extern int g_generic_nodiag;

// ---- hop_select_tpp.cu: one problem per THREAD (d <= 5, large batches).  Returns HOP_E_UNSUPPORTED_DIMS without touching
// the error string when (d, m, p) is not for that kernel.
int dispatch_select_generic_tpp(int d, int m, const SelectArgs& p, cudaStream_t st);
long tpp_min_batch(long set_to);

// ---- hop_select_epl.cu: one matrix element per LANE, fused form of the small systems (same convention)
int dispatch_select_fused_epl(int n, int m, const FusedArgs& p, cudaStream_t st);
extern int g_fused_small_variant;

// ---- hop_select_ref.cu: HOP_MODE_EXACT / HOP_MODE_FP32, reference operation order
int dispatch_select_ref_generic(int d, int m, bool fp32, const SelectArgs& p, cudaStream_t st);
int launch_ref_generic_list(int d, int m, const SelectArgs& p, const int* list, const int* list_count, cudaStream_t st);
int launch_ref_fused_list(int n, int m, const FusedArgs& p, const int* list, const int* list_count, cudaStream_t st);

// ---- hop_verify.cu: HOP_MODE_VERIFIED, FAST + near-tie scan + EXACT on the marked instances
double verify_tie_tol(int n);
int dispatch_select_verified(int n, int m, const FusedArgs& p, cudaStream_t st);
int dispatch_select_generic_verified(int d, int m, double tol, const SelectArgs& p, cudaStream_t st);

// ---- hop_traj.cu
int dispatch_rollout(int B, int sys, const double* params_host, int N, const double* x0, const double* U, long ustride,
                     double max_norm, double* X, cudaStream_t st);
int dispatch_linearize(int B, int sys, const double* params_host, int N, const double* X, const double* U, long ustride,
                       int central, double epsx, double epsu, double relx, double relu, int f0_from_x, const int* skip,
                       double* A, double* Bm, cudaStream_t st);
int sys_dims(int sys, const char* where, int* n, int* m);
extern int g_linearize_variant;

// ---- hop_ddp.cu
int dispatch_backward_linesearch(int sys, int B, const double* params_host, int N, const double* A, const double* Bm,
                                 const double* X, const double* U, const DdpConst& c, const int* T, const double* lm,
                                 const int* done, double* kl, double* Kl, int* ok, int* bw_err, double* Xn, double* Un,
                                 double* Jn, int* acc, bool ordered, cudaEvent_t mid, cudaStream_t st);
int dispatch_linesearch(int sys, int B, const double* params_host, int N, const double* X, const double* U, const DdpConst& c,
                        const int* T, const double* kl, const double* Kl, const int* ok, double* Xn, double* Un, double* Jn,
                        int* acc, cudaStream_t st);
int dispatch_bruteforce(int n, int m, int B, int N, int T_max, const double* A, const double* Bm, const double* X, const double* U,
                        long ustride, const DdpConst& c, double lm, double* J_out, int* status, cudaStream_t st);
int dispatch_cost(int n, int m, int B, int N, const double* X, const double* U, const DdpConst& c, const int* T, double* J,
                  cudaStream_t st);
int launch_init_state(int B, double lm_init, double* lm, int* done, int* n_hist, int* status_out, cudaStream_t st);
int launch_tile_u(int B, int N, int m, const double* u_ref, double* U, cudaStream_t st);
int launch_after_select(int B, const int* sel_status, int* done, int* status_out, cudaStream_t st);
int launch_warm_update(int B, int cap, const int* T_sel, const int* ok, const int* acc, const double* Jn, const int* bw_err,
                       int* done, int* T_bar, double* J_hist, int* T_hist, int* n_hist, int* copy, int* status_out,
                       cudaStream_t st);
int launch_ddp_update(int B, int cap, const int* T_sel, const int* ok, const int* acc, const double* Jn, const int* bw_err,
                      int* done, int* T_bar, double* lm, double* J_hist, int* T_hist, int* n_hist, int* copy,
                      int* status_out, int* n_active, cudaStream_t st);
int launch_copy_accepted(int B, size_t per_x, size_t per_u, const int* copy, const double* Xn, const double* Un, double* X,
                         double* U, cudaStream_t st);
int launch_finalize(int B, int cap, const int* n_hist, const int* T_hist, const int* T_bar, int* T_star, cudaStream_t st);
extern int g_backward_variant;
extern int g_linesearch_variant;

// ---- hop_util.cu
int launch_chol(int B, int d, int c, const double* A, const double* Bm, double* X, double jitter, int max_tries, int* status,
                cudaStream_t st);
int launch_affine_residuals(int B, int sys, const double* params_host, int N, const double* X, const double* U, long ustride,
                            double* a, cudaStream_t st);
int launch_build_augmented(int B, int N, int n, int m, const double* A, const double* Bm, const double* a, const double* X,
                           const double* U, long ustride, const double* xg, const double* w, const double* u_ref,
                           const double* Q, unsigned wrap_mask, double q_reg, double rho_reg, double* A_aug, double* B_aug,
                           double* Q_aug, cudaStream_t st);
int launch_build_terminal(int B, int N, int n, const double* X, const double* xg, const double* Qf, unsigned wrap_mask,
                          double rho_reg, double* QT, cudaStream_t st);
int launch_scan_consts(int B, int d, int m, const double* R_inv1, double* R_inv, double* z0, cudaStream_t st);

}  // namespace hop
