// hop_ddp.cu -- batched HOP-DDP iteration around the horizon selection (one thread per problem) and
// the per-instance solver state machine of solver.py:449-765 (method="propagator").
//
//   k_cost        solver.py:65-105    cost_timeopt_true
//   k_backward    solver.py:156-230   backward_pass_truncated
//   k_linesearch  solver.py:233-286   forward_linesearch_fixedT
//   k_after_select / k_ddp_update / k_copy_accepted   accept-reject, LM schedule, histories, stop rule
//                                                     (solver.py:522,553-555,590,735-748)
// Every kernel takes the per-instance `done` word and skips finished instances, so a batch whose
// members stop at different iterations needs no host-side control flow.
#include "hop_common.cuh"

#include "hop_ddp_core.cuh"
#include "hop_ddp_mma.cuh"
#include "../../include/hop_b200.h"

namespace hop {

// CostConst::diag for the whole CTA: the threads share the off-diagonal entries of Q, R, Qf (at most two loads each) and vote.
// EVERY thread of the CTA calls this before any early return.
template <int d>
__device__ __forceinline__ bool cta_is_diagonal(const double* M) {
    bool dg = true;
    for (int i = threadIdx.x; i < d * d; i += blockDim.x)
        if (i / d != i % d) dg = dg && (M[i] == 0.0);
    return __syncthreads_and(dg) != 0;
}
template <int n, int m>
__device__ __forceinline__ unsigned cta_diag_flags(const DdpConst& c) {
    return (cta_is_diagonal<n>(c.Q) ? 1u : 0u) | (cta_is_diagonal<m>(c.R) ? 2u : 0u) | (cta_is_diagonal<n>(c.Qf) ? 4u : 0u);
}
template <int n, int m>
__device__ __forceinline__ ddp::CostConst cost_const(const DdpConst& c, int b, unsigned diag) {
    ddp::CostConst cc;
    cc.diag = diag;
    cc.xg = c.xg + (size_t)b * n;
    cc.u_ref = c.u_ref; cc.Q = c.Q; cc.R = c.R; cc.Qf = c.Qf;
    cc.w = c.w[b];
    cc.wrap_mask = c.wrap_mask;
    return cc;
}

// per-instance horizon of the stand-alone entry points: a caller's T_star[b] > N is clamped to N (the trajectories hold N
// steps); T_star[b] <= 0 is handled as the reference does (cost = inf, solver.py:71; backward pass: ok = False)
__device__ __forceinline__ int horizon_of(const int* T, int b, int N) {
    const int t = T[b];
    return t > N ? N : t;
}

template <int n, int m>
__global__ void k_cost(int B, int N, const double* X, const double* U, DdpConst c, const int* T, double* J) {
    const unsigned diag = cta_diag_flags<n, m>(c);                              // (all threads, before any return)
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const ddp::CostConst cc = cost_const<n, m>(c, b, diag);
    J[b] = ddp::cost_timeopt_true<n, m>(X + (size_t)b * (N + 1) * n, U + (size_t)b * N * m, cc, horizon_of(T, b, N));
}

template <int n, int m>
__global__ void k_backward(int B, int N, const double* A, const double* Bm, const double* X, const double* U, DdpConst c,
                           const int* T, const double* lm, const int* done, double* k_out, double* K_out, int* ok,
                           int* err) {
    const unsigned diag = cta_diag_flags<n, m>(c);                              // (all threads, before any return)
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (done && done[b]) { ok[b] = 0; return; }
    const ddp::CostConst cc = cost_const<n, m>(c, b, diag);
    int okb = 0;
    const int rc = ddp::backward_pass<n, m>(A + (size_t)b * N * n * n, Bm + (size_t)b * N * n * m, X + (size_t)b * (N + 1) * n,
                                            U + (size_t)b * N * m, cc, horizon_of(T, b, N), lm[b], k_out + (size_t)b * N * m,
                                            K_out + (size_t)b * N * m * n, &okb);
    ok[b] = (rc == 0) ? okb : 0;
    if (err) err[b] = rc;
}

// backward-pass kernel: 0 [default] = the tensor-pipe kernel (backward_pass_mma) for n > 8 unless the caller asks for the
// reference's summation order (HOP_MODE_EXACT solves, the stand-alone entry point), else the warp kernel; 1 = one thread per
// problem; 2 = one warp per problem, ordered sums (1 and 2: identical bits); 3 = tensor-pipe kernel wherever it is instantiated.
// Set by hop_test_set_backward_variant.
int g_backward_variant = 0;

// one warp per problem (backward_pass_warp), kBwWarps problems per CTA
constexpr int kBwWarps = 4;
// small systems: 7 CTAs per SM (<= 72 registers), so that 4 096 instances -- 28 warps per SM -- are one wave; quadrotor: 4 CTAs
// (<= 128 registers; 2 048 instances -- the per-GPU load of configuration 4 on eight GPUs -- are 14 warps per SM)
template <int n, int m>
__global__ void __launch_bounds__(kBwWarps * 32, (n <= 4) ? 7 : 4) k_backward_warp(int B, int N, const double* A, const double* Bm, const double* X,
                                                                 const double* U, DdpConst c, const int* T, const double* lm,
                                                                 const int* done, double* k_out, double* K_out, int* ok, int* err) {
    const unsigned diag = cta_diag_flags<n, m>(c);                              // (all threads, before any return)
    __shared__ __align__(16) double smem[kBwWarps * ddp::BwSmem<n, m>::SIZE];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * kBwWarps + warp;
    if (b >= B) return;
    if (done && done[b]) { if (lane == 0) ok[b] = 0; return; }
    const ddp::CostConst cc = cost_const<n, m>(c, b, diag);
    int okb = 0;
    const int rc = ddp::backward_pass_warp<n, m>(A + (size_t)b * N * n * n, Bm + (size_t)b * N * n * m, X + (size_t)b * (N + 1) * n,
                                                 U + (size_t)b * N * m, cc, horizon_of(T, b, N), lm[b], k_out + (size_t)b * N * m,
                                                 K_out + (size_t)b * N * m * n, &okb, smem + (size_t)warp * ddp::BwSmem<n, m>::SIZE, lane);
    if (lane == 0) {
        ok[b] = (rc == 0) ? okb : 0;
        if (err) err[b] = rc;
    }
}

// same grid, matrix products on the FP64 tensor pipe (hop_ddp_mma.cuh)
template <int n, int m>
__global__ void __launch_bounds__(kBwWarps * 32) k_backward_mma(int B, int N, const double* A, const double* Bm, const double* X,
                                                                const double* U, DdpConst c, const int* T, const double* lm,
                                                                const int* done, double* k_out, double* K_out, int* ok, int* err) {
    const unsigned diag = cta_diag_flags<n, m>(c);                              // (all threads, before any return)
    __shared__ __align__(16) double smem[kBwWarps * ddp::BwSmem<n, m>::SIZE];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * kBwWarps + warp;
    if (b >= B) return;
    if (done && done[b]) { if (lane == 0) ok[b] = 0; return; }
    const ddp::CostConst cc = cost_const<n, m>(c, b, diag);
    int okb = 0;
    const int rc = ddp::backward_pass_mma<n, m>(A + (size_t)b * N * n * n, Bm + (size_t)b * N * n * m, X + (size_t)b * (N + 1) * n,
                                                U + (size_t)b * N * m, cc, horizon_of(T, b, N), lm[b], k_out + (size_t)b * N * m,
                                                K_out + (size_t)b * N * m * n, &okb, smem + (size_t)warp * ddp::BwSmem<n, m>::SIZE, lane);
    if (lane == 0) {
        ok[b] = (rc == 0) ? okb : 0;
        if (err) err[b] = rc;
    }
}

// solver.py:293-358: one warp per (problem, T); J_out [B][T_max], status [B] (DDP_* code of the first failing horizon)
template <int n, int m>
__global__ void __launch_bounds__(kBwWarps * 32) k_bruteforce(int B, int N, int T_max, const double* A, const double* Bm,
                                                              const double* X, const double* U, long ustride, DdpConst c,
                                                              double lm, double* J_out, int* status) {
    const unsigned diag = cta_diag_flags<n, m>(c);                              // (all threads, before any return)
    __shared__ __align__(16) double smem[kBwWarps * ddp::BwSmem<n, m>::SIZE];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t id = (size_t)blockIdx.x * kBwWarps + warp;
    if (id >= (size_t)B * T_max) return;
    const int b = (int)(id / T_max), T = T_max - (int)(id % T_max);          // long horizons first
    const ddp::CostConst cc = cost_const<n, m>(c, b, diag);
    double V0 = 0.0;
    const int rc = ddp::bruteforce_one_T_warp<n, m>(A + (size_t)b * N * n * n, Bm + (size_t)b * N * n * m,
                                                    X + (size_t)b * (N + 1) * n, U + (size_t)b * ustride, cc, T, lm, &V0,
                                                    smem + (size_t)warp * ddp::BwSmem<n, m>::SIZE, lane);
    if (lane == 0) {
        J_out[(size_t)b * T_max + (T - 1)] = rc ? nan("") : V0;
        if (rc) atomicMax(status + b, rc);
    }
}

int dispatch_bruteforce(int n, int m, int B, int N, int T_max, const double* A, const double* Bm, const double* X, const double* U,
                        long ustride, const DdpConst& c, double lm, double* J_out, int* status, cudaStream_t st) {
    if (int rc = report_cuda(cudaMemsetAsync(status, 0, sizeof(int) * (size_t)B, st), "memset(status)")) return rc;
    const size_t warps = (size_t)B * T_max;
    const unsigned grid = (unsigned)((warps + kBwWarps - 1) / kBwWarps);
    if (n == 2 && m == 1) k_bruteforce<2, 1><<<grid, kBwWarps * 32, 0, st>>>(B, N, T_max, A, Bm, X, U, ustride, c, lm, J_out, status);
    else if (n == 4 && m == 1) k_bruteforce<4, 1><<<grid, kBwWarps * 32, 0, st>>>(B, N, T_max, A, Bm, X, U, ustride, c, lm, J_out, status);
    else if (n == 12 && m == 4) k_bruteforce<12, 4><<<grid, kBwWarps * 32, 0, st>>>(B, N, T_max, A, Bm, X, U, ustride, c, lm, J_out, status);
    else { set_last_error("hop_bruteforce_jt_f64: (n, m) not instantiated; supported: (2,1) (4,1) (12,4)"); return HOP_E_UNSUPPORTED_DIMS; }
    return check_launch("k_bruteforce");
}

template <int SYS>
__global__ void k_linesearch(int B, DynParams prm, int N, const double* X, const double* U, DdpConst c, const int* T,
                             const double* k_list, const double* K_list, const int* ok, const int* done, double* Xn,
                             double* Un, double* Jn, int* acc) {
    constexpr int n = SysDims<SYS>::n, m = SysDims<SYS>::m;
    const unsigned diag = cta_diag_flags<n, m>(c);                              // (all threads, before any return)
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    acc[b] = 0;
    if ((done && done[b]) || (ok && !ok[b])) return;
    const ddp::CostConst cc = cost_const<n, m>(c, b, diag);
    double J = 0.0;
    int a = 0;
    ddp::forward_linesearch<SYS>(prm.p, N, X + (size_t)b * (N + 1) * n, U + (size_t)b * N * m, cc, horizon_of(T, b, N),
                                 k_list + (size_t)b * N * m, K_list + (size_t)b * N * m * n, Xn + (size_t)b * (N + 1) * n,
                                 Un + (size_t)b * N * m, &J, &a);
    Jn[b] = J;
    acc[b] = a;
}

// Line search with the five step sizes of solver.py:240 side by side.  A CTA of six warps serves 32 instances
// (lane = instance, warp = role, so no warp diverges): warps 0..4 roll out alpha = (1, .5, .25, .1, .05) and evaluate
// the cost on the fly, warp 5 evaluates J_old at the new T* (solver.py:253).  The reference accepts the FIRST alpha
// with J_new < J_old; the CTA takes the same decision from six values per instance in shared memory.  Warp 0 stores its
// candidate while rolling (alpha = 1 is accepted most of the time); another winner rolls once more with stores.  Every
// candidate is computed by the same instruction sequence as in k_linesearch, so X_new, U_new, J and `accepted` are
// bit-identical -- in one or two roll-out latencies instead of up to five plus a cost pass each (the batch sizes of the
// HOP-DDP configurations leave the machine empty, so the extra threads are free).
constexpr int kLsRoles = 6;
template <int SYS>
__global__ void __launch_bounds__(kLsRoles * 32) k_linesearch_par(int B, DynParams prm, int N, const double* X, const double* U,
                                                                    DdpConst c, const int* T, const double* k_list,
                                                                    const double* K_list, const int* ok, const int* done,
                                                                    double* Xn, double* Un, double* Jn, int* acc) {
    constexpr int n = SysDims<SYS>::n, m = SysDims<SYS>::m;
    const unsigned diag = cta_diag_flags<n, m>(c);                              // (all threads, before any return)
    __shared__ double sJ[kLsRoles][32];
    __shared__ int sOk[kLsRoles][32];
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const int b_raw = blockIdx.x * 32 + lane;
    const bool valid = b_raw < B;
    const int b = valid ? b_raw : B - 1;
    const bool active = valid && !((done && done[b]) || (ok && !ok[b]));
    if (valid && role == 0) acc[b] = 0;
    const ddp::CostConst cc = cost_const<n, m>(c, b, diag);
    const double* Xb = X + (size_t)b * (N + 1) * n;
    const double* Ub = U + (size_t)b * N * m;
    const double* kb = k_list + (size_t)b * N * m;
    const double* Kb = K_list + (size_t)b * N * m * n;
    double* Xnb = Xn + (size_t)b * (N + 1) * n;
    double* Unb = Un + (size_t)b * N * m;
    const int Tb = horizon_of(T, b, N);
    const double alpha = role == 0 ? 1.0 : role == 1 ? 0.5 : role == 2 ? 0.25 : role == 3 ? 0.1 : 0.05;
    double J = HUGE_VAL;
    bool cand_ok = false;
    if (active) {
        if (role == 0) cand_ok = ddp::linesearch_candidate<SYS, true>(prm.p, N, Xb, Ub, cc, Tb, kb, Kb, alpha, Xnb, Unb, &J);
        else if (role < 5) cand_ok = ddp::linesearch_candidate<SYS, false>(prm.p, N, Xb, Ub, cc, Tb, kb, Kb, alpha, nullptr, nullptr, &J);
        else J = ddp::cost_timeopt_true<n, m>(Xb, Ub, cc, Tb);
    }
    sJ[role][lane] = J;
    sOk[role][lane] = cand_ok ? 1 : 0;
    __syncthreads();
    if (!active) return;
    const double J_old = sJ[5][lane];
    int winner = -1;
#pragma unroll
    for (int r = 4; r >= 0; --r)
        if (sOk[r][lane] && sJ[r][lane] < J_old) winner = r;
    if (winner > 0 && role == winner)
        ddp::linesearch_candidate<SYS, true>(prm.p, N, Xb, Ub, cc, Tb, kb, Kb, alpha, Xnb, Unb, &J);
    if (winner >= 0) {
        if (role == winner) { Jn[b] = J; acc[b] = 1; }
        return;
    }
    for (size_t i = role; i < (size_t)(N + 1) * n; i += kLsRoles) Xnb[i] = Xb[i];
    for (size_t i = role; i < (size_t)N * m; i += kLsRoles) Unb[i] = Ub[i];
    if (role == 0) { Jn[b] = J_old; acc[b] = 0; }
}
// line-search kernel: 0 step sizes side by side (default), 1 one thread per problem trying them in turn (test hook;
// identical bits)
int g_linesearch_variant = 0;
template <int SYS>
static int launch_linesearch(int B, const DynParams& prm, int N, const double* X, const double* U, const DdpConst& c, const int* T,
                             const double* kl, const double* Kl, const int* ok, const int* done, double* Xn, double* Un,
                             double* Jn, int* acc, cudaStream_t st) {
    const int threads = 64;
    // Six threads per instance only pay while they fit next to each other: measured on B200, forward phase of a 12-iteration
    // solve: Segway B = 25 7.6 -> 2.5 ms, Cartpole B = 4096 67.5 -> 16.1 ms, Quadrotor B = 16384 22.1 -> 28.3 ms (130
    // registers: the machine holds ~75k such threads, 16384 x 6 no longer fit in one wave).
    constexpr long par_max = 8192;
    if (g_linesearch_variant != 0 || B > par_max) {
        k_linesearch<SYS><<<(B + threads - 1) / threads, threads, 0, st>>>(B, prm, N, X, U, c, T, kl, Kl, ok, done, Xn, Un, Jn, acc);
        return check_launch("k_linesearch");
    }
    k_linesearch_par<SYS><<<(B + 31) / 32, kLsRoles * 32, 0, st>>>(B, prm, N, X, U, c, T, kl, Kl, ok, done, Xn, Un, Jn, acc);
    return check_launch("k_linesearch_par");
}

// After a selection: an instance whose selection raised in the reference (status low byte != 0) stops
// here ("crash", run_suite.py:137-157); otherwise T_sel is the horizon to optimise at.
__global__ void k_after_select(int B, const int* sel_status, int* done, int* status_out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B || done[b]) return;
    const int st = sel_status[b];
    status_out[b] |= (st & ~0xff);
    if (st & 0xff) { done[b] = 2; status_out[b] |= (st & 0xff); }
}

// Warm start bookkeeping (solver.py:546-555): X,U <- line-search result when the backward pass was ok;
// (J0, T_bar) appended when J0 is finite.  `copy` marks instances whose candidate must be copied in.
__global__ void k_warm_update(int B, int cap, const int* T_sel, const int* ok, const int* acc, const double* Jn,
                              const int* bw_err, int* done, int* T_bar, double* J_hist, int* T_hist, int* n_hist,
                              int* copy, int* status_out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    copy[b] = 0;
    if (done[b]) return;
    T_bar[b] = T_sel[b];
    if (bw_err[b]) { done[b] = 2; status_out[b] |= bw_err[b]; return; }     // chol_solve raised (utils.py:120)
    if (!ok[b]) return;
    copy[b] = acc[b];
    if (isfinite(Jn[b])) {
        J_hist[(size_t)b * cap + n_hist[b]] = Jn[b];
        T_hist[(size_t)b * cap + n_hist[b]] = T_sel[b];
        n_hist[b] += 1;
    }
}

// Outer-loop bookkeeping (solver.py:735-748).
__global__ void k_ddp_update(int B, int cap, const int* T_sel, const int* ok, const int* acc, const double* Jn,
                             const int* bw_err, int* done, int* T_bar, double* lm, double* J_hist, int* T_hist,
                             int* n_hist, int* copy, int* status_out, int* n_active) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    copy[b] = 0;
    if (done[b]) return;
    if (bw_err[b]) { done[b] = 2; status_out[b] |= bw_err[b]; return; }
    const bool accept = ok[b] && acc[b] && isfinite(Jn[b]);
    if (accept) {
        copy[b] = 1;
        T_bar[b] = T_sel[b];
        J_hist[(size_t)b * cap + n_hist[b]] = Jn[b];
        T_hist[(size_t)b * cap + n_hist[b]] = T_sel[b];
        n_hist[b] += 1;
        lm[b] = fmax(lm[b] / 10.0, 1e-12);
    } else {
        lm[b] = lm[b] * 10.0;
    }
    const int nh = n_hist[b];
    if (nh >= 2) {
        const double j1 = J_hist[(size_t)b * cap + nh - 1], j2 = J_hist[(size_t)b * cap + nh - 2];
        const double rel = fabs(j1 - j2) / (fabs(j2) + 1e-12);
        if (rel < 1e-4 && nh >= 3) {
            const int* th = T_hist + (size_t)b * cap;
            if (th[nh - 1] == th[nh - 2] && th[nh - 2] == th[nh - 3]) done[b] = 1;
        }
    }
    if (!done[b]) atomicAdd(n_active, 1);
}

__global__ void k_copy_accepted(int B, size_t per_x, size_t per_u, const int* copy, const double* Xn, const double* Un,
                                double* X, double* U) {
    const size_t per = per_x + per_u;
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)B * per) return;
    const size_t b = gid / per, r = gid % per;
    if (!copy[b]) return;
    if (r < per_x) X[b * per_x + r] = Xn[b * per_x + r];
    else U[b * per_u + (r - per_x)] = Un[b * per_u + (r - per_x)];
}

__global__ void k_finalize(int B, int cap, const int* n_hist, const int* T_hist, const int* T_bar, int* T_star) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int nh = n_hist[b];
    T_star[b] = nh ? T_hist[(size_t)b * cap + nh - 1] : T_bar[b];          // solver.py:763
}

__global__ void k_init_state(int B, double lm_init, double* lm, int* done, int* n_hist, int* status_out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    lm[b] = lm_init; done[b] = 0; n_hist[b] = 0; status_out[b] = 0;
}

__global__ void k_tile_u(int B, int N, int m, const double* u_ref, double* U) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)B * N * m) return;
    U[gid] = u_ref[gid % m];
}

template <int SYS>
static int ddp_backward_linesearch(int B, const DynParams& prm, int N, const double* A, const double* Bm, const double* X,
                                   const double* U, const DdpConst& c, const int* T, const double* lm, const int* done,
                                   double* kl, double* Kl, int* ok, int* bw_err, double* Xn, double* Un, double* Jn, int* acc,
                                   bool ordered, cudaEvent_t mid, cudaStream_t st) {
    constexpr int n = SysDims<SYS>::n, m = SysDims<SYS>::m;
    const int threads = 64;
    const int v = g_backward_variant;
    bool use_mma = false;
    // measured on B200 (quadrotor, 12 iterations): backward phase 42.9 -> 37.6 ms at 16 384 instances, 7.06 -> 7.60 ms at 2 048
    // (few instances: the step is bound by the latency of the m x m Cholesky ladder and the vector recursions, which both
    // kernels share, and the fragment loads lengthen that chain) => the tensor-pipe kernel from 4 096 instances on
    if constexpr (n > 8) use_mma = (v == 3) || (v == 0 && !ordered && B >= 4096);
    if (v == 1) k_backward<n, m><<<grid1(B, threads), threads, 0, st>>>(B, N, A, Bm, X, U, c, T, lm, done, kl, Kl, ok, bw_err);
    else if (use_mma) {
        if constexpr (n > 8) k_backward_mma<n, m><<<grid1(B, kBwWarps), kBwWarps * 32, 0, st>>>(B, N, A, Bm, X, U, c, T, lm, done, kl, Kl, ok, bw_err);
    } else k_backward_warp<n, m><<<grid1(B, kBwWarps), kBwWarps * 32, 0, st>>>(B, N, A, Bm, X, U, c, T, lm, done, kl, Kl, ok, bw_err);
    if (int rc = check_launch("k_backward")) return rc;
    if (mid) cudaEventRecord(mid, st);
    return launch_linesearch<SYS>(B, prm, N, X, U, c, T, kl, Kl, ok, done, Xn, Un, Jn, acc, st);
}

int dispatch_backward_linesearch(int sys, int B, const double* params_host, int N, const double* A, const double* Bm,
                                 const double* X, const double* U, const DdpConst& c, const int* T, const double* lm,
                                 const int* done, double* kl, double* Kl, int* ok, int* bw_err, double* Xn, double* Un,
                                 double* Jn, int* acc, bool ordered, cudaEvent_t mid, cudaStream_t st) {
    const DynParams prm = dyn_params(params_host);
    return with_system(sys, "hop_backward_linesearch_f64", [&](auto s) {
        return ddp_backward_linesearch<decltype(s)::value>(B, prm, N, A, Bm, X, U, c, T, lm, done, kl, Kl, ok, bw_err, Xn, Un, Jn,
                                                           acc, ordered, mid, st);
    });
}

int dispatch_linesearch(int sys, int B, const double* params_host, int N, const double* X, const double* U, const DdpConst& c,
                        const int* T, const double* kl, const double* Kl, const int* ok, double* Xn, double* Un, double* Jn,
                        int* acc, cudaStream_t st) {
    const DynParams prm = dyn_params(params_host);
    return with_system(sys, "hop_linesearch_f64", [&](auto s) {
        return launch_linesearch<decltype(s)::value>(B, prm, N, X, U, c, T, kl, Kl, ok, nullptr, Xn, Un, Jn, acc, st);
    });
}

int dispatch_cost(int n, int m, int B, int N, const double* X, const double* U, const DdpConst& c, const int* T, double* J,
                  cudaStream_t st) {
    const int threads = 128;
    if (n == 2 && m == 1) k_cost<2, 1><<<grid1(B, threads), threads, 0, st>>>(B, N, X, U, c, T, J);
    else if (n == 4 && m == 1) k_cost<4, 1><<<grid1(B, threads), threads, 0, st>>>(B, N, X, U, c, T, J);
    else if (n == 12 && m == 4) k_cost<12, 4><<<grid1(B, threads), threads, 0, st>>>(B, N, X, U, c, T, J);
    else { set_last_error("hop_cost_f64: (n, m) not instantiated"); return HOP_E_UNSUPPORTED_DIMS; }
    return check_launch("k_cost");
}

// thin launch helpers used by the solver loop in hop_cabi.cu
int launch_init_state(int B, double lm_init, double* lm, int* done, int* n_hist, int* status_out, cudaStream_t st) {
    k_init_state<<<grid1(B, 128), 128, 0, st>>>(B, lm_init, lm, done, n_hist, status_out);
    return check_launch("k_init_state");
}
int launch_tile_u(int B, int N, int m, const double* u_ref, double* U, cudaStream_t st) {
    k_tile_u<<<grid1((size_t)B * N * m, 256), 256, 0, st>>>(B, N, m, u_ref, U);
    return check_launch("k_tile_u");
}
int launch_after_select(int B, const int* sel_status, int* done, int* status_out, cudaStream_t st) {
    k_after_select<<<grid1(B, 128), 128, 0, st>>>(B, sel_status, done, status_out);
    return check_launch("k_after_select");
}
int launch_warm_update(int B, int cap, const int* T_sel, const int* ok, const int* acc, const double* Jn, const int* bw_err,
                       int* done, int* T_bar, double* J_hist, int* T_hist, int* n_hist, int* copy, int* status_out,
                       cudaStream_t st) {
    k_warm_update<<<grid1(B, 128), 128, 0, st>>>(B, cap, T_sel, ok, acc, Jn, bw_err, done, T_bar, J_hist, T_hist, n_hist, copy,
                                                 status_out);
    return check_launch("k_warm_update");
}
int launch_ddp_update(int B, int cap, const int* T_sel, const int* ok, const int* acc, const double* Jn, const int* bw_err,
                      int* done, int* T_bar, double* lm, double* J_hist, int* T_hist, int* n_hist, int* copy,
                      int* status_out, int* n_active, cudaStream_t st) {
    k_ddp_update<<<grid1(B, 128), 128, 0, st>>>(B, cap, T_sel, ok, acc, Jn, bw_err, done, T_bar, lm, J_hist, T_hist, n_hist,
                                                copy, status_out, n_active);
    return check_launch("k_ddp_update");
}
int launch_copy_accepted(int B, size_t per_x, size_t per_u, const int* copy, const double* Xn, const double* Un, double* X,
                         double* U, cudaStream_t st) {
    k_copy_accepted<<<grid1((size_t)B * (per_x + per_u), 256), 256, 0, st>>>(B, per_x, per_u, copy, Xn, Un, X, U);
    return check_launch("k_copy_accepted");
}
int launch_finalize(int B, int cap, const int* n_hist, const int* T_hist, const int* T_bar, int* T_star, cudaStream_t st) {
    k_finalize<<<grid1(B, 128), 128, 0, st>>>(B, cap, n_hist, T_hist, T_bar, T_star);
    return check_launch("k_finalize");
}

}  // namespace hop
