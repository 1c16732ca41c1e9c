// hop_select.cu -- __global__ wrappers + launchers of the horizon-selection kernels.
//
// Grid: one G-lane group per problem, 32/G problems per warp, WARPS warps per CTA; every warp is
// independent (warp-synchronous code, no CTA barrier inside the sweep), so the hardware scheduler
// load-balances warps across the 148 SMs.  Dynamic shared memory = per-group slab (Geo::SLAB
// doubles) [+ the CTA-wide case constants for the fused form].
#include <cstdint>

#include "hop_common.cuh"
#include "hop_select_body.cuh"
#include "hop_select_mma_body.cuh"
#include "hop_select_pipe_body.cuh"
#include "hop_select_scan_body.cuh"
#include "hop_select_gpipe_body.cuh"
#include "../../include/hop_b200.h"

namespace hop {

constexpr int kWarps = 2;   // warps per CTA (64 threads): small CTAs pack the register file tightly

template <int D, int M, int G>
__global__ void __launch_bounds__(kWarps * 32) k_select_generic(const SelectArgs p) {
    extern __shared__ __align__(16) double smem[];
    constexpr int GPW = 32 / G;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = warp * GPW + lane / G;
    const int b = blockIdx.x * (kWarps * GPW) + slot;
    select_generic_body<D, M, G>(p, b, smem + (size_t)slot * Geo<D, M, G>::SLAB);
}

template <int D, int M, int G>
__global__ void __launch_bounds__(kWarps * 32) k_select_fused(const FusedArgs p) {
    extern __shared__ __align__(16) double smem[];
    constexpr int GPW = 32 / G;
    double* cst = smem + (size_t)(kWarps * GPW) * Geo<D, M, G>::SLAB;
    fused_const_fill<D, M>(p, cst, threadIdx.x, blockDim.x);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = warp * GPW + lane / G;
    const int b = blockIdx.x * (kWarps * GPW) + slot;
    select_fused_body<D, M, G>(p, b, smem + (size_t)slot * Geo<D, M, G>::SLAB, cst);
}

template <int D, int M, int G>
static int launch_generic(const SelectArgs& p, cudaStream_t st) {
    constexpr int GPW = 32 / G;
    const size_t smem = sizeof(double) * (size_t)(kWarps * GPW) * Geo<D, M, G>::SLAB;
    cudaError_t e = cudaFuncSetAttribute(k_select_generic<D, M, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_generic)");
    const int per_cta = kWarps * GPW;
    const int grid = (p.B + per_cta - 1) / per_cta;
    k_select_generic<D, M, G><<<grid, kWarps * 32, smem, st>>>(p);
    return check_launch("k_select_generic");
}

template <int D, int M, int G>
static int launch_fused(const FusedArgs& p, cudaStream_t st) {
    constexpr int GPW = 32 / G;
    const size_t smem = sizeof(double) * ((size_t)(kWarps * GPW) * Geo<D, M, G>::SLAB + FusedConst<D, M>::SIZE);
    cudaError_t e = cudaFuncSetAttribute(k_select_fused<D, M, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_fused)");
    const int per_cta = kWarps * GPW;
    const int grid = (p.B + per_cta - 1) / per_cta;
    k_select_fused<D, M, G><<<grid, kWarps * 32, smem, st>>>(p);
    return check_launch("k_select_fused");
}

// ---- one problem per warp, DMMA register fragments (d in 9..16) -----------------------------------
constexpr int kMmaWarps = 4;   // warps (= problems) per CTA

// sequential FAST body out of line: the cold path of the pipelined kernel (jitter ladder, LU, status word)
template <int D, int M>
__device__ __noinline__ void select_fused_seq_cold(const FusedArgs& p, int b, double* scratch, const double* cst) {
    mma::select_fused_body<D, M, 1>(p, b, scratch, cst);
}

// MODE 0: EXACT, 1: FAST sequential, 2: FAST software-pipelined (hop_select_pipe_body.cuh) with MODE 1 as its cold path,
// 3: as 2 with the pivot sweep as run-time loops over groups of four pivots (a quarter of the code),
// 4: as 3 with the pivot row / column exchange through shared memory instead of shuffles,
// 5: as 4 with two pivots per loop trip (compile-time buffer parity) and high-word zeroing of the pivot row
template <int D, int M, int MODE, int MINB>
__global__ void __launch_bounds__(kMmaWarps * 32, MINB) k_select_fused_mma(const FusedArgs p) {
    extern __shared__ __align__(16) double smem[];
    double* cst = smem + (size_t)kMmaWarps * mma::kWarpScratch;
    const int warp = threadIdx.x >> 5;
    fused_const_fill<D, M>(p, cst, threadIdx.x, blockDim.x);
    __syncthreads();
    if (MODE >= 1) {   // K = (Qs + eps I)^-1, K' = (P + eps I)^-1 once per CTA
        if (warp == 0) mma::fast_const_fill_warp<D, M>(p, cst, smem);
        __syncthreads();
    }
    if (MODE >= 2) {
        mma::pipe_const_fill<D, M>(cst, threadIdx.x, blockDim.x);
        __syncthreads();
    }
    const int b = blockIdx.x * kMmaWarps + warp;
    double* scratch = smem + (size_t)warp * mma::kWarpScratch;
    if (MODE >= 2) {
        if (b >= p.B || (p.skip && p.skip[b])) return;
        if (mma::select_fused_pipe_body<D, M, MODE == 5 ? 3 : MODE == 4 ? 2 : MODE == 3 ? 1 : 0>(p, b, scratch, cst)) return;
        select_fused_seq_cold<D, M>(p, b, scratch, cst);
    } else {
        mma::select_fused_body<D, M, MODE>(p, b, scratch, cst);
    }
}

// HOP_MODE_SCAN: one CTA (kScanWarps warps) per problem, chunked parallel scan over the horizon
template <int D, int M>
__global__ void __launch_bounds__(mma::kScanWarps * 32) k_select_generic_scan(const SelectArgs p) {
    extern __shared__ __align__(16) double smem[];
    const int warp = threadIdx.x >> 5, b = blockIdx.x;
    mma::scan_phase1<D, M>(p, b, warp, mma::kScanWarps, smem);
    __syncthreads();
    mma::scan_phase23<D, M>(p, b, warp, mma::kScanWarps, smem);
    __syncthreads();
    if (threadIdx.x == 0) mma::scan_finish(p, b, mma::kScanWarps, smem);
}
template <int D, int M>
static int launch_generic_scan(const SelectArgs& p, cudaStream_t st) {
    const size_t smem = sizeof(double) * (size_t)mma::ScanSmem::size(mma::kScanWarps);
    cudaError_t e = cudaFuncSetAttribute(k_select_generic_scan<D, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_generic_scan)");
    k_select_generic_scan<D, M><<<p.B, mma::kScanWarps * 32, smem, st>>>(p);
    return check_launch("k_select_generic_scan");
}

// LQR-boundary form, software-pipelined (hop_select_gpipe_body.cuh); the sequential body is its cold path
template <int D, int M>
__device__ __noinline__ void select_generic_seq_cold(const SelectArgs& p, int b, double* scratch) {
    mma::select_generic_body<D, M>(p, b, scratch);
}
template <int D, int M>
__global__ void __launch_bounds__(kMmaWarps * 32, 3) k_select_generic_pipe(const SelectArgs p) {
    extern __shared__ __align__(16) double smem[];
    const int warp = threadIdx.x >> 5;
    const int b = blockIdx.x * kMmaWarps + warp;
    if (b >= p.B) return;
    double* slab = smem + (size_t)warp * mma::GpipeSlab<D, M>::SIZE;
    if (mma::select_generic_pipe_body<D, M>(p, b, slab)) return;
    select_generic_seq_cold<D, M>(p, b, slab);
}
// ---- pre-inverted input blocks: E_k = chol_inv(Q_k), X_t = chol_inv(QT_t) for every (problem, step) in parallel --------
constexpr int kPreWarps = 4;
constexpr int PRE_MINB = 4;   // CTAs per SM the pre-pass is register-bounded for (2 -> 174 registers, 4 -> 128)
// four lanes per matrix, eight matrices per warp; matrix index = 2 (b T_max + k) + {0: Q_aug, 1: QT}
template <int D>
__global__ void __launch_bounds__(kPreWarps * 32, PRE_MINB) k_preinvert(const SelectArgs p, double* E, double* X, int* bad) {
    const size_t mat = ((size_t)blockIdx.x * kPreWarps * 32 + threadIdx.x) >> 2;
    const size_t total = 2 * (size_t)p.B * p.T_max;
    const bool live = mat < total;
    const size_t mm = live ? mat : total - 1;                                    // idle groups shadow the last matrix
    const size_t task = mm >> 1, b = task / p.T_max, k = task % p.T_max;
    const size_t off = (b * p.N + k) * D * D;
    mma::pre_invert_cols<D>(((mm & 1) ? p.QT : p.Q_aug) + off, p.jitter, ((mm & 1) ? X : E) + off, bad + b, live);
}
template <int D, int M>
__global__ void __launch_bounds__(kMmaWarps * 32, 3) k_select_generic_pipe_pre(const SelectArgs p) {
    extern __shared__ __align__(16) double smem[];
    const int warp = threadIdx.x >> 5;
    const int b = blockIdx.x * kMmaWarps + warp;
    if (b >= p.B) return;
    double* slab = smem + (size_t)warp * mma::GpipeSlab<D, M>::SIZE;
    if (mma::select_generic_pipe_body<D, M, true>(p, b, slab)) return;
    select_generic_seq_cold<D, M>(p, b, slab);
}

// workspace of the pre-pass (E, X: 2 N d^2 doubles per problem, + one flag): stream-ordered allocation on the CALLER'S stream
// (cudaMallocAsync / cudaFreeAsync), so concurrent calls on different streams or host threads never share scratch and nothing
// outlives the call; bounded by kPreArenaMax -- larger batches run as consecutive chunks on the same stream, which orders the
// re-use.  The device's default memory pool keeps freed blocks (release threshold raised once per device), so repeated calls
// do not go back to the driver.
namespace {
constexpr size_t kPreArenaMax = (size_t)8 << 30;
int pool_keep_cached() {
    static bool done[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return 0;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    (void)cudaGetLastError();
    done[dev] = true;
    return 0;
}
}  // namespace
int stream_alloc(void** ptr, size_t bytes, cudaStream_t st, const char* what) {
    pool_keep_cached();
    return report_cuda(cudaMallocAsync(ptr, bytes, st), what);
}
void stream_free(void* ptr, cudaStream_t st) {
    if (ptr) cudaFreeAsync(ptr, st);
}
// 1: always, 0: never (sweep B inside the sequential kernel), -1 [default]: for small batches only.  Measured on B200
// (S2, d = 13, N = 128): B = 8: 0.95 -> 0.76 ms (one sweep latency per step instead of two); B = 65 536: 63.3 -> 68.2 ms
// (sequential kernel 63.3 -> 46.5 ms, but the pre-pass moves 45 GB and costs 19.8 ms): it pays where latency matters.
int g_generic_pre = -1;
// 1: diagonal input blocks go through the Gauss-Jordan sweep like any other block (test hook); 0 [default]: element-wise
int g_generic_nodiag = 0;
constexpr int kGenericPreMaxBatch = 1024;

template <int D, int M>
static int launch_generic_pipe(const SelectArgs& p, cudaStream_t st) {
    const size_t smem = sizeof(double) * (size_t)kMmaWarps * mma::GpipeSlab<D, M>::SIZE;
    if (g_generic_pre == 0 || (g_generic_pre < 0 && p.B > kGenericPreMaxBatch)) {
        cudaError_t e = cudaFuncSetAttribute(k_select_generic_pipe<D, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_generic_pipe)");
        const int grid = (p.B + kMmaWarps - 1) / kMmaWarps;
        k_select_generic_pipe<D, M><<<grid, kMmaWarps * 32, smem, st>>>(p);
        return check_launch("k_select_generic_pipe");
    }
    cudaError_t e = cudaFuncSetAttribute(k_select_generic_pipe_pre<D, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_generic_pipe_pre)");
    const size_t per_problem = sizeof(double) * 2 * (size_t)p.N * D * D + sizeof(int);
    size_t chunk = kPreArenaMax / per_problem;
    if (chunk > (size_t)p.B) chunk = (size_t)p.B;
    if (chunk < 1) chunk = 1;
    const size_t s_mat = ((sizeof(double) * chunk * p.N * D * D + 255) / 256) * 256;
    const size_t need = 2 * s_mat + sizeof(int) * chunk;
    void* arena = nullptr;
    if (int rc = stream_alloc(&arena, need, st, "cudaMallocAsync(pre-inversion workspace)")) return rc;
    double* E = (double*)arena;
    double* X = (double*)((char*)arena + s_mat);
    int* bad = (int*)((char*)arena + 2 * s_mat);
    int rc_all = 0;
    const size_t rinv_inst = (size_t)(p.rinv_step_stride ? p.N : 1) * M * M;
    for (size_t b0 = 0; b0 < (size_t)p.B; b0 += chunk) {
        SelectArgs q = p;
        q.B = (int)(((size_t)p.B - b0) < chunk ? ((size_t)p.B - b0) : chunk);
        const size_t om = b0 * p.N * D * D;
        q.A_aug = p.A_aug + om; q.Q_aug = p.Q_aug + om; q.QT = p.QT + om;
        q.B_aug = p.B_aug + b0 * p.N * D * M;
        q.R_inv = p.R_inv + b0 * rinv_inst;
        q.z0 = p.z0 + b0 * D;
        q.w_explicit = p.w_explicit ? p.w_explicit + b0 : nullptr;
        q.J_out = p.J_out + b0 * p.T_max; q.T_out = p.T_out + b0; q.Jstar_out = p.Jstar_out + b0; q.status = p.status + b0;
        q.E_pre = E; q.X_pre = X; q.pre_bad = bad;
        if ((rc_all = report_cuda(cudaMemsetAsync(bad, 0, sizeof(int) * (size_t)q.B, st), "memset(pre_bad)"))) break;
        const size_t mats = 2 * (size_t)q.B * q.T_max;                           // 8 matrices per warp
        k_preinvert<D><<<(unsigned)((mats + 8 * kPreWarps - 1) / (8 * kPreWarps)), kPreWarps * 32, 0, st>>>(q, E, X, bad);
        if ((rc_all = check_launch("k_preinvert"))) break;
        k_select_generic_pipe_pre<D, M><<<(q.B + kMmaWarps - 1) / kMmaWarps, kMmaWarps * 32, smem, st>>>(q);
        if ((rc_all = check_launch("k_select_generic_pipe_pre"))) break;
    }
    stream_free(arena, st);
    return rc_all;
}

// MINB = CTAs per SM the register allocation is bounded for (2 -> 255 regs, 3 [the only one instantiated] -> 168, 4 -> 128).
template <int D, int M, int MODE>
static int launch_fused_mma(const FusedArgs& p, cudaStream_t st) {
    const size_t smem = sizeof(double) * ((size_t)kMmaWarps * mma::kWarpScratch + mma::PipeConst<D, M>::SIZE);
    const int grid = (p.B + kMmaWarps - 1) / kMmaWarps;
    k_select_fused_mma<D, M, MODE, 3><<<grid, kMmaWarps * 32, smem, st>>>(p);
    return check_launch("k_select_fused_mma");
}

int dispatch_select_generic(int d, int m, int mode, const SelectArgs& p, cudaStream_t st) {
    if (mode == HOP_MODE_EXACT || mode == HOP_MODE_FP32) return dispatch_select_ref_generic(d, m, mode == HOP_MODE_FP32, p, st);
    if (mode == HOP_MODE_SCAN) {
        if (d == 12 && m == 4) return launch_generic_scan<12, 4>(p, st);
        if (d == 13 && m == 4) return launch_generic_scan<13, 4>(p, st);
        set_last_error("hop_select_f64: HOP_MODE_SCAN is instantiated for (d, m) = (12,4) and (13,4) only");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    if (d <= 5) {
        const int rc = dispatch_select_generic_tpp(d, m, p, st);
        if (rc != HOP_E_UNSUPPORTED_DIMS) return rc;
    }
    if (d == 3 && m == 1) return launch_generic<3, 1, 4>(p, st);
    if (d == 4 && m == 2) return launch_generic<4, 2, 4>(p, st);
    if (d == 5 && m == 1) return launch_generic<5, 1, 8>(p, st);
    if (d == 12 && m == 4) return launch_generic_pipe<12, 4>(p, st);
    if (d == 13 && m == 4) return launch_generic_pipe<13, 4>(p, st);
    set_last_error("hop_select_f64: (d, m) not instantiated; supported: (3,1) (4,2) (5,1) (12,4) (13,4)");
    return HOP_E_UNSUPPORTED_DIMS;
}

// HOP_MODE_SCAN of the fused form: the scan kernel works at the LQR boundary, so materialise the augmented blocks
// (augmented.py:10-87) in a stream-ordered scratch allocation, then run the chunked parallel scan over the horizon.  Small
// batches only (that is where it pays).
static int select_fused_scan(int n, int m, const FusedArgs& p, cudaStream_t st) {
    if (!hop_select_supported_mode(n + 1, m, HOP_MODE_SCAN)) {
        set_last_error("hop_select_fused_f64: HOP_MODE_SCAN is instantiated for (n, m) = (11,4) and (12,4) only");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    const int B = p.B, N = p.N, d = n + 1;
    const size_t dd = (size_t)B * N * d * d, dm = (size_t)B * N * d * m;
    const size_t total = sizeof(double) * (3 * dd + dm + (size_t)B * m * m + (size_t)B * d + (size_t)m * m) + sizeof(int);
    void* ws = nullptr;
    if (int rc = stream_alloc(&ws, total, st, "cudaMallocAsync(scan workspace)")) return rc;
    double* A_aug = (double*)ws; double* Q_aug = A_aug + dd; double* QT = Q_aug + dd; double* B_aug = QT + dd;
    double* R_inv = B_aug + dm; double* z0 = R_inv + (size_t)B * m * m; double* R1 = z0 + (size_t)B * d;
    int* st1 = (int*)(R1 + m * m);
    int rc = launch_build_augmented(B, N, n, m, p.A, p.Bm, p.a_resid, p.X, p.U, p.u_stride, p.xg, p.w, p.u_ref, p.Q, p.wrap_mask,
                                    p.q_reg, p.rho_reg, A_aug, B_aug, Q_aug, st);
    if (!rc) rc = launch_build_terminal(B, N, n, p.X, p.xg, p.Qf, p.wrap_mask, p.rho_reg, QT, st);
    if (!rc) rc = launch_chol(1, m, 0, p.R, nullptr, R1, p.jitter, p.max_tries, st1, st);          // augmented.py:23
    if (!rc) rc = launch_scan_consts(B, d, m, R1, R_inv, z0, st);                                 // augmented.py:59
    if (!rc) {
        SelectArgs q{B, N, p.T_min, p.T_max, p.jitter, p.max_tries, A_aug, B_aug, Q_aug, R_inv, z0, QT, 0, nullptr,
                     p.J_out, p.T_out, p.Jstar_out, p.status, nullptr, nullptr, nullptr, g_generic_nodiag};
        rc = dispatch_select_generic(d, m, HOP_MODE_SCAN, q, st);
    }
    stream_free(ws, st);
    return rc;
}

int dispatch_select_fused(int n, int m, const FusedArgs& p, cudaStream_t st) {
    if (p.mode == HOP_MODE_SCAN) return select_fused_scan(n, m, p, st);
    if (p.mode == HOP_MODE_EXACT) return launch_ref_fused_list(n, m, p, nullptr, nullptr, st);
    if (p.mode == HOP_MODE_VERIFIED) return dispatch_select_verified(n, m, p, st);
    if (n <= 4) {
        const int rc = dispatch_select_fused_epl(n, m, p, st);
        if (rc != HOP_E_UNSUPPORTED_DIMS) return rc;
    }
    if (n == 2 && m == 1) return launch_fused<3, 1, 4>(p, st);
    if (n == 4 && m == 1) return launch_fused<5, 1, 8>(p, st);
    if (n == 12 && m == 4) {
        if (p.mode != HOP_MODE_FAST) return launch_fused_mma<13, 4, 0>(p, st);
        // (The sequential FAST sweep -- the pipelined kernel's out-of-line cold path -- and the earlier schedules of the pipelined
        // sweep are no longer instantiated as kernels of their own; tests/emul still runs them as cross-checks of the same math.)
        return launch_fused_mma<13, 4, 5>(p, st);
    }
    set_last_error("hop_select_fused_f64: (n, m) not instantiated; supported: (2,1) (4,1) (12,4)");
    return HOP_E_UNSUPPORTED_DIMS;
}

}  // namespace hop
