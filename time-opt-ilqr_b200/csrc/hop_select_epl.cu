// hop_select_epl.cu -- __global__ wrapper + launcher of the element-per-lane fused selection kernel for small systems
// (hop_select_epl_body.cuh).  Grid: one warp per problem, kEplWarps warps per CTA (small CTAs spread a small batch
// over many SMs: these launches are latency bound).  Dynamic shared memory = per-warp LU scratch + the CTA constants.
#include "hop_common.cuh"
#include "hop_select_epl_body.cuh"
#include "../../include/hop_b200.h"

namespace hop {

constexpr int kEplWarps = 2;
template <int D>
struct EplScratch { static constexpr int SIZE = 2 * D * ((D + 1) & ~1); };   // LU fallback: two D x DP buffers per warp

template <int D, int M>
__global__ void __launch_bounds__(kEplWarps * 32) k_select_fused_epl(const FusedArgs p) {
    extern __shared__ __align__(16) double smem[];
    double* cst = smem + kEplWarps * EplScratch<D>::SIZE;
    fused_const_fill<D, M>(p, cst, threadIdx.x, blockDim.x);
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const int b = blockIdx.x * kEplWarps + warp;
    if (b >= p.B || (p.skip && p.skip[b])) return;
    epl::select_fused_epl_body<D, M>(p, b, smem + warp * EplScratch<D>::SIZE, cst);
}

template <int D, int M>
static int launch_fused_epl(const FusedArgs& p, cudaStream_t st) {
    const size_t smem = sizeof(double) * ((size_t)kEplWarps * EplScratch<D>::SIZE + FusedConst<D, M>::SIZE);
    k_select_fused_epl<D, M><<<(p.B + kEplWarps - 1) / kEplWarps, kEplWarps * 32, smem, st>>>(p);
    return check_launch("k_select_fused_epl");
}

// ---- the same sweep as a warp-specialised pipeline: one problem per CTA (3 stage warps, 1 prefix warp, 3 query warps)
template <int D, int M>
__global__ void __launch_bounds__(epl::kWspWarps * 32) k_select_fused_wsp(const FusedArgs p) {
    extern __shared__ __align__(16) double smem[];
    using WS = epl::WspSmem<D>;
    double* cst = smem + WS::SIZE;
    fused_const_fill<D, M>(p, cst, threadIdx.x, blockDim.x);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int* status_words = reinterpret_cast<int*>(smem + WS::RESULT + epl::kWspQueryWarps * 4);
    if (threadIdx.x < epl::kWspWarps) status_words[threadIdx.x] = 0;
    __syncthreads();
    const int b = blockIdx.x;                                                  // (uniform per CTA: no barrier is skipped by a part of it)
    if (p.skip && p.skip[b]) return;
    double* lu = smem + WS::LU + warp * 2 * D * WS::DP;
    double* stage_ring = smem + WS::STAGE;
    double* prefix_ring = smem + WS::PREFIX;
    int status = 0;
    if (warp < epl::kWspStageWarps) epl::wsp_stage_role<D, M>(p, b, warp, lu, stage_ring, cst, status);
    else if (warp == epl::kWspStageWarps) epl::wsp_prefix_role<D, M>(p, lu, stage_ring, prefix_ring, status);
    else {
        const int q = warp - epl::kWspStageWarps - 1;
        epl::wsp_query_role<D, M>(p, b, q, lu, prefix_ring, cst, smem + WS::RESULT + q * 4, status);
    }
    if (lane == 0) status_words[warp] = status;
    __syncthreads();
    if (threadIdx.x == 0) {
        ArgMin am;
        am.init();
        int st = 0;
        for (int q = 0; q < epl::kWspQueryWarps; ++q) {
            const double* r = smem + WS::RESULT + q * 4;
            epl::wsp_merge(am, r[0], (int)r[1], r[2] != 0.0);
        }
        for (int w = 0; w < epl::kWspWarps; ++w) st |= status_words[w];
        p.T_out[b] = am.idx;
        p.Jstar_out[b] = am.best;
        p.status[b] = st;
    }
}

template <int D, int M>
static int launch_fused_wsp(const FusedArgs& p, cudaStream_t st) {
    const size_t smem = sizeof(double) * ((size_t)epl::WspSmem<D>::SIZE + FusedConst<D, M>::SIZE);
    k_select_fused_wsp<D, M><<<p.B, epl::kWspWarps * 32, smem, st>>>(p);
    return check_launch("k_select_fused_wsp");
}

// fused selection kernel of the small systems: 0 routing by batch size (default), 1 lane group per problem, 2 warp-specialised
// pipeline, 3 element per lane, one warp (test hook; all three give identical bits)
int g_fused_small_variant = 0;

// A warp per problem only pays while the batch leaves the machine empty (measured on B200, x0 -> T* pipeline, element per
// lane vs lane group: Segway B = 25 0.86 vs 1.30 ms, Cartpole B = 25 1.42 vs 2.13 ms, DI B = 25 0.28 vs 0.40 ms; at
// B = 4096 the lane-group kernel, which packs 4-8 problems into a warp, is ahead: 2.15 vs 1.88 ms).
// The pipeline spends seven warps on a problem: it pays while the batch leaves most SMs idle (up to 592 =
// 4 CTAs per SM; cartpole select phase, pipeline vs one warp per problem, ms: 148 instances 4.29 / 11.8, 296: 5.72 / 11.8, 444: 10.4 / 12.3,
// 592: 11.1 / 12.3, 1 024 (before the deferred prefix update): 20.7 / 14.3).
constexpr long max_batch = 1024, wsp_max_batch = 592;
int dispatch_select_fused_epl(int n, int m, const FusedArgs& p, cudaStream_t st) {
    const int v = g_fused_small_variant;
    if (v == 1 || (v == 0 && p.B > max_batch)) return HOP_E_UNSUPPORTED_DIMS;
    const bool wsp = (v == 2) || (v == 0 && p.B <= wsp_max_batch);
    if (n == 2 && m == 1) return wsp ? launch_fused_wsp<3, 1>(p, st) : launch_fused_epl<3, 1>(p, st);
    if (n == 4 && m == 1) return wsp ? launch_fused_wsp<5, 1>(p, st) : launch_fused_epl<5, 1>(p, st);
    return HOP_E_UNSUPPORTED_DIMS;
}

}  // namespace hop
