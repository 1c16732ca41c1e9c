// hop_select_tpp.cu -- __global__ wrapper + launcher of the thread-per-problem LQR-boundary selection kernel
// (hop_select_tpp_body.cuh).  Grid: one warp per CTA, 32 problems per warp; dynamic shared memory = the warp's
// double-buffered input stage.
#include <cstdint>

#include "hop_common.cuh"
#include "hop_select_tpp_body.cuh"
#include "../../include/hop_b200.h"

namespace hop {
template <int D, int M>
__global__ void __launch_bounds__(32) k_select_generic_tpp(const SelectArgs p) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x;
    const int b0 = blockIdx.x * 32, b = b0 + lane;
    tpp::SmemFeed<D, M> feed;
    feed.init(p, b0, lane, smem);
    tpp::select_generic_tpp_body<D, M>(p, b < p.B ? b : p.B - 1, b < p.B, feed);
}
template <int D, int M>
static int launch_generic_tpp(const SelectArgs& p, cudaStream_t st) {
    const size_t smem = sizeof(double) * (size_t)tpp::StageGeo<D, M>::WARP_DOUBLES;
    cudaError_t e = cudaFuncSetAttribute(k_select_generic_tpp<D, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_generic_tpp)");
    k_select_generic_tpp<D, M><<<(p.B + 31) / 32, 32, smem, st>>>(p);
    return check_launch("k_select_generic_tpp");
}
// Which batches go to the thread-per-problem kernel (measured on B200, N = 128, profiles/r1h_tpp_vs_lanes.txt): for
// d <= 4 it is faster than the lane-group kernel at EVERY batch size (B = 32: 0.38 vs 0.55 ms, B = 2^19: 8.8 vs 30.6 ms);
// for d = 5 its register spills make one step slower (1.0 vs 0.67 ms for a single wave), so it only pays once the batch
// fills the machine.  -1 = these defaults; >= 0 (test hook) = one threshold for every d.
static long g_tpp_min_batch = -1;
long tpp_min_batch(long set_to) {   // set_to < -1: query only.  Returns the previous value.
    const long old = g_tpp_min_batch;
    if (set_to >= -1) g_tpp_min_batch = set_to;
    return old;
}
static bool use_tpp(int d, int m, const SelectArgs& p) {
    long min_batch = tpp_min_batch(-2);
    if (min_batch < 0) min_batch = (d <= 4) ? 0 : 16384;
    if (p.B < min_batch || p.rinv_step_stride != 0) return false;   // (one R^-1 per instance only)
    if ((d * d) % 2 == 0 && (d * m) % 2 == 0) {
        const uintptr_t bits = (uintptr_t)p.A_aug | (uintptr_t)p.B_aug | (uintptr_t)p.Q_aug | (uintptr_t)p.QT;
        if (bits & 15u) return false;
    }
    return true;
}


int dispatch_select_generic_tpp(int d, int m, const SelectArgs& p, cudaStream_t st) {
    if (!use_tpp(d, m, p)) return HOP_E_UNSUPPORTED_DIMS;
    if (d == 3 && m == 1) return launch_generic_tpp<3, 1>(p, st);
    if (d == 4 && m == 2) return launch_generic_tpp<4, 2>(p, st);
    if (d == 5 && m == 1) return launch_generic_tpp<5, 1>(p, st);
    return HOP_E_UNSUPPORTED_DIMS;
}

}  // namespace hop
