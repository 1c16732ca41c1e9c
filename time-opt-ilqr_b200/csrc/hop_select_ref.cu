// hop_select_ref.cu -- __global__ wrappers + launchers of HOP_MODE_EXACT (reference operation order,
// hop_select_ref_body.cuh) and HOP_MODE_FP32 (the same sweep in single precision, LQR-boundary entry only).
//
// Grid: one warp per problem, no CTA barrier inside the sweep.  Dynamic shared memory = one slab per warp (ref::Layout,
// 19.3 KB at d = 13 in fp64) [+ the CTA-wide case constants of the fused form].  Warps per CTA are chosen at launch: as
// many as the 227 KB of an SM hold (11 at d = 13) when the batch fills the machine, fewer for small batches so that the
// problems spread over the SMs.
#include <type_traits>

#include "hop_common.cuh"
#include "hop_select_ref_body.cuh"
#include "../../include/hop_b200.h"

namespace hop {

constexpr int kRefMaxWarps = 16;
constexpr size_t kSmemPerSm = 227 * 1024;
// warps per CTA of the list mode (HOP_MODE_VERIFIED re-evaluation): a few listed instances should spread over all SMs instead
// of sharing one SM's issue slots, and with one warp per CTA the block scheduler places them breadth-first
#ifndef HOP_REF_LIST_WARPS
#define HOP_REF_LIST_WARPS 1
#endif
constexpr int kRefListWarps = HOP_REF_LIST_WARPS;

// warps per CTA: fill one SM's shared memory when there is at least one such CTA per SM, else spread the batch
static int ref_warps(int B, size_t slab_bytes, size_t cst_bytes) {
    int fit = (int)((kSmemPerSm - cst_bytes - 1024) / slab_bytes);
    fit = fit < 1 ? 1 : (fit > kRefMaxWarps ? kRefMaxWarps : fit);
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if ((long)B >= (long)fit * sms) return fit;
    const int spread = (B + sms - 1) / sms;
    return spread < 1 ? 1 : (spread > fit ? fit : spread);
}

// grid of the list mode (both forms): CTAs of kRefListWarps warps and cta_smem bytes, just enough for B instances or for one
// fill of the machine, whichever is smaller
static int list_grid(int B, size_t cta_smem) {
    const int fit = (int)((kSmemPerSm - 1024) / cta_smem);
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int full = sms * (fit < 1 ? 1 : fit);
    const int grid = (B + kRefListWarps - 1) / kRefListWarps;
    return grid > full ? full : grid;
}

// list == null: warp w of the grid computes instance w.  List mode (HOP_MODE_VERIFIED, fp64 only): as in k_select_ref_fused,
// a fixed grid whose warps take list[0 .. *list_count) with a grid stride (ref::select_generic_list).
template <typename R>
__global__ void __launch_bounds__(kRefMaxWarps * 32) k_select_ref_generic(const SelectArgs p, int d, int m, int slab,
                                                                         const int* list, const int* list_count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5;
    R* s = reinterpret_cast<R*>(smem_raw) + (size_t)warp * slab;
    if constexpr (std::is_same<R, double>::value) {
        if (list) {
            ref::select_generic_list(p, d, m, list, *list_count, blockIdx.x * warps + warp, gridDim.x * warps, s);
            return;
        }
    }
    const int b = blockIdx.x * warps + warp;
    if (b >= p.B) return;
    ref::select_generic_body<R>(p, d, m, b, s);
}

// list == null: warp w of the grid computes instance w.  List mode (HOP_MODE_VERIFIED): the grid is fixed at launch and its warps
// take the instances list[0 .. *list_count) with a grid stride, so the launch needs no host-side count; each computed instance
// gets HOP_ST_FLAG_REEVALUATED.
__global__ void __launch_bounds__(kRefMaxWarps * 32) k_select_ref_fused(const FusedArgs p, int n, int m, int slab, const int* list,
                                                                       const int* list_count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* smem = reinterpret_cast<double*>(smem_raw);
    const int warps = blockDim.x >> 5;
    double* cst = smem + (size_t)warps * slab;
    const int warp = threadIdx.x >> 5;
    if (list) {
        const int count = *list_count;
        if (blockIdx.x * warps >= count) return;                                  // CTA-uniform: no work for this CTA
        ref::fused_cst_fill(p, n, m, cst, threadIdx.x, blockDim.x);
        __syncthreads();
        for (int i = blockIdx.x * warps + warp; i < count; i += gridDim.x * warps) {
            const int b = list[i];
            __syncwarp();                                                         // the previous instance's slab reads are done
            ref::select_fused_body(p, n, m, b, smem + (size_t)warp * slab, cst);
            if ((threadIdx.x & 31) == 0) p.status[b] |= HOP_ST_FLAG_REEVALUATED;
        }
        return;
    }
    ref::fused_cst_fill(p, n, m, cst, threadIdx.x, blockDim.x);
    __syncthreads();
    const int b = blockIdx.x * warps + warp;
    if (b >= p.B || (p.skip && p.skip[b])) return;
    ref::select_fused_body(p, n, m, b, smem + (size_t)warp * slab, cst);
}

template <typename R>
static int launch_ref_generic(int d, int m, const SelectArgs& p, const int* list, const int* list_count, cudaStream_t st) {
    const int slab = (ref::Layout::make(d, m).size + 1) & ~1;
    int warps = ref_warps(p.B, sizeof(R) * (size_t)slab, 0), grid = (p.B + warps - 1) / warps;
    if (list) {
        warps = kRefListWarps;
        grid = list_grid(p.B, sizeof(R) * (size_t)warps * slab);
    }
    const size_t smem = sizeof(R) * (size_t)warps * slab;
    cudaError_t e = cudaFuncSetAttribute(k_select_ref_generic<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_ref_generic)");
    k_select_ref_generic<R><<<grid, warps * 32, smem, st>>>(p, d, m, slab, list, list_count);
    return check_launch("k_select_ref_generic");
}

int dispatch_select_ref_generic(int d, int m, bool fp32, const SelectArgs& p, cudaStream_t st) {
    if (d < 1 || d > ref::kMaxD || m < 1 || m > ref::kMaxD) {
        set_last_error("hop_select_f64: HOP_MODE_EXACT / HOP_MODE_FP32 need 1 <= d, m <= 16");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    return fp32 ? launch_ref_generic<float>(d, m, p, nullptr, nullptr, st) : launch_ref_generic<double>(d, m, p, nullptr, nullptr, st);
}

// HOP_MODE_EXACT on the instances list[0 .. *list_count) only (device memory, *list_count <= p.B, each instance at most once),
// each then flagged HOP_ST_FLAG_REEVALUATED; fp64, 1 <= d, m <= 16.
int launch_ref_generic_list(int d, int m, const SelectArgs& p, const int* list, const int* list_count, cudaStream_t st) {
    if (d < 1 || d > ref::kMaxD || m < 1 || m > ref::kMaxD) {
        set_last_error("hop_select_verified_f64: HOP_MODE_EXACT needs 1 <= d, m <= 16");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    return launch_ref_generic<double>(d, m, p, list, list_count, st);
}

// list == null: every instance of p (b < p.B, skip honoured).  Otherwise the instances list[0 .. *list_count) (device memory,
// *list_count <= p.B, each instance at most once), on the grid of list_grid.
int launch_ref_fused_list(int n, int m, const FusedArgs& p, const int* list, const int* list_count, cudaStream_t st) {
    if (n < 1 || n + 1 > ref::kMaxD || m < 1 || m > n + 1) {
        set_last_error("hop_select_fused_f64: HOP_MODE_EXACT needs 1 <= n <= 15 and 1 <= m <= n + 1");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    const int slab = (ref::Layout::make(n + 1, m).size + 1) & ~1;
    const size_t cst_bytes = sizeof(double) * (size_t)ref::FusedCst::make(n, m).size;
    int warps = ref_warps(p.B, sizeof(double) * (size_t)slab, cst_bytes), grid = (p.B + warps - 1) / warps;
    if (list) {
        warps = kRefListWarps;
        grid = list_grid(p.B, sizeof(double) * (size_t)warps * slab + cst_bytes);
    }
    const size_t smem = sizeof(double) * (size_t)warps * slab + cst_bytes;
    cudaError_t e = cudaFuncSetAttribute(k_select_ref_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return report_cuda(e, "cudaFuncSetAttribute(k_select_ref_fused)");
    k_select_ref_fused<<<grid, warps * 32, smem, st>>>(p, n, m, slab, list, list_count);
    return check_launch("k_select_ref_fused");
}

}  // namespace hop
