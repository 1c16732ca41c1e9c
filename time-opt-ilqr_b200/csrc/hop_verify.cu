// hop_verify.cu -- HOP_MODE_VERIFIED (include/hop_b200.h) for the fused forms and hop_select_verified_f64 (LQR boundary):
// FAST selection, near-tie scan, EXACT re-evaluation of the marked instances.  Three launches on the caller's stream and no host synchronisation: the scan appends the marked instances to a
// device list, and the EXACT kernel's list mode runs a fixed grid whose warps take instances from that list until its count
// runs out, so the host never reads the count.
#include "hop_common.cuh"
#include "hop_select_body.cuh"
#include "hop_verify_body.cuh"
#include "../../include/hop_b200.h"

namespace hop {

constexpr int kScanWarps = 8;

// w_explicit: null, or [B] at the LQR boundary (the scanned curve is then J + w t, hop_verify_body.cuh)
__global__ void __launch_bounds__(kScanWarps * 32) k_tie_scan(const verify::TieScanArgs a, const double* w_explicit, int* list,
                                                             int* list_count) {
    const int b = blockIdx.x * kScanWarps + (threadIdx.x >> 5);
    if (b >= a.B || (a.skip && a.skip[b])) return;
    const bool mark = verify::tie_scan_warp(a, b, w_explicit);
    // one instance per warp, so one atomic per marked warp; the list order is arbitrary and no output depends on it
    if (mark && (threadIdx.x & 31) == 0) list[atomicAdd(list_count, 1)] = b;
}

// Steps 2 and 3 of VERIFIED, after the FAST selection has written a.J / a.T_star / a.status: stream-ordered scratch of B + 1
// ints (count, list), the near-tie scan, then exact(list, count), which launches the EXACT kernel's list mode.  No host
// synchronisation.
template <typename Exact>
static int scan_and_reevaluate(const verify::TieScanArgs& a, const double* w_explicit, cudaStream_t st, Exact exact) {
    void* ws = nullptr;
    if (int rc = stream_alloc(&ws, sizeof(int) * ((size_t)a.B + 1), st, "cudaMallocAsync(verification list)")) return rc;
    int* count = (int*)ws;
    int* list = count + 1;
    int rc = report_cuda(cudaMemsetAsync(count, 0, sizeof(int), st), "memset(verification count)");
    if (!rc) {
        k_tie_scan<<<(a.B + kScanWarps - 1) / kScanWarps, kScanWarps * 32, 0, st>>>(a, w_explicit, list, count);
        rc = check_launch("k_tie_scan");
    }
    if (!rc) rc = exact(list, count);
    stream_free(ws, st);
    return rc;
}

// relative tie tolerance of the scan for state dimension n, measured per n (include/hop_b200.h); 0 = VERIFIED is not offered
// for that n (n = 4: the cartpole embedding has no tolerance that both holds and re-evaluates a minority)
double verify_tie_tol(int n) {
    if (n == 12) return HOP_VERIFY_TIE_TOL;
    if (n == 2) return HOP_VERIFY_TIE_TOL_N2;
    return 0.0;
}

int dispatch_select_verified(int n, int m, const FusedArgs& p, cudaStream_t st) {
    const double tol = verify_tie_tol(n);
    if (!(tol > 0.0)) {
        set_last_error("HOP_MODE_VERIFIED: no calibrated tie tolerance for this state dimension (include/hop_b200.h)");
        return HOP_E_UNSUPPORTED_DIMS;
    }
    FusedArgs f = p;
    f.mode = HOP_MODE_FAST;
    if (int rc = dispatch_select_fused(n, m, f, st)) return rc;
    const verify::TieScanArgs a{p.B, p.T_min, p.T_max, tol, p.J_out, p.T_out, p.status, p.skip};
    return scan_and_reevaluate(a, nullptr, st, [&](const int* list, const int* count) {
        FusedArgs e = p;
        e.mode = HOP_MODE_EXACT;
        return launch_ref_fused_list(n, m, e, list, count, st);
    });
}

// hop_select_verified_f64: the LQR-boundary form with the caller's tolerance.  The FAST step is dispatch_select_generic's
// FAST routing unchanged (thread per problem, lane group, pipelined with or without the pre-pass, the test hooks); the scan
// reads J + w t when w_explicit is given, the curve the kernels minimised.
int dispatch_select_generic_verified(int d, int m, double tol, const SelectArgs& p, cudaStream_t st) {
    if (int rc = dispatch_select_generic(d, m, HOP_MODE_FAST, p, st)) return rc;
    const verify::TieScanArgs a{p.B, p.T_min, p.T_max, tol, p.J_out, p.T_out, p.status, nullptr};
    return scan_and_reevaluate(a, p.w_explicit, st, [&](const int* list, const int* count) {
        return launch_ref_generic_list(d, m, p, list, count, st);
    });
}

}  // namespace hop
