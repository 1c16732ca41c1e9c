// emul_verify_lqr.cpp -- host entry points that run the LQR-boundary HOP_MODE_VERIFIED kernels under the SIMT emulator (test
// infrastructure; mirrors k_tie_scan with w_explicit in hop_verify.cu and the list mode of k_select_ref_generic in
// hop_select_ref.cu, whose per-warp loop is ref::select_generic_list).
#include <vector>

#include "hop_select_ref_body.cuh"
#include "hop_verify_body.cuh"
#include "../../include/hop_b200.h"

namespace {
struct ScanJob { const hop::verify::TieScanArgs* a; const double* w; int b; int mark; };
void scan_lane(void* p) {
    auto* j = (ScanJob*)p;
    const bool m = hop::verify::tie_scan_warp(*j->a, j->b, j->w);
    if (hop::simt::lane_id() == 0) j->mark = m ? 1 : 0;
}
struct RefGenericListJob { const hop::SelectArgs* p; int d, m; const int* list; int count; double* slab; };
void ref_generic_list_lane(void* a) {
    auto* j = (RefGenericListJob*)a;
    hop::ref::select_generic_list(*j->p, j->d, j->m, j->list, j->count, 0, 1, j->slab);
}
}  // namespace

// k_tie_scan with the scanned curve J + w t (w: [B]) or J (w null): the marked instances are appended in ascending order (the
// device order is arbitrary)
extern "C" int emul_tie_scan_w(const hop::verify::TieScanArgs* a, const double* w, int* list, int* count) {
    *count = 0;
    for (int b = 0; b < a->B; ++b) {
        if (a->skip && a->skip[b]) continue;
        ScanJob j{a, w, b, 0};
        if (hop::simt::run_warp(scan_lane, &j)) return -1;
        if (j.mark) list[(*count)++] = b;
    }
    return 0;
}

// k_select_ref_generic in list mode (one warp taking every listed instance): list[0 .. count), each followed by
// HOP_ST_FLAG_REEVALUATED
extern "C" int emul_select_generic_ref_list(int d, int m, const hop::SelectArgs* p, const int* list, int count) {
    if (d < 1 || d > hop::ref::kMaxD || m < 1 || m > hop::ref::kMaxD) return -2;
    std::vector<double> slab(hop::ref::Layout::make(d, m).size, -7.0);
    RefGenericListJob j{p, d, m, list, count, slab.data()};
    return hop::simt::run_warp(ref_generic_list_lane, &j) ? -1 : 0;
}
