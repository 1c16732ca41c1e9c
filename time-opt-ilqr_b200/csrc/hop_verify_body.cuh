// hop_verify_body.cuh -- HOP_MODE_VERIFIED: near-tie scan of a selection curve (one warp per instance).
//
// The scan decides which instances of a FAST selection are recomputed by the EXACT kernel (include/hop_b200.h,
// HOP_MODE_VERIFIED).  It reads the window J[b][T_min-1 .. T_max-1] of the curve the kernel minimised and marks the instance
// when another horizon lies within the relative tolerance of the minimum, when the window holds a NaN or an infinity, when
// the selection reported a non-zero status, or when its own argmin differs from the selection's T* (defensive).
//
// Argmin rules are np.argmin's: the first minimum wins and the first NaN wins.  Lane l reads horizons T_min + l + 32 i
// (coalesced), keeps its own (value, horizon) by those rules, and the warp combines the 32 candidates with a butterfly whose
// combine step is commutative and associative (a NaN beats a number, then the smaller value, then the smaller horizon), so
// every lane ends with the same, order-independent result.  "Within the tolerance" is evaluated per horizon as
// (J(t) - J1) / |J1| < tol with individually rounded operations: rounding is monotone, so some horizon passes exactly when
// oracle/census.py argmin_gap (the same expression on the minimum over t != T*) is below tol.
//
// At the LQR boundary with an explicit time weight (hop_select_verified_f64, w_explicit given) the kernel minimised
// v(t) = J(t) + w t while J_out holds the raw J(t); the scan then reads v(t) = add_rn(J(t), mul_rn(w, t)), the expression
// (and the two roundings) of the EXACT body, so that the scan's argmin is EXACT's argmin on the same curve.
#pragma once
#include "hop_simt.cuh"

namespace hop { namespace verify {

struct TieScanArgs {
    int B, T_min, T_max;
    double tol;
    const double* J;        // [B][T_max]
    const int* T_star;      // [B]
    const int* status;      // [B]
    const int* skip;        // optional [B]: non-zero => not scanned (never marked)
};

// (v, t) with t = 0 for "no candidate"; returns true when (v2, t2) wins over (v1, t1)
HOP_DEVICE bool argmin_takes(double v1, int t1, double v2, int t2) {
    if (t2 == 0) return false;
    if (t1 == 0) return true;
    const bool n1 = v1 != v1, n2 = v2 != v2;
    if (n1 != n2) return n2;
    if (!n1 && v2 != v1) return v2 < v1;
    return t2 < t1;
}

// warp-uniform: true when instance b is to be re-evaluated.  w_explicit: null (the curve is J_out), or [B] (the curve is
// J_out + w t).  A separate argument rather than a TieScanArgs field, so that the struct keeps its layout.
HOP_DEVICE bool tie_scan_warp(const TieScanArgs& a, int b, const double* w_explicit = nullptr) {
    const int lane = simt::lane_id();
    const double* row = a.J + (size_t)b * a.T_max;
    const double w = w_explicit ? w_explicit[b] : 0.0;
    auto curve = [&](int t) { return w_explicit ? simt::add_rn(row[t - 1], simt::mul_rn(w, (double)t)) : row[t - 1]; };
    double best = 0.0;
    int tb = 0;
    bool nonfinite = false;
    for (int t = a.T_min + lane; t <= a.T_max; t += 32) {
        const double v = curve(t);
        nonfinite = nonfinite || !isfinite(v);
        if (argmin_takes(best, tb, v, t)) { best = v; tb = t; }
    }
    for (int off = 16; off >= 1; off >>= 1) {
        const double v = simt::shfl_xor(best, off, 32);
        const int t = (int)simt::shfl_xor((double)tb, off, 32);
        if (argmin_takes(best, tb, v, t)) { best = v; tb = t; }
    }
    bool close = false;
    if (!nonfinite) {            // (a lane that saw a non-finite value marks the instance anyway)
        const double scale = fabs(best);
        for (int t = a.T_min + lane; t <= a.T_max; t += 32)
            if (t != tb) close = close || ((curve(t) - best) / scale < a.tol);
    }
    const bool mark_here = nonfinite || close;
    return simt::ballot(mark_here) != 0u || a.status[b] != 0 || tb != a.T_star[b];
}

}}  // namespace hop::verify
