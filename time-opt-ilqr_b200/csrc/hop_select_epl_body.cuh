// hop_select_epl_body.cuh -- fused HOP horizon selection for small systems (d = n+1 <= 5), ONE WARP PER PROBLEM,
// ONE MATRIX ELEMENT PER LANE.
//
// Replaces (reference file:line, dmmsjtu-umich/time-opt-ilqr), same as select_fused_body in hop_select_body.cuh:
//   augmented.py:10-87            build_augmented_sequence_QR + build_terminal_aug_list (built in registers)
//   utils.py:35-37,69-93          _sym, chol_inv (jitter ladder, LU fallback)
//   horizon_selection.py:57-86    stage, prefix composition, per-horizon query J(T)
//   solver.py:522,590             argmin over [T_min, T_max]
//
// Why a third mapping: the HOP-DDP configurations of the small systems (Segway 25 trials, Cartpole 4096 initial
// states, N = 240 / 360) are LATENCY bound -- the sweep over the horizon is sequential and the batch does not fill
// the machine.  The lane-group kernel (row per lane, operands through shared memory, a __syncwarp per pivot and per
// product) needs 11-14 k clocks per horizon step at d = 5.  Here lane 5r + c owns element (r, c) of every block:
// a product is d shuffle pairs + d dependent DFMAs per lane, a Gauss-Jordan pivot is three shuffles, one division and
// one FMA, _sym is one shuffle, the pivot (hence "Cholesky failed") is the same value on every lane so the jitter
// ladder needs no vote, and nothing goes through shared memory except the case constants.
//
// Every element is produced by the same IEEE operations in the same order as in select_fused_body (fma chains in
// ascending index order, same divisions, same ladder decisions, same summation trees), so the two kernels are
// bit-identical; tests assert that on the host emulator and on the GPU.
#pragma once
#include "hop_select_body.cuh"

namespace hop { namespace epl {

template <int D>
struct Geo {   // lane = D r + c for lane < D^2; the idle lanes mirror element (0, 0) and never write
    int lane, r, c;
    bool act;
    HOP_DEVICE void init() {
        lane = simt::lane_id();
        act = lane < D * D;
        r = act ? lane / D : 0;
        c = act ? lane % D : 0;
    }
};

HOP_DEVICE double at(double v, int src) { return simt::shfl(v, src, 32); }

// C = X Y, C = X Y^T, C = X^T Y on D x D blocks (one element per lane); fma chains in ascending l from +0.0
template <int D>
HOP_DEVICE double mul_nn(double x, double y, int r, int c) {
    double s = 0.0;
#pragma unroll
    for (int l = 0; l < D; ++l) s = fma(at(x, r * D + l), at(y, l * D + c), s);
    return s;
}
template <int D>
HOP_DEVICE double mul_nt(double x, double y, int r, int c) {
    double s = 0.0;
#pragma unroll
    for (int l = 0; l < D; ++l) s = fma(at(x, r * D + l), at(y, c * D + l), s);
    return s;
}
template <int D>
HOP_DEVICE double mul_tn(double x, double y, int r, int c) {
    double s = 0.0;
#pragma unroll
    for (int l = 0; l < D; ++l) s = fma(at(x, l * D + r), at(y, l * D + c), s);
    return s;
}
// utils.py:35-37
template <int D>
HOP_DEVICE double sym(double v, int r, int c) { return 0.5 * (v + at(v, c * D + r)); }

// One Gauss-Jordan inversion attempt (hop::gj_attempt element for element).  The pivot is the same value on every
// lane, so the returned flag is warp-uniform.  (Forming the next pivot on every lane from the pre-update entries -- same
// bits, one shuffle latency less per elimination step -- was measured three times: one-warp kernel -3 %, pipeline unchanged or slower,
// also when applied to the prefix warp's inversion only: three more shuffles per pivot cost more than the latency saved.  Not kept.)
template <int D>
HOP_DEVICE bool gj_attempt(double& a, int r, int c) {
    bool ok = true;
#pragma unroll
    for (int j = 0; j < D; ++j) {
        const double p = at(a, j * D + j);
        ok = ok && (p > 0.0) && (p <= 1.7976931348623157e308);   // +Inf is non-finite input (utils.py:75), not a pivot
        const double rinv = simt::rcp_newton(p);
        const double rowv = at(a, j * D + c);      // pivot row, my column
        const double colv = at(a, r * D + j);      // my row, pivot column
        if (r == j) {
            a = (c == j) ? rinv : fma(rinv, rowv, 0.0);
        } else {
            const double nf = -(colv * rinv);
            a = (c == j) ? nf : fma(nf, rowv, a);
        }
    }
    return ok;
}

// chol_inv (utils.py:69-93) of a symmetrised block s (element per lane).  scratch: 2 D DP doubles of per-warp shared
// memory, touched by the LU fallback only.  `act`: lane owns an element of this block.
template <int D>
HOP_DEVICE double chol_inv(double s, int r, int c, bool act, double* scratch, double jitter, int max_tries, int& status) {
    constexpr int DP = (D + 1) & ~1;
    double eps = jitter;
    for (int tries = 0;;) {
        double a = s + ((r == c) ? eps : 0.0);
        if (gj_attempt<D>(a, r, c)) return a;
        if (tries == 0 && !simt::all(!act || isfinite(s))) {   // utils.py:75: a non-finite input raises before any attempt
            status |= ST_NONFINITE;
            return nan("");
        }
        status |= ST_FLAG_RETRY;
        eps *= 10.0;
        ++tries;
        if (tries >= max_tries) {                               // utils.py:90-93: LU with partial pivoting on (s + eps I)
            double* f1 = scratch;
            double* f2 = scratch + D * DP;
            simt::sync();
            if (act) f1[r * DP + c] = s + ((r == c) ? eps : 0.0);
            simt::sync();
            bool lu_ok = true;
            if (simt::lane_id() == 0) lu_ok = lu_inverse_serial<D, DP>(f1, f2);
            simt::sync();
            lu_ok = simt::shfl(lu_ok ? 1.0 : 0.0, 0, 32) != 0.0;
            const double out = f2[r * DP + c];
            simt::sync();
            status |= ST_FLAG_LU;
            if (!lu_ok) status |= ST_LINALG;
            return out;
        }
    }
}

// hop::group_sum<G> of the values v_0 .. v_{CNT-1} held by lanes 0 .. CNT-1 (zeros on the other lanes of the group):
// every lane gathers them and walks the same xor tree, so the sum has the lane-group kernel's association order.
template <int CNT, int G>
HOP_DEVICE double tree_sum(double v, int stride) {
    double part[G];
#pragma unroll
    for (int i = 0; i < G; ++i) part[i] = (i < CNT) ? at(v, i * stride) : 0.0;
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1)
#pragma unroll
        for (int i = 0; i < o; ++i) part[i] = simt::add_rn(part[i], part[i + o]);
    return part[0];
}

// scratch: per-warp shared memory, 2 D DP doubles.  cst: CTA constants (FusedConst, fused_const_fill).
template <int D, int M>
HOP_DEVICE void select_fused_epl_body(const FusedArgs& p, int b, double* scratch, const double* cst) {
    using FC = FusedConst<D, M>;
    constexpr int n = D - 1;
    constexpr int G = (D <= 4) ? 4 : 8;            // group width of the lane-group kernel (its summation trees)
    static_assert(D * D <= 32 && D * M <= 32 && M * M <= 32 && M <= D, "one element per lane");
    Geo<D> L;
    L.init();
    const int lane = L.lane, r = L.r, c = L.c;
    const bool isx = lane < n;                      // lane i < n also owns component i of the small vectors
    const int li = isx ? lane : 0;
    const bool isb = lane < D * M;                  // lane rB M + cB owns B_aug[rB][cB]
    const int rB = isb ? lane / M : 0, cB = isb ? lane % M : 0;
    const bool ism = lane < M * M;                  // lane rM M + cM owns R^-1[rM][cM]
    const int rM = ism ? lane / M : 0, cM = ism ? lane % M : 0;
    int status = 0;

    // R_inv = chol_inv(sym(R))  (augmented.py:23)
    const double rinv_e = chol_inv<M>(cst[FC::RS + rM * M + cM], rM, cM, ism, scratch, p.jitter, p.max_tries, status);
    const double xg_l = isx ? p.xg[(size_t)b * n + li] : 0.0;
    const bool wrap_l = isx && ((p.wrap_mask >> li) & 1u);
    const double uref_l = (lane < M) ? cst[FC::UREF + lane] : 0.0;
    const double w = p.w[b];
    // constants of this lane: rows / columns of Q, P for the matvecs; own elements of Qs, P
    const double qs_e = (r < n && c < n) ? cst[FC::QS + r * n + c] : 0.0;
    const double pf_e = (r < n && c < n) ? cst[FC::PF + r * n + c] : 0.0;

    const size_t baseN = (size_t)b * p.N;
    const double* Xb = p.X + (size_t)b * (p.N + 1) * n;
    const double* Ub = p.U + (size_t)b * p.u_stride;
    auto wrapped = [&](double x) {                  // e = wrap(X - xg) on this lane's component (augmented.py:28,80)
        double v = 0.0;
        if (isx) {
            v = x - xg_l;
            if (wrap_l) v = wrap_pi(v);
        }
        return v;
    };
    // loads of one step: own element of A_k, own element of B_k, row li of B_k, a_k, U_k, X_{k+1}
    struct Step { double a, bm, brow[M], ar, u, x1; };
    auto load_step = [&](int k) {
        Step s;
        const bool in = k < p.T_max;
        const double* Ak = p.A + (baseN + k) * n * n;
        const double* Bk = p.Bm + (baseN + k) * n * M;
        s.a = (in && L.act && r < n && c < n) ? Ak[r * n + c] : 0.0;
        s.bm = (in && isb && rB < n) ? Bk[rB * M + cB] : 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j) s.brow[j] = (in && isx) ? Bk[li * M + j] : 0.0;
        s.ar = (in && isx && p.a_resid) ? p.a_resid[(baseN + k) * n + li] : 0.0;
        s.u = (in && lane < M) ? Ub[(size_t)k * M + lane] : 0.0;
        s.x1 = (in && isx) ? Xb[(size_t)(k + 1) * n + li] : 0.0;
        return s;
    };

    double eb = 0.0, fb = 0.0, gb = 0.0;
    ArgMin am;
    am.init();
    double ev = wrapped(isx ? Xb[li] : 0.0);       // e_0; afterwards e_{k+1} of step k is e_k of step k+1 (same expression)
    Step cur = load_step(0);
    for (int k = 0; k < p.T_max; ++k) {
        const Step nxt = load_step(k + 1);          // in flight while step k computes
        // ---- augmented blocks of step k (augmented.py:31-56)
        const double du = (lane < M) ? cur.u - uref_l : 0.0;
        double colA = 0.0;                          // A_aug[i][n] = a_k - B_k du
        {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < M; ++j) s = fma(cur.brow[j], at(du, j), s);
            colA = cur.ar - s;
        }
        const double colA_r = at(colA, r);
        const double a_e = (r < n) ? ((c < n) ? cur.a : colA_r) : ((c == n) ? 1.0 : 0.0);
        const double b_e = cur.bm;                  // (row n of B_aug is zero: load_step returned 0)
        double qe = 0.0, qc = 0.0;
#pragma unroll
        for (int j = 0; j < n; ++j) {
            const double ej = at(ev, j);
            qe = fma(cst[FC::QRAW + li * n + j], ej, qe);                       // (Q e)_i
            qc = fma(ej, cst[FC::QRAW + j * n + li], qc);                       // (e^T Q)_i
        }
        const double eQe = tree_sum<n, G>(isx ? simt::mul_rn(qc, ev) : 0.0, 1);
        const double qe_x = at(qe, (r == n) ? c : r);
        const double q_e = (r < n) ? ((c < n) ? qs_e : qe_x) : ((c < n) ? qe_x : (eQe + 2.0 * w + p.rho_reg));

        // ---- stage (horizon_selection.py:57-64)
        const double e = chol_inv<D>(q_e, r, c, L.act, scratch, p.jitter, p.max_tries, status);
        double wv = 0.0;
        if (k > 0) {
            const double s = sym<D>(e + gb, r, c);
            wv = chol_inv<D>(s, r, c, L.act, scratch, p.jitter, p.max_tries, status);      // W = chol_inv(E_k + Gbar)  (:72)
        }
        const double f = mul_nt<D>(e, a_e, r, c);                                          // F_k = E_k A_k^T
        double g;
        {
            const double t = mul_nn<D>(a_e, e, r, c);                                      // A E
            g = mul_nt<D>(t, a_e, r, c);                                                   // (A E) A^T
            double br = 0.0;                                                               // (B R^-1)[rB][cB]
#pragma unroll
            for (int l = 0; l < M; ++l) br = fma(at(b_e, rB * M + l), at(rinv_e, l * M + cB), br);
#pragma unroll
            for (int l = 0; l < M; ++l) g = fma(at(br, r * M + l), at(b_e, c * M + l), g);  // + (B R^-1) B^T
            g = sym<D>(g, r, c);
        }
        if (k == 0) {
            eb = e; fb = f; gb = g;
        } else {
            // ---- prefix composition (:70-75); every right-hand side uses the OLD (Ebar, Fbar, Gbar)
            const double t1 = mul_nn<D>(fb, wv, r, c);                                     // Fbar W
            const double acc = mul_nt<D>(t1, fb, r, c);                                    // (Fbar W) Fbar^T
            const double eb_new = eb - acc;
            const double fb_new = mul_nn<D>(t1, f, r, c);                                  // (Fbar W) F_k
            const double t2 = mul_tn<D>(f, wv, r, c);                                      // F_k^T W
            const double acc2 = mul_nn<D>(t2, f, r, c);                                    // (F_k^T W) F_k
            const double gb_new = g - acc2;
            fb = fb_new;
            eb = sym<D>(eb_new, r, c);
            gb = sym<D>(gb_new, r, c);
        }
        // ---- terminal block QT_{k+1} from X[k+1] (augmented.py:78-86)
        const double et = wrapped(cur.x1);
        double px = 0.0;
#pragma unroll
        for (int j = 0; j < n; ++j) px = fma(cst[FC::PF + li * n + j], at(et, j), px);       // (P e)_i
        const double ePe = tree_sum<n, G>(isx ? simt::mul_rn(et, px) : 0.0, 1);
        const double px_x = at(px, (r == n) ? c : r);
        const double qt_e = (r < n) ? ((c < n) ? pf_e : px_x) : ((c < n) ? px_x : (2.0 * (0.5 * ePe) + p.rho_reg));
        // ---- query of horizon t = k+1 (:77-86)
        const double xt = chol_inv<D>(qt_e, r, c, L.act, scratch, p.jitter, p.max_tries, status);
        const double wt = chol_inv<D>(sym<D>(xt + gb, r, c), r, c, L.act, scratch, p.jitter, p.max_tries, status);
        const double t3 = mul_nn<D>(fb, wt, r, c);                                         // Fbar W_t
        const double acc3 = mul_nt<D>(t3, fb, r, c);                                       // (Fbar W_t) Fbar^T
        const double x0 = sym<D>(eb - acc3, r, c);
        const double p0 = chol_inv<D>(x0, r, c, L.act, scratch, p.jitter, p.max_tries, status);
        double dot = 0.0;                                                                  // (P0 z0)_r, z0 = e_n (augmented.py:59)
#pragma unroll
        for (int j = 0; j < D; ++j) dot = fma(at(p0, r * D + j), (j == n) ? 1.0 : 0.0, dot);
        const double part = simt::mul_rn((r == n) ? 1.0 : 0.0, dot);
        const double J = 0.5 * tree_sum<D, G>(part, D);
        if (lane == 0) {
            p.J_out[(size_t)b * p.T_max + k] = J;
            const int t = k + 1;
            if (t >= p.T_min) am.push(J, t);
        }
        ev = et;
        cur = nxt;
    }
    if (lane == 0) {
        p.T_out[b] = am.idx;
        p.Jstar_out[b] = am.best;
        p.status[b] = status;
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// The same sweep as a WARP-SPECIALISED PIPELINE: one problem per CTA of kWspWarps warps.
//
// A horizon step of select_fused_epl_body is three pieces with different dependencies:
//   stage   (E_k, F_k, G_k)            depends on the inputs of step k only
//   prefix  (Ebar, Fbar, Gbar)_k       the loop-carried recursion: needs the prefix of step k-1 and the stage of step k
//   query   J(k+1)                     hangs off the prefix of step k, nothing depends on it
// A single warp executes them back to back (~850 dependent instructions, 4.8 k clocks per step on an otherwise idle SM --
// the 25-trial configurations).  Here three warps compute the stages of the steps k = s (mod 3) ahead of time, one warp runs
// the recursion (one chol_inv and five products per step), three warps take the queries of the steps k = q (mod 3), and the
// blocks travel between them through shared-memory rings (one element per lane, as in the registers) guarded by named
// barriers (producer: fence + bar.arrive, consumer: bar.sync).  Every element goes through the same IEEE operations in the
// same order as in the one-warp body -- the functions below are that body cut at the hand-over points -- so the two kernels
// are bit-identical (asserted on the GPU; the host emulator runs one warp at a time and does not cover this body).
// Role counts (measured on B200, select phase of the Segway 25-trial / cartpole 148-instance HOP-DDP solves, ms; one warp:
// 7.56 / 11.8): 2 + 1 + 3 warps 2.68 / 5.94, 1 + 1 + 3: 2.98 / 6.10, 3 + 1 + 3: 2.34 / 4.98 [default], 4 + 1 + 3 and 3 + 1 + 4:
// 2.70 / 6.03 -- with seven warps the recursion (warp 3) is alone on its SM sub-partition, an eighth warp shares it.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kWspStageWarps = 3, kWspQueryWarps = 3, kWspWarps = kWspStageWarps + 1 + kWspQueryWarps;
constexpr int kWspRingPerStage = 1;
constexpr int kWspStageRing = kWspStageWarps * kWspRingPerStage;   // stage -> prefix ring slots
// named barrier ids (0 is __syncthreads): full / empty per ring slot
constexpr int kBarStageFull = 1, kBarStageEmpty = kBarStageFull + kWspStageRing;
constexpr int kBarPrefixFull = kBarStageEmpty + kWspStageRing, kBarPrefixEmpty = kBarPrefixFull + kWspQueryWarps;
static_assert(kBarPrefixEmpty + kWspQueryWarps <= 16, "sixteen named barriers per CTA");

#ifndef HOP_HOST_EMUL
HOP_DEVICE void bar_arrive(int id) {   // producer / releasing side: this warp's shared-memory accesses first
    __threadfence_block();
    asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory");
}
HOP_DEVICE void bar_wait(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

template <int D>
struct WspSmem {   // doubles; per CTA, after the constants
    static constexpr int DP = (D + 1) & ~1;
    static constexpr int LU = 0;                                           // kWspWarps x (2 D DP): LU fallback scratch per warp
    static constexpr int STAGE = LU + kWspWarps * 2 * D * DP;              // [kWspStageRing][3][32]: e, f, g
    static constexpr int PREFIX = STAGE + kWspStageRing * 3 * 32;          // [kWspQueryWarps][3][32]: eb, fb, gb
    static constexpr int RESULT = PREFIX + kWspQueryWarps * 3 * 32;        // [kWspQueryWarps][4]: best, idx, nan_hit, -; then status words
    static constexpr int SIZE = RESULT + kWspQueryWarps * 4 + kWspWarps + (kWspWarps & 1);
};

// role 0 .. kWspStageWarps-1: stages of the steps k = role (mod kWspStageWarps)
template <int D, int M>
HOP_DEVICE void wsp_stage_role(const FusedArgs& p, int b, int role, double* lu, double* ring, const double* cst, int& status) {
    using FC = FusedConst<D, M>;
    constexpr int n = D - 1;
    constexpr int G = (D <= 4) ? 4 : 8;
    Geo<D> L;
    L.init();
    const int lane = L.lane, r = L.r, c = L.c;
    const bool isx = lane < n;
    const int li = isx ? lane : 0;
    const bool isb = lane < D * M;
    const int rB = isb ? lane / M : 0, cB = isb ? lane % M : 0;
    const bool ism = lane < M * M;
    const int rM = ism ? lane / M : 0, cM = ism ? lane % M : 0;
    const double rinv_e = chol_inv<M>(cst[FC::RS + rM * M + cM], rM, cM, ism, lu, p.jitter, p.max_tries, status);
    const double xg_l = isx ? p.xg[(size_t)b * n + li] : 0.0;
    const bool wrap_l = isx && ((p.wrap_mask >> li) & 1u);
    const double uref_l = (lane < M) ? cst[FC::UREF + lane] : 0.0;
    const double w = p.w[b];
    const double qs_e = (r < n && c < n) ? cst[FC::QS + r * n + c] : 0.0;
    const size_t baseN = (size_t)b * p.N;
    const double* Xb = p.X + (size_t)b * (p.N + 1) * n;
    const double* Ub = p.U + (size_t)b * p.u_stride;
    struct Step { double a, bm, brow[M], ar, u, x0; };
    auto load_step = [&](int k) {
        Step s;
        const bool in = k < p.T_max;
        const double* Ak = p.A + (baseN + k) * n * n;
        const double* Bk = p.Bm + (baseN + k) * n * M;
        s.a = (in && L.act && r < n && c < n) ? Ak[r * n + c] : 0.0;
        s.bm = (in && isb && rB < n) ? Bk[rB * M + cB] : 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j) s.brow[j] = (in && isx) ? Bk[li * M + j] : 0.0;
        s.ar = (in && isx && p.a_resid) ? p.a_resid[(baseN + k) * n + li] : 0.0;
        s.u = (in && lane < M) ? Ub[(size_t)k * M + lane] : 0.0;
        s.x0 = (in && isx) ? Xb[(size_t)k * n + li] : 0.0;
        return s;
    };
    Step cur = load_step(role);
    for (int k = role; k < p.T_max; k += kWspStageWarps) {
        const Step nxt = load_step(k + kWspStageWarps);
        double ev = 0.0;                              // e_k = wrap(X_k - xg)  (augmented.py:28)
        if (isx) {
            ev = cur.x0 - xg_l;
            if (wrap_l) ev = wrap_pi(ev);
        }
        const double du = (lane < M) ? cur.u - uref_l : 0.0;
        double colA = 0.0;
        {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < M; ++j) s = fma(cur.brow[j], at(du, j), s);
            colA = cur.ar - s;
        }
        const double colA_r = at(colA, r);
        const double a_e = (r < n) ? ((c < n) ? cur.a : colA_r) : ((c == n) ? 1.0 : 0.0);
        const double b_e = cur.bm;
        double qe = 0.0, qc = 0.0;
#pragma unroll
        for (int j = 0; j < n; ++j) {
            const double ej = at(ev, j);
            qe = fma(cst[FC::QRAW + li * n + j], ej, qe);
            qc = fma(ej, cst[FC::QRAW + j * n + li], qc);
        }
        const double eQe = tree_sum<n, G>(isx ? simt::mul_rn(qc, ev) : 0.0, 1);
        const double qe_x = at(qe, (r == n) ? c : r);
        const double q_e = (r < n) ? ((c < n) ? qs_e : qe_x) : ((c < n) ? qe_x : (eQe + 2.0 * w + p.rho_reg));
        const double e = chol_inv<D>(q_e, r, c, L.act, lu, p.jitter, p.max_tries, status);
        const double f = mul_nt<D>(e, a_e, r, c);                                          // F_k = E_k A_k^T
        double g;
        {
            const double t = mul_nn<D>(a_e, e, r, c);
            g = mul_nt<D>(t, a_e, r, c);
            double br = 0.0;
#pragma unroll
            for (int l = 0; l < M; ++l) br = fma(at(b_e, rB * M + l), at(rinv_e, l * M + cB), br);
#pragma unroll
            for (int l = 0; l < M; ++l) g = fma(at(br, r * M + l), at(b_e, c * M + l), g);
            g = sym<D>(g, r, c);
        }
        const int slot = k % kWspStageRing;
        if (k >= kWspStageRing) bar_wait(kBarStageEmpty + slot);    // the prefix warp has read step k - kWspStageRing
        double* dst = ring + slot * 96;
        dst[lane] = e; dst[32 + lane] = f; dst[64 + lane] = g;
        bar_arrive(kBarStageFull + slot);
        cur = nxt;
    }
}

// the recursion: one warp, every step.  Only Gbar is loop-carried through the inversion (gb -> W -> gb); the (Ebar, Fbar) update of
// step k needs W_k but nothing of step k+1 needs it before ITS products, so it is deferred by one step and placed in the same
// basic block as the first Gauss-Jordan attempt of step k+1 -- the compiler interleaves the three products with the pivot chain
// (a reciprocal and two shuffle latencies per pivot, otherwise idle issue slots).  The prefix of step k is published one
// inversion later; the queries are off the critical path.  Same operations on the same operands: identical bits.
template <int D, int M>
HOP_DEVICE void wsp_prefix_role(const FusedArgs& p, double* lu, const double* stage_ring, double* prefix_ring, int& status) {
    Geo<D> L;
    L.init();
    const int lane = L.lane, r = L.r, c = L.c;
    double eb = 0.0, fb = 0.0, gb = 0.0;
    double gb_pub = 0.0, wv_prev = 0.0, f_prev = 0.0;       // state of the step whose (Ebar, Fbar) update / publication is pending
    auto publish = [&](int k, double ebv, double fbv, double gbv) {
        const int q = k % kWspQueryWarps;
        if (k >= kWspQueryWarps) bar_wait(kBarPrefixEmpty + q);     // query warp q has read step k - kWspQueryWarps
        double* dst = prefix_ring + q * 96;
        dst[lane] = ebv; dst[32 + lane] = fbv; dst[64 + lane] = gbv;
        bar_arrive(kBarPrefixFull + q);
    };
    for (int k = 0; k < p.T_max; ++k) {
        const int slot = k % kWspStageRing;
        bar_wait(kBarStageFull + slot);
        const double* src = stage_ring + slot * 96;
        const double e = src[lane], f = src[32 + lane], g = src[64 + lane];
        if (k + kWspStageRing < p.T_max) bar_arrive(kBarStageEmpty + slot);
        if (k == 0) {
            eb = e; fb = f; gb = g;
            gb_pub = g;
            continue;                                                // published at the top of step 1 (or after the loop)
        }
        // ---- one basic block: first attempt of W = chol_inv(E_k + Gbar) (:72)  ||  (Ebar, Fbar) update of step k-1 (:73-74)
        const double s = sym<D>(e + gb, r, c);
        double wv = s + ((r == c) ? p.jitter : 0.0);
        const bool first_ok = gj_attempt<D>(wv, r, c);
        if (k >= 2) {
            const double t1 = mul_nn<D>(fb, wv_prev, r, c);          // Fbar W
            const double acc = mul_nt<D>(t1, fb, r, c);              // (Fbar W) Fbar^T
            const double fb_new = mul_nn<D>(t1, f_prev, r, c);       // (Fbar W) F_k
            eb = sym<D>(eb - acc, r, c);
            fb = fb_new;
        }
        if (!first_ok) wv = chol_inv<D>(s, r, c, L.act, lu, p.jitter, p.max_tries, status);   // the ladder, from its first rung
        publish(k - 1, eb, fb, gb_pub);
        // ---- Gbar of step k (:75)
        const double t2 = mul_tn<D>(f, wv, r, c);                    // F_k^T W
        const double acc2 = mul_nn<D>(t2, f, r, c);                  // (F_k^T W) F_k
        gb = sym<D>(g - acc2, r, c);
        gb_pub = gb;
        wv_prev = wv;
        f_prev = f;
    }
    if (p.T_max >= 1) {
        const int k = p.T_max - 1;
        if (k >= 1) {                                                // pending (Ebar, Fbar) update of the last step
            const double t1 = mul_nn<D>(fb, wv_prev, r, c);
            const double acc = mul_nt<D>(t1, fb, r, c);
            const double fb_new = mul_nn<D>(t1, f_prev, r, c);
            eb = sym<D>(eb - acc, r, c);
            fb = fb_new;
        }
        publish(k, eb, fb, gb_pub);
    }
}

// queries of the steps k = q (mod kWspQueryWarps); leaves its running argmin in res[0..2]
template <int D, int M>
HOP_DEVICE void wsp_query_role(const FusedArgs& p, int b, int q, double* lu, const double* prefix_ring, const double* cst, double* res,
                               int& status) {
    using FC = FusedConst<D, M>;
    constexpr int n = D - 1;
    constexpr int G = (D <= 4) ? 4 : 8;
    Geo<D> L;
    L.init();
    const int lane = L.lane, r = L.r, c = L.c;
    const bool isx = lane < n;
    const int li = isx ? lane : 0;
    const double xg_l = isx ? p.xg[(size_t)b * n + li] : 0.0;
    const bool wrap_l = isx && ((p.wrap_mask >> li) & 1u);
    const double pf_e = (r < n && c < n) ? cst[FC::PF + r * n + c] : 0.0;
    const double* Xb = p.X + (size_t)b * (p.N + 1) * n;
    ArgMin am;
    am.init();
    double x1 = (q < p.T_max && isx) ? Xb[(size_t)(q + 1) * n + li] : 0.0;
    for (int k = q; k < p.T_max; k += kWspQueryWarps) {
        const int kn = k + kWspQueryWarps;
        const double x1n = (kn < p.T_max && isx) ? Xb[(size_t)(kn + 1) * n + li] : 0.0;
        // ---- terminal block QT_{k+1} from X[k+1] (augmented.py:78-86): does not need the prefix
        double et = 0.0;
        if (isx) {
            et = x1 - xg_l;
            if (wrap_l) et = wrap_pi(et);
        }
        double px = 0.0;
#pragma unroll
        for (int j = 0; j < n; ++j) px = fma(cst[FC::PF + li * n + j], at(et, j), px);
        const double ePe = tree_sum<n, G>(isx ? simt::mul_rn(et, px) : 0.0, 1);
        const double px_x = at(px, (r == n) ? c : r);
        const double qt_e = (r < n) ? ((c < n) ? pf_e : px_x) : ((c < n) ? px_x : (2.0 * (0.5 * ePe) + p.rho_reg));
        const double xt = chol_inv<D>(qt_e, r, c, L.act, lu, p.jitter, p.max_tries, status);
        bar_wait(kBarPrefixFull + q);
        const double* src = prefix_ring + q * 96;
        const double eb = src[lane], fb = src[32 + lane], gb = src[64 + lane];
        if (kn < p.T_max) bar_arrive(kBarPrefixEmpty + q);
        // ---- query of horizon t = k+1 (:77-86)
        const double wt = chol_inv<D>(sym<D>(xt + gb, r, c), r, c, L.act, lu, p.jitter, p.max_tries, status);
        const double t3 = mul_nn<D>(fb, wt, r, c);
        const double acc3 = mul_nt<D>(t3, fb, r, c);
        const double x0 = sym<D>(eb - acc3, r, c);
        const double p0 = chol_inv<D>(x0, r, c, L.act, lu, p.jitter, p.max_tries, status);
        double dot = 0.0;
#pragma unroll
        for (int j = 0; j < D; ++j) dot = fma(at(p0, r * D + j), (j == n) ? 1.0 : 0.0, dot);
        const double part = simt::mul_rn((r == n) ? 1.0 : 0.0, dot);
        const double J = 0.5 * tree_sum<D, G>(part, D);
        if (lane == 0) {
            p.J_out[(size_t)b * p.T_max + k] = J;
            const int t = k + 1;
            if (t >= p.T_min) am.push(J, t);
        }
        x1 = x1n;
    }
    if (lane == 0) { res[0] = am.best; res[1] = (double)am.idx; res[2] = am.nan_hit ? 1.0 : 0.0; }
}

// np.argmin over the union of the query warps' horizons: the first NaN wins, else the first minimum
HOP_DEVICE void wsp_merge(ArgMin& a, double best, int idx, bool nan_hit) {
    if (idx == 0) return;
    if (a.idx == 0) { a.best = best; a.idx = idx; a.nan_hit = nan_hit; return; }
    if (a.nan_hit || nan_hit) {
        if (nan_hit && (!a.nan_hit || idx < a.idx)) { a.best = best; a.idx = idx; a.nan_hit = true; }
        return;
    }
    if (best < a.best || (best == a.best && idx < a.idx)) { a.best = best; a.idx = idx; }
}
#endif  // !HOP_HOST_EMUL

}}  // namespace hop::epl
