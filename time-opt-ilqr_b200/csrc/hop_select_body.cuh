// hop_select_body.cuh -- per-problem kernel bodies built on hop_select_core.cuh.
//
//   select_generic_body : LQR-boundary form, inputs are the augmented blocks themselves
//                         (drop-in for horizon_selection.py:36-86 propagator_all_Jt_aug + solver.py:522 argmin)
//   select_fused_body   : fused form, inputs are the raw linearisation (A_k, B_k, a_k) and the nominal
//                         trajectory (X, U); the homogeneous embedding of augmented.py:10-87
//                         (build_augmented_sequence_QR + build_terminal_aug_list) is built in-kernel,
//                         so the (n+1)^2 blocks never exist in HBM.
#pragma once
#include "hop_select_core.cuh"

namespace hop {

struct SelectArgs {
    int B, N, T_min, T_max;
    double jitter;
    int max_tries;
    const double *A_aug, *B_aug, *Q_aug, *R_inv, *z0, *QT;
    long rinv_step_stride;      // 0: one R^-1 [m][m] per instance; m*m: R_inv is [B][N][m][m] (R_list varies with k)
    const double* w_explicit;   // optional [B]: argmin is taken over J(t) + w t (S2 workload)
    double* J_out;              // [B][T_max]
    int* T_out;                 // [B]
    double* Jstar_out;          // [B]
    int* status;                // [B]
    // pre-inverted input blocks (hop_select.cu: k_preinvert + k_select_generic_pipe<.., PRE>), else null:
    // E_pre[b][k] = chol_inv(Q_aug[b][k]), X_pre[b][k] = chol_inv(QT[b][k]), pre_bad[b] != 0 => some inversion needs the ladder
    const double *E_pre, *X_pre;
    const int* pre_bad;
    // test hook (hop_test_set_generic_diag): non-zero => the pipelined LQR-boundary kernel inverts DIAGONAL
    // input blocks by the Gauss-Jordan sweep like any other block instead of element-wise (identical bits either way)
    int no_diag_fastpath;
};

struct FusedArgs {
    int B, N, T_min, T_max;
    double jitter;
    int max_tries;
    const double *A, *Bm, *a_resid, *X, *U;   // [B][N][n][n], [B][N][n][m], [B][N][n] or null, [B][N+1][n], [B][N][m]
    long u_stride;                             // doubles between consecutive instances' U (N*m, or 0 = shared)
    const double *xg, *w;                      // [B][n], [B]
    const double *u_ref, *Q, *R, *Qf;          // shared case constants: [m], [n][n], [m][m], [n][n]
    unsigned wrap_mask;
    double q_reg, rho_reg;
    int mode;                                  // HOP_MODE_EXACT / HOP_MODE_FAST / HOP_MODE_GJ
    const int* skip;                           // optional [B]: non-zero => instance is left untouched
    double* J_out;
    int* T_out;
    double* Jstar_out;
    int* status;
};

// utils.py:127-128: (a + pi) % (2 pi) - pi with Python's floored modulo.  For s = a + pi in (-2 pi, 4 pi) the floored modulo
// is s, s + 2 pi or s - 2 pi -- exactly what fmod and the sign fix-up return (fmod is exact, the subtraction is exact by
// Sterbenz) -- so those ranges skip the library call: same bits, a shorter dependent chain in every roll-out / sweep step.
HOP_DEVICE double wrap_pi(double a) {
    const double pi = 3.141592653589793, two_pi = 6.283185307179586;
    const double s = a + pi;
    if (s >= 0.0 && s < two_pi) return s - pi;                        // (fmod(s, 2 pi) = s; -0.0 and +0.0 both give 0.0 - pi below)
    if (s >= two_pi && s < 2.0 * two_pi) return (s - two_pi) - pi;
    if (s < 0.0 && s > -two_pi) return (s + two_pi) - pi;
    double r = fmod(s, two_pi);
    if (r != 0.0) {
        if (r < 0.0) r += two_pi;
    } else {
        r = 0.0;
    }
    return r - pi;
}

template <int D, int M, int G>
HOP_DEVICE void select_generic_body(const SelectArgs& p, int b_raw, double* sm) {
    using Ge = Geo<D, M, G>;
    constexpr int DP = Ge::DP;
    const int lane = simt::lane_id();
    const int r = lane % G;
    const bool act = r < D;
    const int rr = act ? r : 0;
    const bool valid = b_raw < p.B;
    const int b = valid ? b_raw : p.B - 1;

    for (int i = r; i < Ge::SLAB; i += G) sm[i] = 0.0;
    simt::sync();
    const size_t rinv_inst = (size_t)(p.rinv_step_stride ? p.N : 1) * M * M;
    for (int i = r; i < M * M; i += G) sm[Ge::SR + (i / M) * Ge::MP + (i % M)] = p.R_inv[(size_t)b * rinv_inst + i];
    if (act) sm[Ge::Z0 + r] = p.z0[(size_t)b * D + r];

    Prefix<D> P;
#pragma unroll
    for (int j = 0; j < D; ++j) { P.eb[j] = 0.0; P.fb[j] = 0.0; P.gb[j] = 0.0; }
    int status = 0;
    ArgMin am;
    am.init();
    const double wexp = p.w_explicit ? p.w_explicit[b] : 0.0;
    const size_t base = (size_t)b * p.N;
    double* SA = sm + Ge::SA; double* SX = sm + Ge::SX; double* SQ = sm + Ge::SQ; double* SB = sm + Ge::SB;

    // The blocks of step k+1 are loaded into registers while step k computes (every lane owns the elements
    // i = r, r + G, ... of each block) and moved to the slab at the top of step k+1: the global-load latency, which
    // was exposed once per step (ncu: long_scoreboard 2.2 per issue, the top stall), hides behind the sweep.
    constexpr int PA = (D * D + G - 1) / G, PB = (D * M + G - 1) / G, PR = (M * M + G - 1) / G;
    struct Fetch { double a[PA], q[PA], t[PA], b[PB], ri[PR]; };
    auto fetch = [&](int k, Fetch& f) {
        const double* Ak = p.A_aug + (base + k) * D * D;
        const double* Qk = p.Q_aug + (base + k) * D * D;
        const double* Tk = p.QT + (base + k) * D * D;
        const double* Bk = p.B_aug + (base + k) * D * M;
#pragma unroll
        for (int u = 0; u < PA; ++u) {
            const int i = r + u * G;
            const bool in = i < D * D;
            f.a[u] = in ? Ak[i] : 0.0; f.q[u] = in ? Qk[i] : 0.0; f.t[u] = in ? Tk[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < PB; ++u) { const int i = r + u * G; f.b[u] = (i < D * M) ? Bk[i] : 0.0; }
        if (p.rinv_step_stride) {
#pragma unroll
            for (int u = 0; u < PR; ++u) {
                const int i = r + u * G;
                f.ri[u] = (i < M * M) ? p.R_inv[(size_t)b * rinv_inst + (size_t)k * p.rinv_step_stride + i] : 0.0;
            }
        }
    };
    Fetch cur;
    fetch(0, cur);
    for (int k = 0; k < p.T_max; ++k) {
        simt::sync();
#pragma unroll
        for (int u = 0; u < PA; ++u) {
            const int i = r + u * G;
            if (i < D * D) {
                const int row = i / D, col = i % D;
                SA[col * DP + row] = cur.a[u];
                SX[row * DP + col] = cur.q[u];
                SQ[row * DP + col] = cur.t[u];
            }
        }
#pragma unroll
        for (int u = 0; u < PB; ++u) { const int i = r + u * G; if (i < D * M) SB[(i % M) * DP + (i / M)] = cur.b[u]; }
        if (p.rinv_step_stride) {
#pragma unroll
            for (int u = 0; u < PR; ++u) { const int i = r + u * G; if (i < M * M) sm[Ge::SR + (i / M) * Ge::MP + (i % M)] = cur.ri[u]; }
        }
        if (k + 1 < p.T_max) fetch(k + 1, cur);
        simt::sync();
        {
            double q[D];
#pragma unroll
            for (int j = 0; j < D; ++j) q[j] = 0.5 * (SX[rr * DP + j] + SX[j * DP + rr]);
            stage_prefix_step<D, M, G>(k, P, q, sm, r, act, lane, p.jitter, p.max_tries, status);
        }
        double J;
        {
            double qt[D];
#pragma unroll
            for (int j = 0; j < D; ++j) qt[j] = 0.5 * (SQ[rr * DP + j] + SQ[j * DP + rr]);
            J = query_step<D, M, G>(P, qt, sm, r, act, lane, p.jitter, p.max_tries, status);
        }
        if (r == 0 && valid) {
            p.J_out[(size_t)b * p.T_max + k] = J;
            const int t = k + 1;
            if (t >= p.T_min) am.push(simt::add_rn(J, simt::mul_rn(wexp, (double)t)), t);   // J + w t as numpy: two roundings
        }
    }
    if (r == 0 && valid) {
        p.T_out[b] = am.idx;
        p.Jstar_out[b] = am.best;
        p.status[b] = status;
    }
}

// Case constants shared by the whole CTA (fused form): Qs = sym(Q) + q_reg I, Qraw, P = sym(Qf), u_ref.
template <int D, int M>
struct FusedConst {
    static constexpr int n = D - 1;
    static constexpr int QS = 0, QRAW = n * n, PF = 2 * n * n, UREF = 3 * n * n, RS = UREF + ((M + 1) & ~1);
    static constexpr int SIZE = RS + M * M + ((M * M) & 1);
};

// Fill the CTA constant block; `tid`/`nthr` enumerate the cooperating threads.
template <int D, int M>
HOP_DEVICE void fused_const_fill(const FusedArgs& p, double* cst, int tid, int nthr) {
    using FC = FusedConst<D, M>;
    constexpr int n = D - 1;
    for (int i = tid; i < n * n; i += nthr) {
        const int a = i / n, c = i % n;
        cst[FC::QS + i] = 0.5 * (p.Q[a * n + c] + p.Q[c * n + a]) + (a == c ? p.q_reg : 0.0);   // augmented.py:32
        cst[FC::QRAW + i] = p.Q[i];
        cst[FC::PF + i] = 0.5 * (p.Qf[a * n + c] + p.Qf[c * n + a]);                           // augmented.py:76
    }
    for (int i = tid; i < M; i += nthr) cst[FC::UREF + i] = p.u_ref[i];
    for (int i = tid; i < M * M; i += nthr) {
        const int a = i / M, c = i % M;
        cst[FC::RS + i] = 0.5 * (p.R[a * M + c] + p.R[c * M + a]);                              // augmented.py:23
    }
}

template <int D, int M, int G>
HOP_DEVICE void select_fused_body(const FusedArgs& p, int b_raw, double* sm, const double* cst) {
    using Ge = Geo<D, M, G>;
    using FC = FusedConst<D, M>;
    constexpr int DP = Ge::DP;
    constexpr int n = D - 1;
    static_assert(M <= D, "control dimension must not exceed the augmented dimension");
    const int lane = simt::lane_id();
    const int r = lane % G;
    const bool act = r < D;
    const bool isx = r < n;          // lane owns a state row
    const int rr = act ? r : 0;
    const int rx = isx ? r : 0;
    const int b = (b_raw < p.B) ? b_raw : p.B - 1;
    const bool valid = (b_raw < p.B) && !(p.skip && p.skip[b]);

    for (int i = r; i < Ge::SLAB; i += G) sm[i] = 0.0;
    simt::sync();
    double* SA = sm + Ge::SA; double* SB = sm + Ge::SB; double* SR = sm + Ge::SR;
    double* V0 = sm + Ge::VEC; double* V1 = V0 + DP; double* V2 = V1 + DP; double* V3 = V2 + DP;
    int status = 0;

    // R_inv = chol_inv(sym(R))  (augmented.py:23), rows on lanes r < M
    {
        double rs[M], ri[M];
#pragma unroll
        for (int j = 0; j < M; ++j) rs[j] = cst[FC::RS + ((r < M) ? r : 0) * M + j];
        chol_inv_rows<M, G, Ge::MP>(rs, ri, r, r < M, lane, sm + Ge::ROW, sm + Ge::SX, sm + Ge::SY, p.jitter,
                                    p.max_tries, status);
        simt::sync();
        if (r < M) st_row<M, Ge::MP>(SR, r, ri);
    }
    if (act) sm[Ge::Z0 + r] = (r == n) ? 1.0 : 0.0;   // augmented.py:59
    if (isx) V0[r] = p.xg[(size_t)b * n + r];
    const double xg_r = isx ? p.xg[(size_t)b * n + r] : 0.0;
    const bool wrap_r = isx && ((p.wrap_mask >> r) & 1u);
    const double w = p.w[b];

    Prefix<D> P;
#pragma unroll
    for (int j = 0; j < D; ++j) { P.eb[j] = 0.0; P.fb[j] = 0.0; P.gb[j] = 0.0; }
    ArgMin am;
    am.init();
    const size_t baseN = (size_t)b * p.N;
    const size_t baseX = (size_t)b * (p.N + 1);

    // Inputs of step k+1 are loaded into registers while step k computes (lane r owns the elements i = r, r + G, ... of
    // A_k and B_k, and component r of U_k, X_k, X_{k+1}, a_k) and moved to the slab at the top of step k+1, so the
    // global-load latency hides behind the sweep instead of being exposed once per step.
    constexpr int PA = (n * n + G - 1) / G, PB = (n * M + G - 1) / G;
    struct Fetch { double a[PA], b[PB], u, x0, x1, ar; };
    auto fetch = [&](int k, Fetch& f) {
        const double* Ak = p.A + (baseN + k) * n * n;
        const double* Bk = p.Bm + (baseN + k) * n * M;
#pragma unroll
        for (int q = 0; q < PA; ++q) { const int i = r + q * G; f.a[q] = (i < n * n) ? Ak[i] : 0.0; }
#pragma unroll
        for (int q = 0; q < PB; ++q) { const int i = r + q * G; f.b[q] = (i < n * M) ? Bk[i] : 0.0; }
        f.u = (r < M) ? p.U[(size_t)b * p.u_stride + (size_t)k * M + r] : 0.0;
        f.x0 = isx ? p.X[(baseX + k) * n + r] : 0.0;
        f.x1 = isx ? p.X[(baseX + k + 1) * n + r] : 0.0;
        f.ar = (isx && p.a_resid) ? p.a_resid[(baseN + k) * n + r] : 0.0;
    };
    Fetch cur;
    fetch(0, cur);
    for (int k = 0; k < p.T_max; ++k) {
        simt::sync();
        // ---- A_aug^T, B_aug^T (augmented.py:50-56)
#pragma unroll
        for (int q = 0; q < PA; ++q) { const int i = r + q * G; if (i < n * n) SA[(i % n) * DP + (i / n)] = cur.a[q]; }
#pragma unroll
        for (int q = 0; q < PB; ++q) { const int i = r + q * G; if (i < n * M) SB[(i % M) * DP + (i / M)] = cur.b[q]; }
        if (r < M) V3[r] = cur.u - cst[FC::UREF + r];   // du
        double ev = 0.0;
        if (isx) {
            ev = cur.x0 - xg_r;                                                      // e = wrap(X_k - xg)
            if (wrap_r) ev = wrap_pi(ev);
        }
        if (act) V1[r] = ev;
        const double ak = cur.ar;
        const double x_next = cur.x1;
        if (k + 1 < p.T_max) fetch(k + 1, cur);
        simt::sync();
        if (isx) {
            double s = 0.0;
#pragma unroll
            for (int c = 0; c < M; ++c) s = fma(SB[c * DP + r], V3[c], s);          // (B_k du)_r
            SA[n * DP + r] = ak - s;                                                // A_aug[r][n] = a_k - B_k du
            SA[r * DP + n] = 0.0;                                                   // A_aug[n][r] = 0
        } else if (r == n) {
            SA[n * DP + n] = 1.0;
#pragma unroll
            for (int c = 0; c < M; ++c) SB[c * DP + n] = 0.0;
        }
        // ---- Q_aug row (augmented.py:31-48).  sym() of that block is the identity on these values.
        double qe = 0.0, qc = 0.0;
#pragma unroll
        for (int j = 0; j < n; ++j) {
            qe = fma(cst[FC::QRAW + rx * n + j], V1[j], qe);                        // (Q e)_r
            qc = fma(V1[j], cst[FC::QRAW + j * n + rx], qc);                        // (e^T Q)_r
        }
        const double eQe = group_sum<G>(isx ? qc * ev : 0.0);
        if (isx) V2[r] = qe;
        simt::sync();
        {
            double q[D];
#pragma unroll
            for (int j = 0; j < n; ++j) q[j] = isx ? cst[FC::QS + rx * n + j] : V2[j];
            q[n] = isx ? qe : (eQe + 2.0 * w + p.rho_reg);
            stage_prefix_step<D, M, G>(k, P, q, sm, r, act, lane, p.jitter, p.max_tries, status);
        }
        // ---- terminal block QT_{k+1} from X[k+1] (augmented.py:78-86)
        simt::sync();
        double et = 0.0;
        if (isx) {
            et = x_next - xg_r;
            if (wrap_r) et = wrap_pi(et);
        }
        if (act) V1[r] = et;
        simt::sync();
        double px = 0.0;
#pragma unroll
        for (int j = 0; j < n; ++j) px = fma(cst[FC::PF + rx * n + j], V1[j], px);  // (P e)_r
        const double ePe = group_sum<G>(isx ? et * px : 0.0);
        if (isx) V2[r] = px;
        simt::sync();
        double J;
        {
            double qt[D];
#pragma unroll
            for (int j = 0; j < n; ++j) qt[j] = isx ? cst[FC::PF + rx * n + j] : V2[j];
            qt[n] = isx ? px : (2.0 * (0.5 * ePe) + p.rho_reg);
            J = query_step<D, M, G>(P, qt, sm, r, act, lane, p.jitter, p.max_tries, status);
        }
        if (r == 0 && valid) {
            p.J_out[(size_t)b * p.T_max + k] = J;
            const int t = k + 1;
            if (t >= p.T_min) am.push(J, t);
        }
    }
    (void)rr;
    if (r == 0 && valid) {
        p.T_out[b] = am.idx;
        p.Jstar_out[b] = am.best;
        p.status[b] = status;
    }
}

}  // namespace hop
