// hop_traj.cu -- batched nominal rollout and finite-difference linearisation.
//
//   k_rollout   : solver.py:42-62   one thread per problem, sequential in k
//   k_linearize : linearization.py:216-262 (forward) / :177-211 (central)
//                 one thread per (problem, step, perturbed coordinate); the n+m threads of a
//                 (problem, step) pair are adjacent, so each row of A_k / B_k is written coalesced.
#include "hop_common.cuh"
#include "hop_dynamics.cuh"
#include "../../include/hop_b200.h"

namespace hop {

// quadrotor finite-difference kernel: 0 thread-per-step (default), 2 generic (test hook; identical bits)
int g_linearize_variant = 0;

template <int SYS>
__global__ void k_rollout(int B, DynParams prm, int N, const double* __restrict__ x0, const double* __restrict__ U,
                          long ustride, double max_norm, double* __restrict__ X) {
    constexpr int n = SysDims<SYS>::n, m = SysDims<SYS>::m;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double x[n], xn[n], u[m];
#pragma unroll
    for (int i = 0; i < n; ++i) x[i] = x0[(size_t)b * n + i];
    double* Xb = X + (size_t)b * (N + 1) * n;
#pragma unroll
    for (int i = 0; i < n; ++i) Xb[i] = x[i];
    const double* Ub = U + (size_t)b * ustride;
    bool dead = false;
    for (int k = 0; k < N; ++k) {
        if (!dead) {
#pragma unroll
            for (int i = 0; i < m; ++i) u[i] = Ub[(size_t)k * m + i];
            dynamics<SYS>(prm.p, x, u, xn);
            double ss = 0.0;
            bool fin = true;
#pragma unroll
            for (int i = 0; i < n; ++i) { fin = fin && isfinite(xn[i]); ss = add(ss, mul(xn[i], xn[i])); }
            if (!fin || sqrt(ss) > max_norm) dead = true;   // solver.py:57-59: NaN-fill the remainder
        }
#pragma unroll
        for (int i = 0; i < n; ++i) {
            x[i] = dead ? nan("") : xn[i];
            Xb[(size_t)(k + 1) * n + i] = x[i];
        }
    }
}

template <int SYS>
__global__ void k_linearize(int B, DynParams prm, int N, const double* __restrict__ X, const double* __restrict__ U,
                            long ustride, int central, double epsx, double epsu, double relx, double relu,
                            const int* __restrict__ skip, double* __restrict__ A, double* __restrict__ Bm) {
    constexpr int n = SysDims<SYS>::n, m = SysDims<SYS>::m, P = n + m;
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)B * N * P;
    if (gid >= total) return;
    const int c = (int)(gid % P);            // perturbed coordinate: state c < n, else control c - n
    const size_t bk = gid / P;
    const int k = (int)(bk % N);
    const size_t b = bk / N;
    if (skip && skip[b]) return;
    double x[n], u[m], f0[n], fp[n], fm[n];
    const double* xs = X + (b * (N + 1) + k) * n;
    const double* us = U + b * ustride + (size_t)k * m;
#pragma unroll
    for (int i = 0; i < n; ++i) x[i] = xs[i];
#pragma unroll
    for (int i = 0; i < m; ++i) u[i] = us[i];
    double h = 0.0, base = 0.0;
    // h = max(eps, rel * max(1, |v|))  (linearization.py:253,257)
#pragma unroll
    for (int i = 0; i < n; ++i) if (i == c) { base = x[i]; h = fmax(epsx, mul(relx, fmax(1.0, fabs(x[i])))); }
#pragma unroll
    for (int i = 0; i < m; ++i) if (i + n == c) { base = u[i]; h = fmax(epsu, mul(relu, fmax(1.0, fabs(u[i])))); }
    bool nanout = false;
    if (!central) {
        dynamics<SYS>(prm.p, x, u, f0);
        bool fin = true;
#pragma unroll
        for (int i = 0; i < n; ++i) fin = fin && isfinite(f0[i]);
        nanout = !fin;                        // linearization.py:243-248
    }
    const double vp = add(base, h), vm = sub(base, h);
#pragma unroll
    for (int i = 0; i < n; ++i) if (i == c) x[i] = vp;
#pragma unroll
    for (int i = 0; i < m; ++i) if (i + n == c) u[i] = vp;
    dynamics<SYS>(prm.p, x, u, fp);
    double col[n];
    if (central) {
#pragma unroll
        for (int i = 0; i < n; ++i) if (i == c) x[i] = vm;
#pragma unroll
        for (int i = 0; i < m; ++i) if (i + n == c) u[i] = vm;
        dynamics<SYS>(prm.p, x, u, fm);
        const double den = mul(2.0, h);
#pragma unroll
        for (int i = 0; i < n; ++i) col[i] = sub(fp[i], fm[i]) / den;
    } else {
#pragma unroll
        for (int i = 0; i < n; ++i) col[i] = nanout ? nan("") : sub(fp[i], f0[i]) / h;
    }
    if (c < n) {
        double* Ak = A + bk * n * n;
#pragma unroll
        for (int i = 0; i < n; ++i) Ak[i * n + c] = col[i];
    } else {
        double* Bk = Bm + bk * n * m;
#pragma unroll
        for (int i = 0; i < n; ++i) Bk[i * m + (c - n)] = col[i];
    }
}

// out-of-line copy of the full dynamics for cold paths
__device__ __noinline__ void quad_dynamics_cold(const double* p, const double* x, const double* u, double* xn) {
    dynamics<2>(p, x, u, xn);
}

// ---- quadrotor forward differences, ONE THREAD PER (problem, step) -----------------------------------------
// A lane-per-column mapping (16 lanes per (problem, step), lane c perturbs coordinate c) spent 1584 warp-instructions
// per 32 lanes (ncu: 80 % of them selects / moves / integer tests that exist only because the perturbed coordinate is
// a run-time lane index).  Here the 16 perturbations are a compile-time unrolled loop in one thread, so that
//   * the perturbed evaluations share every sub-expression that does not depend on the perturbed coordinate
//     (same operations on the same values -> same bits; the compiler's CSE does the sharing),
//   * entries (i, c) whose output F_i does not depend on coordinate c are written as the exact 0.0 the reference
//     obtains from (F_i - F_i) / h  (quad_affects below is the dependency structure of systems.py:170-210),
//   * A_k and B_k are stored as full 32-byte sectors (four columns of a row at a time),
//   * the 12 quotients (fp - f0) / h of a column share one reciprocal: q0 = d * r, q = q0 + fma(-q0, h, d) * r, which
//     is the correctly rounded quotient for r = RN(1/h) (Markstein), i.e. what the division returns.
// f0 = F(X_k, U_k) is read from X[k+1] when the caller guarantees a consistent rollout (f0_from_x: the rollout /
// line-search kernels produced X with this very dynamics function), evaluated otherwise; NaN / guard semantics as in
// k_linearize.  Bit-identical to k_linearize<2> (tests/test_gpu_parity.py compares them on random states).
// bit i of quad_affects(c): F_i depends on coordinate c of (x, u)
__host__ __device__ constexpr unsigned quad_affects(int c) {
    return c == 0 ? 0x001u : c == 1 ? 0x002u : c == 2 ? 0x004u          // x, y, z        -> their own row
         : c == 3 ? 0x009u : c == 4 ? 0x012u : c == 5 ? 0x024u          // vx, vy, vz     -> position and velocity rows
         : c == 6 ? 0x1f8u : c == 7 ? 0x1f8u : c == 8 ? 0x118u          // roll, pitch -> v and Euler-rate rows; yaw -> vx, vy, yaw
         : c == 9 ? 0xe40u : c == 10 ? 0xfc0u : c == 11 ? 0xfc0u        // wp -> {roll rate, w}; wq, wr -> Euler rates and w
         : c == 12 ? 0x038u : c == 13 ? 0x200u : c == 14 ? 0x400u : 0x800u;   // thrust -> v rows; torques -> their w row
}

// one perturbed evaluation F(x + dv e_C, u) (or u + dv e_{C-n}); *bad = the reference's guards returned NaN(12)
template <int C>
__device__ __forceinline__ void quad_fd_eval(const double* p, const double* x0v, const double* u0v, const QuadTrig& Tb, double vp,
                                             double dist, double ss_sqrt, double* fp, bool* bad_out) {
    constexpr int n = 12, m = 4;
    double x[n], u[m];
#pragma unroll
    for (int i = 0; i < n; ++i) x[i] = x0v[i];
#pragma unroll
    for (int i = 0; i < m; ++i) u[i] = u0v[i];
    if (C < n) x[C < n ? C : 0] = vp; else u[C >= n ? C - n : 0] = vp;
    QuadTrig T = Tb;
    if (C == 6) sincos(vp, &T.sph, &T.cph);
    if (C == 7) { sincos(vp, &T.sth, &T.cth); T.tth = tan(vp); }
    if (C == 8) sincos(vp, &T.sps, &T.cps);
    // guards (systems.py:175-191).  The norm test can only change if the unperturbed norm is within |dv| of the limit:
    // ||x + dv e_c|| <= ||x|| + |dv|.  Otherwise evaluate it exactly (cold).
    bool bad = !isfinite(vp);
    if (C < n && ss_sqrt + 1.0000001 * dist + 1e-9 * ss_sqrt >= p[13]) bad = bad || quad_guard(p, x, u);
    bad = bad || (fabs(T.cth) < p[11]);                                        // nominal pitch unless C == 7
    bad = bad || (fabs(x[9]) > p[12]) || (fabs(x[10]) > p[12]) || (fabs(x[11]) > p[12]);   // nominal rates except coordinate C
    quad_core(p, x, u, T, fp);
    *bad_out = bad;
}

// column C of [A_k | B_k]: forward (fp - f0) / h or central (fp - fm) / (2 h) differences (linearization.py:177-262)
template <int C, bool CENTRAL>
__device__ __forceinline__ void quad_fd_column(const double* p, const double* x0v, const double* u0v, const QuadTrig& Tb,
                                               const double* f0, bool nanout, double ss_sqrt, double epsx, double epsu,
                                               double relx, double relu, double* col) {
    constexpr int n = 12;
    constexpr unsigned aff = quad_affects(C);
    const double base = C < n ? x0v[C < n ? C : 0] : u0v[C >= n ? C - n : 0];
    const double h = C < n ? fmax(epsx, mul(relx, fmax(1.0, fabs(base)))) : fmax(epsu, mul(relu, fmax(1.0, fabs(base))));
    double fp[n], fm[n];
    bool bad = false, badm = false;
    quad_fd_eval<C>(p, x0v, u0v, Tb, add(base, h), h, ss_sqrt, fp, &bad);
    if (CENTRAL) quad_fd_eval<C>(p, x0v, u0v, Tb, sub(base, h), h, ss_sqrt, fm, &badm);
    const double den = CENTRAL ? mul(2.0, h) : h;
    const double rh = 1.0 / den;
#pragma unroll
    for (int i = 0; i < n; ++i) {
        double q = 0.0;
        if ((aff >> i) & 1u) {
            const double d = sub(fp[i], CENTRAL ? fm[i] : f0[i]);
            const double q0 = mul(d, rh);
            q = fma(fma(-q0, den, d), rh, q0);
        }
        col[i] = (nanout || bad || badm) ? nan("") : q;
    }
}

// MINB: CTAs per SM the register allocation is bounded for (3 -> 168 registers; 4 -> 128 with ~130 B of spills was slower:
// profiles/r1_experiments_overlap.txt)
template <bool CENTRAL, int MINB = 3>
__global__ void __launch_bounds__(128, MINB) k_linearize_quad_row(int B, DynParams prm, int N, const double* __restrict__ X,
                                                            const double* __restrict__ U, long ustride, double epsx, double epsu,
                                                            double relx, double relu, int f0_from_x, const int* __restrict__ skip,
                                                            double* __restrict__ A, double* __restrict__ Bm) {
    constexpr int n = 12, m = 4;
    const size_t total = (size_t)B * N;
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = gid < total;
    const size_t bk = live ? gid : total - 1;     // dead lanes shadow the last step: the pair exchange below needs every lane
    const int k = (int)(bk % N);
    const size_t b = bk / N;
    const bool active = live && !(skip && skip[b]);
    if (__all_sync(0xffffffffu, !active)) return;
    double x[n], u[m], f0[n];
    const double* xs = X + (b * (N + 1) + k) * n;
    const double* us = U + b * ustride + (size_t)k * m;
#pragma unroll
    for (int i = 0; i < n; ++i) x[i] = xs[i];
#pragma unroll
    for (int i = 0; i < m; ++i) u[i] = us[i];
    bool nanout = false;
    if (!CENTRAL) {
        bool have_f0 = false;
        if (f0_from_x) {
            bool fin = true, finx = true;
#pragma unroll
            for (int i = 0; i < n; ++i) { f0[i] = xs[n + i]; fin = fin && isfinite(f0[i]); finx = finx && isfinite(x[i]); }
            // X[k+1] non-finite although X[k] is finite: either F is non-finite there or the rollout cut the trajectory
            // on its norm test (solver.py:57-59) -- only F itself can tell, so recompute
            have_f0 = fin || !finx;
        }
        if (!have_f0) {                     // cold; through copies so that x, u, f0 themselves never live in local memory
            double xc[n], uc[m], fc[n];
#pragma unroll
            for (int i = 0; i < n; ++i) xc[i] = x[i];
#pragma unroll
            for (int i = 0; i < m; ++i) uc[i] = u[i];
            quad_dynamics_cold(prm.p, xc, uc, fc);
#pragma unroll
            for (int i = 0; i < n; ++i) f0[i] = fc[i];
        }
#pragma unroll
        for (int i = 0; i < n; ++i) nanout = nanout || !isfinite(f0[i]);      // linearization.py:243-248
    } else {
        // central differences never evaluate F at the nominal point; a non-finite nominal makes every evaluation NaN
#pragma unroll
        for (int i = 0; i < n; ++i) { f0[i] = 0.0; nanout = nanout || !isfinite(x[i]); }
#pragma unroll
        for (int i = 0; i < m; ++i) nanout = nanout || !isfinite(u[i]);
    }
    // unperturbed trigonometry and norm, shared by all 16 columns
    QuadTrig T;
    sincos(x[6], &T.sph, &T.cph);
    sincos(x[7], &T.sth, &T.cth);
    sincos(x[8], &T.sps, &T.cps);
    T.tth = tan(x[7]);
    double ss = 0.0;
#pragma unroll
    for (int i = 0; i < n; ++i) ss = add(ss, mul(x[i], x[i]));
    const double nrm = sqrt(ss);
    // Stores: a thread owns 32 contiguous bytes per (row, 4-column group).  Two half-sector stores per thread make the
    // L2 read-fill every sector (ncu: 19 GB written + 6.5 GB read for 12.9 GB of output); instead neighbouring lanes
    // swap halves so that every store instruction writes FULL 32-byte sectors (lane pair = one sector).
    const bool odd = (threadIdx.x & 1) != 0;
    const bool pair_active = __shfl_xor_sync(0xffffffffu, active ? 1 : 0, 1) != 0;
    char* Aown = reinterpret_cast<char*>(A + bk * n * n);
    char* Bown = reinterpret_cast<char*>(Bm + bk * n * m);
    const size_t bk_pair = (size_t)__shfl_xor_sync(0xffffffffu, (unsigned long long)bk, 1);   // (a dead lane shadows total - 1)
    char* Apair = reinterpret_cast<char*>(A + bk_pair * n * n);
    char* Bpair = reinterpret_cast<char*>(Bm + bk_pair * n * m);
#define HOP_FD4(C0, OWN, PAIR, LDB)                                                                                       \
    {                                                                                                                     \
        double c0[n], c1[n], c2[n], c3[n];                                                                                \
        quad_fd_column<C0 + 0, CENTRAL>(prm.p, x, u, T, f0, nanout, nrm, epsx, epsu, relx, relu, c0);                              \
        quad_fd_column<C0 + 1, CENTRAL>(prm.p, x, u, T, f0, nanout, nrm, epsx, epsu, relx, relu, c1);                              \
        quad_fd_column<C0 + 2, CENTRAL>(prm.p, x, u, T, f0, nanout, nrm, epsx, epsu, relx, relu, c2);                              \
        quad_fd_column<C0 + 3, CENTRAL>(prm.p, x, u, T, f0, nanout, nrm, epsx, epsu, relx, relu, c3);                              \
        _Pragma("unroll") for (int i = 0; i < n; ++i) {                                                                   \
            /* even lane keeps (c0,c1) and sends (c2,c3); odd lane keeps (c2,c3) and sends (c0,c1) */                     \
            const double s0 = odd ? c0[i] : c2[i], s1 = odd ? c1[i] : c3[i];                                              \
            const double r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);              \
            /* sector of the even lane's step: even writes its low half, odd writes the even lane's high half */          \
            if (odd ? pair_active : active)                                                                               \
                *reinterpret_cast<double2*>((odd ? (PAIR) : (OWN)) + i * (LDB) + (odd ? 16 : 0)) =                         \
                    odd ? make_double2(r0, r1) : make_double2(c0[i], c1[i]);                                              \
            /* sector of the odd lane's step */                                                                           \
            if (odd ? active : pair_active)                                                                               \
                *reinterpret_cast<double2*>((odd ? (OWN) : (PAIR)) + i * (LDB) + (odd ? 16 : 0)) =                         \
                    odd ? make_double2(c2[i], c3[i]) : make_double2(r0, r1);                                              \
        }                                                                                                                 \
    }
    HOP_FD4(0, Aown + 0, Apair + 0, n * 8)
    HOP_FD4(4, Aown + 32, Apair + 32, n * 8)
    HOP_FD4(8, Aown + 64, Apair + 64, n * 8)
    HOP_FD4(12, Bown, Bpair, m * 8)
#undef HOP_FD4
}

int dispatch_rollout(int B, int sys, const double* params_host, int N, const double* x0, const double* U, long ustride,
                     double max_norm, double* X, cudaStream_t st) {
    const DynParams prm = dyn_params(params_host);
    return with_system(sys, "hop_rollout_f64", [&](auto s) {
        const int threads = 128;
        k_rollout<decltype(s)::value><<<(B + threads - 1) / threads, threads, 0, st>>>(B, prm, N, x0, U, ustride, max_norm, X);
        return check_launch("k_rollout");
    });
}

int dispatch_linearize(int B, int sys, const double* params_host, int N, const double* X, const double* U, long ustride,
                       int central, double epsx, double epsu, double relx, double relu, int f0_from_x, const int* skip,
                       double* A, double* Bm, cudaStream_t st) {
    const DynParams prm = dyn_params(params_host);
    return with_system(sys, "hop_linearize_f64", [&](auto s) {
        constexpr int SYS = decltype(s)::value;
        constexpr int P = SysDims<SYS>::n + SysDims<SYS>::m;
        const size_t total = (size_t)B * N * P;
        const int threads = 128;
        const size_t grid = (total + threads - 1) / threads;
        if (SYS == 2 && g_linearize_variant == 0) {
            const size_t rows = (size_t)B * N;
            const unsigned g = (unsigned)((rows + threads - 1) / threads);
            if (central) k_linearize_quad_row<true><<<g, threads, 0, st>>>(B, prm, N, X, U, ustride, epsx, epsu, relx, relu, 0, skip, A, Bm);
            else k_linearize_quad_row<false><<<g, threads, 0, st>>>(B, prm, N, X, U, ustride, epsx, epsu, relx, relu, f0_from_x, skip, A, Bm);
            return check_launch("k_linearize_quad_row");
        }
        k_linearize<SYS><<<(unsigned)grid, threads, 0, st>>>(B, prm, N, X, U, ustride, central, epsx, epsu, relx, relu, skip, A, Bm);
        return check_launch("k_linearize");
    });
}

int sys_dims(int sys, const char* where, int* n, int* m) {
    return with_system(sys, where, [&](auto s) {
        *n = SysDims<decltype(s)::value>::n;
        *m = SysDims<decltype(s)::value>::m;
        return 0;
    });
}

}  // namespace hop
