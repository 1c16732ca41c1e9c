/* hop_oracle.c -- CPU ORACLE (test infrastructure; see hop_oracle.h for the usage contract).
 *
 * Plain-C restatement of the reference's HOP hot path.  Citations are file:line into the reference
 * tree (dmmsjtu-umich/time-opt-ilqr).  Build with -ffp-contract=off so that scalar expressions
 * round like the Python/numpy scalar arithmetic they restate.
 */
#include "hop_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#define HOP_MAXD 16
#define HOP_MAXN 16 /* max state dim */
#define HOP_MAXM 16 /* max control dim */

/* state / control dimensions an entry point can hold in its stack arrays (the augmented d = n + 1 <= HOP_MAXD) */
static int dims_ok(int n, int m) { return n >= 1 && n + 1 <= HOP_MAXD && m >= 1 && m <= HOP_MAXM; }

/* ------------------------------------------------------------------------------------------ */
/* precision-generic linear algebra + propagator                                               */
/* ------------------------------------------------------------------------------------------ */
#define REAL double
#define SFX(x) x##_f64
#include "hop_la.inc"
#undef REAL
#undef SFX

#define REAL long double
#define SFX(x) x##_f80
#define HOP_REAL_IS_LD 1
#include "hop_la.inc"
#undef HOP_REAL_IS_LD
#undef REAL
#undef SFX

static const double HOP_JITTER = 1e-9; /* utils.py:69,96 defaults */
static const int HOP_TRIES = 8;

const char *hopo_version(void) { return "hop-oracle 0.1 (restates dmmsjtu-umich/time-opt-ilqr modular code)"; }

int hopo_chol_inv(int d, const double *A, double *X, double jitter, int max_tries, int *info)
{
    if (d < 1 || d > HOP_MAXD) return HOP_ERR_ARG;
    return la_chol_inv_f64(d, A, X, jitter, max_tries, info);
}
int hopo_chol_solve(int d, int c, const double *A, const double *B, double *X, double jitter, int max_tries)
{
    if (d < 1 || d > HOP_MAXD || c < 1 || c > HOP_MAXD) return HOP_ERR_ARG;
    return la_chol_solve_f64(d, c, A, B, X, jitter, max_tries);
}

/* utils.py:127-128  (a + pi) % (2 pi) - pi with Python's FLOORED modulo */
double hopo_angle_normalize(double a)
{
    const double two_pi = 2.0 * M_PI;
    double s = a + M_PI;
    double r = fmod(s, two_pi);
    if (r != 0.0) {
        if (r < 0.0) r += two_pi;
    } else {
        r = 0.0;
    }
    return r - M_PI;
}
/* utils.py:131-137 */
void hopo_wrap_error(int n, double *e, unsigned wrap_mask)
{
    for (int i = 0; i < n; ++i)
        if (wrap_mask & (1u << i)) e[i] = hopo_angle_normalize(e[i]);
}

/* ------------------------------------------------------------------------------------------ */
/* systems.py : discrete dynamics F(x,u)                                                        */
/* ------------------------------------------------------------------------------------------ */
int hopo_sys_dims(int sys, int *n, int *m)
{
    switch (sys) {
    case HOP_SYS_DOUBLE_INTEGRATOR: *n = 2; *m = 1; return HOP_OK;
    case HOP_SYS_CARTPOLE: *n = 4; *m = 1; return HOP_OK;
    case HOP_SYS_QUADROTOR: *n = 12; *m = 4; return HOP_OK;
    case HOP_SYS_SEGWAY: *n = 4; *m = 1; return HOP_OK;
    }
    return HOP_ERR_ARG;
}

/* systems.py:30-33.  p = [dt] */
static void dyn_double_integrator(const double *p, const double *x, const double *u, double *xn)
{
    const double dt = p[0];
    double a = x[0] + dt * x[1], b = x[1] + dt * u[0];
    xn[0] = a; xn[1] = b;
}
/* systems.py:72-95.  p = [dt, g, m_pole, length, total_mass, polemass_length] */
static void dyn_cartpole(const double *p, const double *x, const double *u, double *xn)
{
    const double dt = p[0], g = p[1], m_pole = p[2], length = p[3], total_mass = p[4], pml = p[5];
    const double x_pos = x[0], x_dot = x[1], th = x[2], th_dot = x[3], force = u[0];
    const double th_u = th - M_PI;
    const double costh = cos(th_u), sinth = sin(th_u);
    const double temp = (force + pml * th_dot * th_dot * sinth) / total_mass;
    const double denom = length * (4.0 / 3.0 - m_pole * costh * costh / total_mass);
    const double th_acc = (g * sinth - costh * temp) / denom;
    const double x_acc = temp - pml * th_acc * costh / total_mass;
    xn[0] = x_pos + dt * x_dot;
    xn[1] = x_dot + dt * x_acc;
    xn[2] = hopo_angle_normalize(th + dt * th_dot);
    xn[3] = th_dot + dt * th_acc;
}
/* systems.py:321-333.  p = [dt, A_tau, A_th, B_tau, B_th] */
static void dyn_segway(const double *p, const double *x, const double *u, double *xn)
{
    const double dt = p[0], A_tau = p[1], A_th = p[2], B_tau = p[3], B_th = p[4];
    const double x_pos = x[0], x_dot = x[1], th = x[2], th_dot = x[3], tau = u[0];
    const double xdd = A_tau * tau + A_th * th;
    const double thdd = B_tau * tau + B_th * th;
    xn[0] = x_pos + dt * x_dot;
    xn[1] = x_dot + dt * xdd;
    xn[2] = hopo_angle_normalize(th + dt * th_dot);
    xn[3] = th_dot + dt * thdd;
}
/* systems.py:170-210 (rotm :145-156, Tmat :158-163, guards :175-191).
 * p = [dt, m, g, Ix, Iy, Iz, 1/Ix, 1/Iy, 1/Iz, kv, kw, cos_pitch_min, omg_abs_max, state_norm_max] */
static void dyn_quadrotor(const double *p, const double *x, const double *u, double *xn)
{
    const double dt = p[0], mass = p[1], g = p[2], Ix = p[3], Iy = p[4], Iz = p[5];
    const double iIx = p[6], iIy = p[7], iIz = p[8], kv = p[9], kw = p[10];
    const double cos_pitch_min = p[11], omg_abs_max = p[12], state_norm_max = p[13];
    int bad = 0;
    double ss = 0.0;
    for (int i = 0; i < 12; ++i) { if (!isfinite(x[i])) bad = 1; ss += x[i] * x[i]; }
    for (int i = 0; i < 4; ++i) if (!isfinite(u[i])) bad = 1;
    if (!bad && sqrt(ss) > state_norm_max) bad = 1;
    const double phi = x[6], th = x[7], psi = x[8];
    const double wp = x[9], wq = x[10], wr = x[11];
    const double cth = cos(th);
    if (!bad && fabs(cth) < cos_pitch_min) bad = 1;
    if (!bad && (fabs(wp) > omg_abs_max || fabs(wq) > omg_abs_max || fabs(wr) > omg_abs_max)) bad = 1;
    if (bad) { for (int i = 0; i < 12; ++i) xn[i] = NAN; return; }

    const double thrust = u[0];
    const double sphi = sin(phi), cphi = cos(phi), sth = sin(th), spsi = sin(psi), cpsi = cos(psi);
    const double tth = tan(th), secth = 1.0 / cth;
    /* third column of (Rz Ry) Rx */
    const double r02 = (-spsi) * (-sphi) + (cpsi * sth) * cphi;
    const double r12 = cpsi * (-sphi) + (spsi * sth) * cphi;
    const double r22 = cth * cphi;
    double xdot[12];
    xdot[0] = x[3]; xdot[1] = x[4]; xdot[2] = x[5];
    xdot[3] = (r02 * thrust) / mass - 0.0 - kv * x[3];
    xdot[4] = (r12 * thrust) / mass - 0.0 - kv * x[4];
    xdot[5] = (r22 * thrust) / mass - g - kv * x[5];
    xdot[6] = 1.0 * wp + (sphi * tth) * wq + (cphi * tth) * wr;
    xdot[7] = cphi * wq + (-sphi) * wr;
    xdot[8] = (sphi * secth) * wq + (cphi * secth) * wr;
    const double Iw0 = Ix * wp, Iw1 = Iy * wq, Iw2 = Iz * wr;
    const double c0 = wq * Iw2 - wr * Iw1, c1 = wr * Iw0 - wp * Iw2, c2 = wp * Iw1 - wq * Iw0;
    xdot[9] = iIx * (u[1] - c0) - kw * wp;
    xdot[10] = iIy * (u[2] - c1) - kw * wq;
    xdot[11] = iIz * (u[3] - c2) - kw * wr;
    for (int i = 0; i < 12; ++i) xn[i] = x[i] + dt * xdot[i];
}

void hopo_dynamics(int sys, const double *p, const double *x, const double *u, double *xn)
{
    switch (sys) {
    case HOP_SYS_DOUBLE_INTEGRATOR: dyn_double_integrator(p, x, u, xn); break;
    case HOP_SYS_CARTPOLE: dyn_cartpole(p, x, u, xn); break;
    case HOP_SYS_QUADROTOR: dyn_quadrotor(p, x, u, xn); break;
    case HOP_SYS_SEGWAY: dyn_segway(p, x, u, xn); break;
    default: break;
    }
}

static int vec_finite(int n, const double *x)
{
    for (int i = 0; i < n; ++i) if (!isfinite(x[i])) return 0;
    return 1;
}

/* solver.py:42-62  rollout: X[k+1] = F(X[k],U[k]); on non-finite or ||x|| > max_state_norm the
 * remainder is NaN-filled. */
void hopo_rollout(int sys, const double *p, int N, const double *x0, const double *U, double *X,
                  double max_state_norm)
{
    int n, m;
    if (hopo_sys_dims(sys, &n, &m)) return;
    memcpy(X, x0, sizeof(double) * n);
    for (int k = 0; k < N; ++k) {
        double xn[HOP_MAXN];
        hopo_dynamics(sys, p, X + (size_t)k * n, U + (size_t)k * m, xn);
        double ss = 0.0;
        for (int i = 0; i < n; ++i) ss += xn[i] * xn[i];
        if (!vec_finite(n, xn) || sqrt(ss) > max_state_norm) {
            for (size_t i = (size_t)(k + 1) * n; i < (size_t)(N + 1) * n; ++i) X[i] = NAN;
            return;
        }
        memcpy(X + (size_t)(k + 1) * n, xn, sizeof(double) * n);
    }
}

/* e^T (M e), as `e @ (M @ e)` */
static double quad_form(int n, const double *M, const double *e)
{
    double acc = 0.0;
    double Me[HOP_MAXN];
    for (int i = 0; i < n; ++i) {
        double s = 0.0;
        for (int j = 0; j < n; ++j) s += M[i * n + j] * e[j];
        Me[i] = s;
    }
    for (int i = 0; i < n; ++i) acc += e[i] * Me[i];
    return acc;
}

/* solver.py:65-105  cost_timeopt_true */
double hopo_cost_timeopt_true(int n, int m, const double *X, const double *U, const double *xg,
                              const double *u_ref, const double *Q, const double *R, const double *Qf,
                              double w, int T_star, unsigned wrap_mask)
{
    if (!dims_ok(n, m)) return NAN;
    if (T_star <= 0) return INFINITY;
    if (!vec_finite((T_star + 1) * n, X) || !vec_finite(T_star * m, U)) return INFINITY;
    double c = 0.0, e[HOP_MAXN], du[HOP_MAXM];
    for (int k = 0; k < T_star; ++k) {
        for (int i = 0; i < n; ++i) e[i] = X[(size_t)k * n + i] - xg[i];
        hopo_wrap_error(n, e, wrap_mask);
        for (int i = 0; i < m; ++i) du[i] = U[(size_t)k * m + i] - u_ref[i];
        if (!vec_finite(n, e) || !vec_finite(m, du)) return INFINITY;
        c += 0.5 * quad_form(n, Q, e) + 0.5 * quad_form(m, R, du) + w;
    }
    for (int i = 0; i < n; ++i) e[i] = X[(size_t)T_star * n + i] - xg[i];
    hopo_wrap_error(n, e, wrap_mask);
    if (!vec_finite(n, e)) return INFINITY;
    c += 0.5 * quad_form(n, Qf, e);
    return c;
}

/* linearization.py:216-262 (forward, f0 non-finite => NaN blocks) and :177-211 (central).
 * h_i = max(eps, rel * max(1, |x_i|)). */
void hopo_linearize(int sys, const double *p, int N, const double *X, const double *U, int central,
                    double epsx, double epsu, double relx, double relu, double *A, double *B)
{
    int n, m;
    if (hopo_sys_dims(sys, &n, &m)) return;
    for (int k = 0; k < N; ++k) {
        const double *x = X + (size_t)k * n, *u = U + (size_t)k * m;
        double *Ak = A + (size_t)k * n * n, *Bk = B + (size_t)k * n * m;
        double f0[HOP_MAXN], fp[HOP_MAXN], fm[HOP_MAXN], xp[HOP_MAXN], up[HOP_MAXM];
        if (!central) {
            hopo_dynamics(sys, p, x, u, f0);
            if (!vec_finite(n, f0)) {
                for (int i = 0; i < n * n; ++i) Ak[i] = NAN;
                for (int i = 0; i < n * m; ++i) Bk[i] = NAN;
                continue;
            }
        }
        for (int i = 0; i < n; ++i) {
            double ax = fabs(x[i]);
            double hi = fmax(epsx, relx * fmax(1.0, ax));
            memcpy(xp, x, sizeof(double) * n);
            if (central) {
                xp[i] = x[i] + hi; hopo_dynamics(sys, p, xp, u, fp);
                xp[i] = x[i] - hi; hopo_dynamics(sys, p, xp, u, fm);
                for (int r = 0; r < n; ++r) Ak[r * n + i] = (fp[r] - fm[r]) / (2.0 * hi);
            } else {
                xp[i] = x[i] + hi; hopo_dynamics(sys, p, xp, u, fp);
                for (int r = 0; r < n; ++r) Ak[r * n + i] = (fp[r] - f0[r]) / hi;
            }
        }
        for (int j = 0; j < m; ++j) {
            double au = fabs(u[j]);
            double hj = fmax(epsu, relu * fmax(1.0, au));
            memcpy(up, u, sizeof(double) * m);
            if (central) {
                up[j] = u[j] + hj; hopo_dynamics(sys, p, x, up, fp);
                up[j] = u[j] - hj; hopo_dynamics(sys, p, x, up, fm);
                for (int r = 0; r < n; ++r) Bk[r * m + j] = (fp[r] - fm[r]) / (2.0 * hj);
            } else {
                up[j] = u[j] + hj; hopo_dynamics(sys, p, x, up, fp);
                for (int r = 0; r < n; ++r) Bk[r * m + j] = (fp[r] - f0[r]) / hj;
            }
        }
    }
}

/* linearization.py:269-270  a_k = F(X_k,U_k) - X_{k+1} */
void hopo_affine_residuals(int sys, const double *p, int N, const double *X, const double *U, double *a)
{
    int n, m;
    if (hopo_sys_dims(sys, &n, &m)) return;
    for (int k = 0; k < N; ++k) {
        double f[HOP_MAXN];
        hopo_dynamics(sys, p, X + (size_t)k * n, U + (size_t)k * m, f);
        for (int i = 0; i < n; ++i) a[(size_t)k * n + i] = f[i] - X[(size_t)(k + 1) * n + i];
    }
}

/* augmented.py:10-60  build_augmented_sequence_QR (extra_stage_cost=None).
 * a may be NULL (treated as exactly zero).  Outputs: A_aug[N][d][d], B_aug[N][d][m],
 * Q_aug[N][d][d], R_inv[m][m] = chol_inv(sym(R)). */
int hopo_build_augmented(int n, int m, int N, const double *A, const double *B, const double *a,
                         const double *X, const double *U, const double *xg, const double *u_ref,
                         const double *Q, const double *R, double w, unsigned wrap_mask, double q_reg,
                         double rho_reg, double *A_aug, double *B_aug, double *Q_aug, double *R_inv)
{
    const int d = n + 1;
    if (!dims_ok(n, m)) return HOP_ERR_ARG;
    double Rs[HOP_MAXM * HOP_MAXM], Qs[HOP_MAXN * HOP_MAXN];
    la_sym_f64(m, R, Rs);
    int rc = la_chol_inv_f64(m, Rs, R_inv, HOP_JITTER, HOP_TRIES, NULL); /* :23 */
    if (rc) return rc;
    la_sym_f64(n, Q, Qs);
    for (int k = 0; k < N; ++k) {
        double e[HOP_MAXN], du[HOP_MAXM], Qe[HOP_MAXN], Qk[HOP_MAXD * HOP_MAXD];
        for (int i = 0; i < n; ++i) e[i] = X[(size_t)k * n + i] - xg[i];
        hopo_wrap_error(n, e, wrap_mask);
        for (int i = 0; i < m; ++i) du[i] = U[(size_t)k * m + i] - u_ref[i];
        for (int i = 0; i < n; ++i) {
            double s = 0.0;
            for (int j = 0; j < n; ++j) s += Q[i * n + j] * e[j];
            Qe[i] = s;
        }
        /* :31-37 ; e^T Q e evaluated as (e^T Q) e */
        double eQe = 0.0;
        for (int j = 0; j < n; ++j) {
            double s = 0.0;
            for (int i = 0; i < n; ++i) s += e[i] * Q[i * n + j];
            eQe += s * e[j];
        }
        for (int i = 0; i < n; ++i) {
            for (int j = 0; j < n; ++j) Qk[i * d + j] = Qs[i * n + j] + (i == j ? q_reg : 0.0);
            Qk[i * d + n] = Qe[i];
            Qk[n * d + i] = Qe[i];
        }
        Qk[n * d + n] = eQe + 2.0 * w + rho_reg;
        la_sym_f64(d, Qk, Q_aug + (size_t)k * d * d); /* :48 */
        /* :50-56 */
        double *Ak = A_aug + (size_t)k * d * d, *Bk = B_aug + (size_t)k * d * m;
        for (int i = 0; i < d * d; ++i) Ak[i] = 0.0;
        for (int i = 0; i < d * m; ++i) Bk[i] = 0.0;
        for (int i = 0; i < n; ++i) {
            double Bdu = 0.0;
            for (int j = 0; j < m; ++j) Bdu += B[(size_t)k * n * m + i * m + j] * du[j];
            double ak = a ? a[(size_t)k * n + i] : 0.0;
            for (int j = 0; j < n; ++j) Ak[i * d + j] = A[(size_t)k * n * n + i * n + j];
            Ak[i * d + n] = ak - Bdu;
            for (int j = 0; j < m; ++j) Bk[i * m + j] = B[(size_t)k * n * m + i * m + j];
        }
        Ak[n * d + n] = 1.0;
    }
    return HOP_OK;
}

/* augmented.py:63-87  build_terminal_aug_list: QT[t-1] from X[t], t = 1..N */
int hopo_build_terminal(int n, int N, const double *X, const double *xg, const double *Qf,
                        unsigned wrap_mask, double rho_reg, double *QT)
{
    const int d = n + 1;
    if (!dims_ok(n, 1)) return HOP_ERR_ARG;
    double P[HOP_MAXN * HOP_MAXN];
    la_sym_f64(n, Qf, P);
    for (int t = 1; t <= N; ++t) {
        double e[HOP_MAXN], px[HOP_MAXN], Qt[HOP_MAXD * HOP_MAXD];
        for (int i = 0; i < n; ++i) e[i] = X[(size_t)t * n + i] - xg[i];
        hopo_wrap_error(n, e, wrap_mask);
        double ePe = 0.0;
        for (int i = 0; i < n; ++i) {
            double s = 0.0;
            for (int j = 0; j < n; ++j) s += P[i * n + j] * e[j];
            px[i] = s;
        }
        for (int i = 0; i < n; ++i) ePe += e[i] * px[i];
        const double p0 = 0.5 * ePe;
        for (int i = 0; i < n; ++i) {
            for (int j = 0; j < n; ++j) Qt[i * d + j] = P[i * n + j];
            Qt[i * d + n] = px[i];
            Qt[n * d + i] = px[i];
        }
        Qt[n * d + n] = 2.0 * p0 + rho_reg;
        la_sym_f64(d, Qt, QT + (size_t)(t - 1) * d * d);
    }
    return HOP_OK;
}

int hopo_propagator_all_Jt_f64(int T_use, int d, int m, const double *A_aug, const double *B_aug,
                               const double *Q_aug, const double *R_inv, long rinv_stride, const double *z0,
                               const double *QT, double *J, double jitter, int max_tries, long *retries)
{
    if (d < 1 || d > HOP_MAXD || m < 1 || m > HOP_MAXD) return HOP_ERR_ARG;
    if (rinv_stride != 0 && rinv_stride != (long)m * m) return HOP_ERR_ARG;
    return propagator_all_Jt_f64(T_use, d, m, A_aug, B_aug, Q_aug, R_inv, rinv_stride, z0, QT, J, jitter, max_tries, retries);
}
int hopo_propagator_all_Jt_f80(int T_use, int d, int m, const double *A_aug, const double *B_aug,
                               const double *Q_aug, const double *R_inv, long rinv_stride, const double *z0,
                               const double *QT, double *J, double jitter, int max_tries, long *retries)
{
    if (d < 1 || d > HOP_MAXD || m < 1 || m > HOP_MAXD) return HOP_ERR_ARG;
    if (rinv_stride != 0 && rinv_stride != (long)m * m) return HOP_ERR_ARG;
    return propagator_all_Jt_f80(T_use, d, m, A_aug, B_aug, Q_aug, R_inv, rinv_stride, z0, QT, J, jitter, max_tries, retries);
}

/* solver.py:522,590.  np.argmin returns the first minimum and treats NaN as the minimum. */
int hopo_argmin_window(const double *J, int T_min, int T_max)
{
    int best = T_min - 1;
    for (int i = T_min - 1; i < T_max; ++i) {
        if (isnan(J[i])) { best = i; break; }
        if (J[i] < J[best]) best = i;
    }
    return best + 1; /* = argmin + T_min in the reference's indexing */
}

int hopo_select_fused(int sys, const double *p, int n, int m, int N, int T_min, int T_max,
                      const double *A, const double *B, const double *a_resid, const double *X,
                      const double *U, const double *xg, const double *u_ref, const double *Q,
                      const double *R, const double *Qf, double w, unsigned wrap_mask, int use_f80,
                      double *J, int *T_star)
{
    const int d = n + 1;
    if (!dims_ok(n, m) || T_max > N || T_min < 1 || T_min > T_max) return HOP_ERR_ARG;
    size_t tot = (size_t)N * (3 * d * d + d * m) + (size_t)N * n;
    double *buf = (double *)malloc(sizeof(double) * tot);
    if (!buf) return HOP_ERR_ALLOC;
    double *A_aug = buf, *Q_aug = A_aug + (size_t)N * d * d, *QT = Q_aug + (size_t)N * d * d;
    double *B_aug = QT + (size_t)N * d * d, *a_own = B_aug + (size_t)N * d * m;
    double R_inv[HOP_MAXM * HOP_MAXM], z0[HOP_MAXD];
    const double *a = a_resid;
    if (!a && sys >= 0) { hopo_affine_residuals(sys, p, N, X, U, a_own); a = a_own; }
    int rc = hopo_build_augmented(n, m, N, A, B, a, X, U, xg, u_ref, Q, R, w, wrap_mask, 1e-9, 1e-12,
                                  A_aug, B_aug, Q_aug, R_inv);
    if (!rc) {
        hopo_build_terminal(n, N, X, xg, Qf, wrap_mask, 1e-12, QT);
        for (int i = 0; i < d; ++i) z0[i] = 0.0;
        z0[d - 1] = 1.0; /* augmented.py:59 */
        rc = use_f80 ? propagator_all_Jt_f80(T_max, d, m, A_aug, B_aug, Q_aug, R_inv, 0, z0, QT, J, HOP_JITTER, HOP_TRIES, NULL)
                     : propagator_all_Jt_f64(T_max, d, m, A_aug, B_aug, Q_aug, R_inv, 0, z0, QT, J, HOP_JITTER, HOP_TRIES, NULL);
    }
    if (!rc) *T_star = hopo_argmin_window(J, T_min, T_max);
    free(buf);
    return rc;
}

static int select_from_x0_impl(int sys, const double *p, int N, int T_min, int T_max, const double *x0,
                               const double *U, const double *xg, const double *u_ref, const double *Q,
                               const double *R, const double *Qf, double w, unsigned wrap_mask, int central,
                               int use_f80, double *J, int *T_star);
int hopo_select_from_x0(int sys, const double *p, int N, int T_min, int T_max, const double *x0,
                        const double *U, const double *xg, const double *u_ref, const double *Q,
                        const double *R, const double *Qf, double w, unsigned wrap_mask, int central,
                        double *J, int *T_star)
{
    return select_from_x0_impl(sys, p, N, T_min, T_max, x0, U, xg, u_ref, Q, R, Qf, w, wrap_mask, central, 0, J, T_star);
}
/* use_f80: the SELECTION sweep in x87 extended precision on the same fp64 rollout / linearisation ("truth" of the
 * jittered algorithm, for noise accounting only) */
static int select_from_x0_impl(int sys, const double *p, int N, int T_min, int T_max, const double *x0,
                               const double *U, const double *xg, const double *u_ref, const double *Q,
                               const double *R, const double *Qf, double w, unsigned wrap_mask, int central,
                               int use_f80, double *J, int *T_star)
{
    int n, m;
    if (hopo_sys_dims(sys, &n, &m)) return HOP_ERR_ARG;
    double *buf = (double *)malloc(sizeof(double) * ((size_t)(N + 1) * n + (size_t)N * n * (n + m)));
    if (!buf) return HOP_ERR_ALLOC;
    double *X = buf, *A = X + (size_t)(N + 1) * n, *B = A + (size_t)N * n * n;
    hopo_rollout(sys, p, N, x0, U, X, 1e6);
    hopo_linearize(sys, p, N, X, U, central, 1e-5, 1e-5, 1e-6, 1e-6, A, B);
    int rc = hopo_select_fused(sys, p, n, m, N, T_min, T_max, A, B, NULL, X, U, xg, u_ref, Q, R, Qf, w,
                               wrap_mask, use_f80, J, T_star);
    free(buf);
    return rc;
}

/* solver.py:156-230  backward_pass_truncated (extra_stage_cost=None).
 * k_out [T*][m], K_out [T*][m][n].  *ok = 0 reproduces the reference's `return None, None, False`.
 * A non-zero return reproduces an exception escaping (chol_solve raising, utils.py:120). */
int hopo_backward_pass(int n, int m, const double *A, const double *B, const double *X, const double *U,
                       const double *xg, const double *u_ref, const double *Q, const double *R,
                       const double *Qf, int T_star, double lm_lambda, unsigned wrap_mask,
                       double *k_out, double *K_out, int *ok)
{
    *ok = 0;
    if (!dims_ok(n, m)) return HOP_ERR_ARG;
    if (T_star <= 0) return HOP_OK;
    double e[HOP_MAXN], du[HOP_MAXM], Vx[HOP_MAXN], Vxx[HOP_MAXN * HOP_MAXN];
    for (int i = 0; i < n; ++i) e[i] = X[(size_t)T_star * n + i] - xg[i];
    hopo_wrap_error(n, e, wrap_mask);
    if (!vec_finite(n, e)) return HOP_OK;
    for (int i = 0; i < n; ++i) {
        double s = 0.0;
        for (int j = 0; j < n; ++j) s += Qf[i * n + j] * e[j];
        Vx[i] = s;
    }
    la_sym_f64(n, Qf, Vxx);
    for (int k = T_star - 1; k >= 0; --k) {
        const double *Ak = A + (size_t)k * n * n, *Bk = B + (size_t)k * n * m;
        for (int i = 0; i < n; ++i) e[i] = X[(size_t)k * n + i] - xg[i];
        hopo_wrap_error(n, e, wrap_mask);
        for (int i = 0; i < m; ++i) du[i] = U[(size_t)k * m + i] - u_ref[i];
        if (!vec_finite(n, e) || !vec_finite(m, du)) return HOP_OK;
        double lx[HOP_MAXN], lu[HOP_MAXM], Qx[HOP_MAXN], Qu[HOP_MAXM];
        double Qxx[HOP_MAXN * HOP_MAXN], Quu[HOP_MAXM * HOP_MAXM], Qux[HOP_MAXM * HOP_MAXN];
        double AtV[HOP_MAXN * HOP_MAXN], BtV[HOP_MAXM * HOP_MAXN], t[HOP_MAXN * HOP_MAXN];
        for (int i = 0; i < n; ++i) { double s = 0.0; for (int j = 0; j < n; ++j) s += Q[i * n + j] * e[j]; lx[i] = s; }
        for (int i = 0; i < m; ++i) { double s = 0.0; for (int j = 0; j < m; ++j) s += R[i * m + j] * du[j]; lu[i] = s; }
        for (int i = 0; i < n; ++i) { double s = 0.0; for (int l = 0; l < n; ++l) s += Ak[l * n + i] * Vx[l]; Qx[i] = lx[i] + s; }
        for (int i = 0; i < m; ++i) { double s = 0.0; for (int l = 0; l < n; ++l) s += Bk[l * m + i] * Vx[l]; Qu[i] = lu[i] + s; }
        la_mtm_f64(n, n, n, Ak, Vxx, AtV);       /* A^T Vxx */
        la_mm_f64(n, n, n, AtV, Ak, t);          /* (A^T Vxx) A */
        for (int i = 0; i < n * n; ++i) Qxx[i] = Q[i] + t[i];
        la_mtm_f64(m, n, n, Bk, Vxx, BtV);       /* B^T Vxx */
        la_mm_f64(m, n, m, BtV, Bk, t);
        for (int i = 0; i < m * m; ++i) Quu[i] = R[i] + t[i];
        la_mm_f64(m, n, n, BtV, Ak, Qux);
        double Quu_reg[HOP_MAXM * HOP_MAXM], Ltmp[HOP_MAXM * HOP_MAXM];
        la_sym_f64(m, Quu, Quu_reg);
        for (int i = 0; i < m; ++i) Quu_reg[i * m + i] += lm_lambda;
        if (la_cholesky_f64(m, Quu_reg, Ltmp) != 0) return HOP_OK; /* :213-216 */
        double kap[HOP_MAXM], Kk[HOP_MAXM * HOP_MAXN];
        int rc = la_chol_solve_f64(m, 1, Quu_reg, Qu, kap, HOP_JITTER, HOP_TRIES);
        if (rc) return rc;
        rc = la_chol_solve_f64(m, n, Quu_reg, Qux, Kk, HOP_JITTER, HOP_TRIES);
        if (rc) return rc;
        for (int i = 0; i < m; ++i) kap[i] = -kap[i];
        for (int i = 0; i < m * n; ++i) Kk[i] = -Kk[i];
        memcpy(k_out + (size_t)k * m, kap, sizeof(double) * m);
        memcpy(K_out + (size_t)k * m * n, Kk, sizeof(double) * m * n);
        /* Vx = Qx + K^T Qu + Qux^T kappa + (K^T Quu) kappa   (:224) */
        double KtQuu[HOP_MAXN * HOP_MAXM];
        la_mtm_f64(n, m, m, Kk, Quu, KtQuu);
        double Vxn[HOP_MAXN], Vxxn[HOP_MAXN * HOP_MAXN];
        for (int i = 0; i < n; ++i) {
            double s1 = 0.0, s2 = 0.0, s3 = 0.0;
            for (int l = 0; l < m; ++l) s1 += Kk[l * n + i] * Qu[l];
            for (int l = 0; l < m; ++l) s2 += Qux[l * n + i] * kap[l];
            for (int l = 0; l < m; ++l) s3 += KtQuu[i * m + l] * kap[l];
            Vxn[i] = ((Qx[i] + s1) + s2) + s3;
        }
        /* Vxx = sym(Qxx + K^T Qux + Qux^T K + (K^T Quu) K)   (:225) */
        double t1[HOP_MAXN * HOP_MAXN], t2[HOP_MAXN * HOP_MAXN], t3[HOP_MAXN * HOP_MAXN];
        la_mtm_f64(n, m, n, Kk, Qux, t1);
        la_mtm_f64(n, m, n, Qux, Kk, t2);
        la_mm_f64(n, m, n, KtQuu, Kk, t3);
        for (int i = 0; i < n * n; ++i) t[i] = ((Qxx[i] + t1[i]) + t2[i]) + t3[i];
        la_sym_f64(n, t, Vxxn);
        memcpy(Vx, Vxn, sizeof(double) * n);
        memcpy(Vxx, Vxxn, sizeof(double) * n * n);
        if (!vec_finite(n, Vx) || !vec_finite(n * n, Vxx)) return HOP_OK;
    }
    *ok = 1;
    return HOP_OK;
}

/* solver.py:233-286  forward_linesearch_fixedT, alphas = (1, .5, .25, .1, .05) */
int hopo_forward_linesearch(int sys, const double *p, int N, const double *X, const double *U,
                            const double *xg, const double *u_ref, const double *Q, const double *R,
                            const double *Qf, double w, int T_star, const double *k_list,
                            const double *K_list, unsigned wrap_mask, double *X_new, double *U_new,
                            double *J_out, int *accepted)
{
    static const double alphas[5] = {1.0, 0.5, 0.25, 0.1, 0.05};
    int n, m;
    if (hopo_sys_dims(sys, &n, &m)) return HOP_ERR_ARG;
    const double J_old = hopo_cost_timeopt_true(n, m, X, U, xg, u_ref, Q, R, Qf, w, T_star, wrap_mask);
    for (int ai = 0; ai < 5; ++ai) {
        const double a = alphas[ai];
        memcpy(U_new, U, sizeof(double) * (size_t)N * m);
        memset(X_new, 0, sizeof(double) * (size_t)(N + 1) * n);
        memcpy(X_new, X, sizeof(double) * n);
        int ok = 1;
        for (int k = 0; k < N; ++k) {
            if (k < T_star) {
                double dx[HOP_MAXN];
                for (int i = 0; i < n; ++i) dx[i] = X_new[(size_t)k * n + i] - X[(size_t)k * n + i];
                hopo_wrap_error(n, dx, wrap_mask);
                for (int i = 0; i < m; ++i) {
                    double s = 0.0;
                    for (int j = 0; j < n; ++j) s += K_list[(size_t)k * m * n + i * n + j] * dx[j];
                    double du = s + a * k_list[(size_t)k * m + i];
                    U_new[(size_t)k * m + i] = U[(size_t)k * m + i] + du;
                }
            }
            hopo_dynamics(sys, p, X_new + (size_t)k * n, U_new + (size_t)k * m, X_new + (size_t)(k + 1) * n);
            if (!vec_finite(n, X_new + (size_t)(k + 1) * n)) { ok = 0; break; }
        }
        if (!ok) continue;
        const double J_new = hopo_cost_timeopt_true(n, m, X_new, U_new, xg, u_ref, Q, R, Qf, w, T_star, wrap_mask);
        if (J_new < J_old) { *J_out = J_new; *accepted = 1; return HOP_OK; }
    }
    memcpy(X_new, X, sizeof(double) * (size_t)(N + 1) * n);
    memcpy(U_new, U, sizeof(double) * (size_t)N * m);
    *J_out = J_old;
    *accepted = 0;
    return HOP_OK;
}

/* solver.py:293-358  bruteforce_all_Jt_backward_expansion (baseline-1, CPU comparator only) */
int hopo_bruteforce_all_Jt(int n, int m, const double *A, const double *B, const double *X, const double *U,
                           const double *xg, const double *u_ref, const double *Q, const double *R,
                           const double *Qf, double w, int T_max, double lm_lambda, unsigned wrap_mask,
                           double *J)
{
    if (!dims_ok(n, m)) return HOP_ERR_ARG;
    for (int T = 1; T <= T_max; ++T) {
        double e[HOP_MAXN], du[HOP_MAXM], Vx[HOP_MAXN], Vxx[HOP_MAXN * HOP_MAXN], V0;
        for (int i = 0; i < n; ++i) e[i] = X[(size_t)T * n + i] - xg[i];
        hopo_wrap_error(n, e, wrap_mask);
        la_sym_f64(n, Qf, Vxx);
        for (int i = 0; i < n; ++i) { double s = 0.0; for (int j = 0; j < n; ++j) s += Qf[i * n + j] * e[j]; Vx[i] = s; }
        V0 = 0.5 * quad_form(n, Qf, e);
        for (int t = T - 1; t >= 0; --t) {
            const double *Ak = A + (size_t)t * n * n, *Bk = B + (size_t)t * n * m;
            for (int i = 0; i < n; ++i) e[i] = X[(size_t)t * n + i] - xg[i];
            hopo_wrap_error(n, e, wrap_mask);
            for (int i = 0; i < m; ++i) du[i] = U[(size_t)t * m + i] - u_ref[i];
            double lx[HOP_MAXN], lu[HOP_MAXM], Qx[HOP_MAXN], Qu[HOP_MAXM];
            double Qxx[HOP_MAXN * HOP_MAXN], Quu[HOP_MAXM * HOP_MAXM], Qux[HOP_MAXM * HOP_MAXN];
            double AtV[HOP_MAXN * HOP_MAXN], BtV[HOP_MAXM * HOP_MAXN], tt[HOP_MAXN * HOP_MAXN];
            for (int i = 0; i < n; ++i) { double s = 0.0; for (int j = 0; j < n; ++j) s += Q[i * n + j] * e[j]; lx[i] = s; }
            for (int i = 0; i < m; ++i) { double s = 0.0; for (int j = 0; j < m; ++j) s += R[i * m + j] * du[j]; lu[i] = s; }
            const double l0 = 0.5 * quad_form(n, Q, e) + 0.5 * quad_form(m, R, du) + w;
            for (int i = 0; i < n; ++i) { double s = 0.0; for (int l = 0; l < n; ++l) s += Ak[l * n + i] * Vx[l]; Qx[i] = lx[i] + s; }
            for (int i = 0; i < m; ++i) { double s = 0.0; for (int l = 0; l < n; ++l) s += Bk[l * m + i] * Vx[l]; Qu[i] = lu[i] + s; }
            la_mtm_f64(n, n, n, Ak, Vxx, AtV);
            la_mm_f64(n, n, n, AtV, Ak, tt);
            for (int i = 0; i < n * n; ++i) Qxx[i] = Q[i] + tt[i];
            la_mtm_f64(m, n, n, Bk, Vxx, BtV);
            la_mm_f64(m, n, m, BtV, Bk, tt);
            for (int i = 0; i < m * m; ++i) Quu[i] = R[i] + tt[i];
            la_mm_f64(m, n, n, BtV, Ak, Qux);
            double Quu_reg[HOP_MAXM * HOP_MAXM], iQu[HOP_MAXM], iQux[HOP_MAXM * HOP_MAXN];
            la_sym_f64(m, Quu, Quu_reg);
            for (int i = 0; i < m; ++i) Quu_reg[i * m + i] += lm_lambda;
            int rc = la_chol_solve_f64(m, 1, Quu_reg, Qu, iQu, HOP_JITTER, HOP_TRIES);
            if (rc) return rc;
            rc = la_chol_solve_f64(m, n, Quu_reg, Qux, iQux, HOP_JITTER, HOP_TRIES);
            if (rc) return rc;
            double t1[HOP_MAXN * HOP_MAXN], Vxxn[HOP_MAXN * HOP_MAXN], Vxn[HOP_MAXN];
            la_mtm_f64(n, m, n, Qux, iQux, t1);
            for (int i = 0; i < n * n; ++i) tt[i] = Qxx[i] - t1[i];
            la_sym_f64(n, tt, Vxxn);
            double qq = 0.0;
            for (int i = 0; i < n; ++i) { double s = 0.0; for (int l = 0; l < m; ++l) s += Qux[l * n + i] * iQu[l]; Vxn[i] = Qx[i] - s; }
            for (int l = 0; l < m; ++l) qq += Qu[l] * iQu[l];
            V0 = l0 + V0 - 0.5 * qq;
            memcpy(Vx, Vxn, sizeof(double) * n);
            memcpy(Vxx, Vxxn, sizeof(double) * n * n);
        }
        J[T - 1] = V0;
    }
    return HOP_OK;
}

/* solver.py:449-765  ilqr_timeopt, method="propagator" branch.
 * J_hist/T_hist have capacity max_iter+1.  J_curve[T_max] = last selection curve. */
int hopo_ilqr_timeopt(int sys, const double *p, int N, int T_min, int T_max, const double *x0,
                      const double *U_init, const double *xg, const double *u_ref, const double *Q,
                      const double *R, const double *Qf, double w, unsigned wrap_mask,
                      const hopo_ilqr_opts *opts, double *X_out, double *U_out, double *J_hist,
                      int *T_hist, int *n_hist, double *J_curve, int *T_star, int *n_outer)
{
    int n, m;
    if (hopo_sys_dims(sys, &n, &m)) return HOP_ERR_ARG;
    const size_t szX = (size_t)(N + 1) * n, szU = (size_t)N * m;
    double *buf = (double *)malloc(sizeof(double) * (2 * szX + 2 * szU + (size_t)N * n * (n + m) + (size_t)N * (m + m * n)));
    if (!buf) return HOP_ERR_ALLOC;
    double *X = buf, *U = X + szX, *Xn = U + szU, *Un = Xn + szX;
    double *A = Un + szU, *B = A + (size_t)N * n * n, *kl = B + (size_t)N * n * m, *Kl = kl + (size_t)N * m;
    int rc = HOP_OK, nh = 0, T_bar = T_min, ok = 0, acc = 0, iters = 0;
    double lm = opts->lm_init, Jn = 0.0;

    memcpy(U, U_init, sizeof(double) * szU);
    hopo_rollout(sys, p, N, x0, U, X, 1e6);                                               /* :492 */
    hopo_linearize(sys, p, N, X, U, opts->use_central_diff, 1e-5, 1e-5, 1e-6, 1e-6, A, B); /* :504-509 */
    rc = hopo_select_fused(sys, p, n, m, N, T_min, T_max, A, B, NULL, X, U, xg, u_ref, Q, R, Qf, w,
                           wrap_mask, opts->use_f80_select, J_curve, &T_bar);              /* :516-522 */
    if (rc) goto done;
    rc = hopo_backward_pass(n, m, A, B, X, U, xg, u_ref, Q, R, Qf, T_bar, lm, wrap_mask, kl, Kl, &ok); /* :541 */
    if (rc) goto done;
    if (ok) {
        rc = hopo_forward_linesearch(sys, p, N, X, U, xg, u_ref, Q, R, Qf, w, T_bar, kl, Kl, wrap_mask, Xn, Un, &Jn, &acc);
        if (rc) goto done;
        memcpy(X, Xn, sizeof(double) * szX);
        memcpy(U, Un, sizeof(double) * szU);
        if (isfinite(Jn)) { J_hist[nh] = Jn; T_hist[nh] = T_bar; ++nh; }                   /* :553-555 */
    }
    for (int it = 0; it < opts->max_iter; ++it) {                                          /* :564 */
        ++iters;
        hopo_linearize(sys, p, N, X, U, opts->use_central_diff, 1e-5, 1e-5, 1e-6, 1e-6, A, B);
        int T_sel = T_bar;
        acc = 0;
        rc = hopo_select_fused(sys, p, n, m, N, T_min, T_max, A, B, NULL, X, U, xg, u_ref, Q, R, Qf, w,
                               wrap_mask, opts->use_f80_select, J_curve, &T_sel);          /* :581-590 */
        if (rc) goto done;
        rc = hopo_backward_pass(n, m, A, B, X, U, xg, u_ref, Q, R, Qf, T_sel, lm, wrap_mask, kl, Kl, &ok);
        if (rc) goto done;
        if (ok) {
            rc = hopo_forward_linesearch(sys, p, N, X, U, xg, u_ref, Q, R, Qf, w, T_sel, kl, Kl, wrap_mask, Xn, Un, &Jn, &acc);
            if (rc) goto done;
        }
        if (ok && acc && isfinite(Jn)) {                                                   /* :735-742 */
            memcpy(X, Xn, sizeof(double) * szX);
            memcpy(U, Un, sizeof(double) * szU);
            T_bar = T_sel;
            J_hist[nh] = Jn; T_hist[nh] = T_sel; ++nh;
            lm = fmax(lm / 10.0, 1e-12);
        } else {
            lm *= 10.0;
        }
        if (nh >= 2) {                                                                     /* :745-748 */
            double rel = fabs(J_hist[nh - 1] - J_hist[nh - 2]) / (fabs(J_hist[nh - 2]) + 1e-12);
            if (rel < 1e-4 && nh >= 3 && T_hist[nh - 1] == T_hist[nh - 2] && T_hist[nh - 2] == T_hist[nh - 3]) break;
        }
    }
done:
    memcpy(X_out, X, sizeof(double) * szX);
    memcpy(U_out, U, sizeof(double) * szU);
    *n_hist = nh;
    *T_star = nh ? T_hist[nh - 1] : T_bar;                                                 /* :763 */
    if (n_outer) *n_outer = iters;
    free(buf);
    return rc;
}

/* ------------------------------------------------------------------------------------------ */
/* pthread fan-out over a batch (static contiguous partition)                                   */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    int kind, lo, hi;
    int sys, N, T_min, T_max, central, T_use, d, m, use_f80;
    long rinv_stride;
    const double *A, *B, *X, *a_resid;
    unsigned wrap_mask;
    const double *p, *x0, *U, *xg, *u_ref, *Q, *R, *Qf, *w;
    const double *A_aug, *B_aug, *Q_aug, *R_inv, *z0, *QT;
    const hopo_ilqr_opts *opts;
    double *J, *X_out, *U_out, *J_hist;
    int *T_star, *status, *T_hist, *n_hist;
} hopo_job;

static void *hopo_worker(void *arg)
{
    hopo_job *j = (hopo_job *)arg;
    int n = 0, m = 0;
    if (j->kind != 1 && j->kind != 3) hopo_sys_dims(j->sys, &n, &m);
    for (int b = j->lo; b < j->hi; ++b) {
        if (j->kind == 0) {
            j->status[b] = select_from_x0_impl(j->sys, j->p, j->N, j->T_min, j->T_max, j->x0 + (size_t)b * n,
                                               j->U, j->xg + (size_t)b * n, j->u_ref, j->Q, j->R, j->Qf, j->w[b],
                                               j->wrap_mask, j->central, j->use_f80, j->J + (size_t)b * j->T_max,
                                               &j->T_star[b]);
        } else if (j->kind == 3) {
            const size_t N_ = (size_t)j->N;
            j->status[b] = hopo_select_fused(-1, NULL, j->d, j->m, j->N, j->T_min, j->T_max,
                                             j->A + (size_t)b * N_ * j->d * j->d, j->B + (size_t)b * N_ * j->d * j->m,
                                             j->a_resid ? j->a_resid + (size_t)b * N_ * j->d : NULL,
                                             j->X + (size_t)b * (N_ + 1) * j->d, j->U + (size_t)b * N_ * j->m,
                                             j->xg + (size_t)b * j->d, j->u_ref, j->Q, j->R, j->Qf, j->w[b], j->wrap_mask,
                                             j->use_f80, j->J + (size_t)b * j->T_max, &j->T_star[b]);
        } else if (j->kind == 1) {
            const size_t dd = (size_t)j->d * j->d, dm = (size_t)j->d * j->m;
            j->status[b] = propagator_all_Jt_f64(j->T_use, j->d, j->m, j->A_aug + (size_t)b * j->N * dd,
                                                 j->B_aug + (size_t)b * j->N * dm, j->Q_aug + (size_t)b * j->N * dd,
                                                 j->R_inv + (size_t)b * (j->rinv_stride ? j->N : 1) * j->m * j->m,
                                                 j->rinv_stride, j->z0 + (size_t)b * j->d,
                                                 j->QT + (size_t)b * j->N * dd, j->J + (size_t)b * j->T_use,
                                                 HOP_JITTER, HOP_TRIES, NULL);
        } else {
            const int cap = j->opts->max_iter + 1;
            j->status[b] = hopo_ilqr_timeopt(j->sys, j->p, j->N, j->T_min, j->T_max, j->x0 + (size_t)b * n, j->U,
                                             j->xg + (size_t)b * n, j->u_ref, j->Q, j->R, j->Qf, j->w[b], j->wrap_mask,
                                             j->opts, j->X_out + (size_t)b * (j->N + 1) * n, j->U_out + (size_t)b * j->N * m,
                                             j->J_hist + (size_t)b * cap, j->T_hist + (size_t)b * cap, &j->n_hist[b],
                                             j->J + (size_t)b * j->T_max, &j->T_star[b], NULL);
        }
    }
    return NULL;
}

static int hopo_fan_out(int nthreads, int Bsz, const hopo_job *proto)
{
    if (nthreads < 1) nthreads = 1;
    if (nthreads > Bsz) nthreads = Bsz > 0 ? Bsz : 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * nthreads);
    hopo_job *jobs = (hopo_job *)malloc(sizeof(hopo_job) * nthreads);
    if (!th || !jobs) { free(th); free(jobs); return HOP_ERR_ALLOC; }
    for (int t = 0; t < nthreads; ++t) {
        jobs[t] = *proto;
        jobs[t].lo = (int)((long)Bsz * t / nthreads);
        jobs[t].hi = (int)((long)Bsz * (t + 1) / nthreads);
        if (t > 0) pthread_create(&th[t], NULL, hopo_worker, &jobs[t]);
    }
    hopo_worker(&jobs[0]);
    for (int t = 1; t < nthreads; ++t) pthread_join(th[t], NULL);
    free(th); free(jobs);
    return HOP_OK;
}

int hopo_select_from_x0_batch(int nthreads, int Bsz, int sys, const double *p, int N, int T_min, int T_max,
                              const double *x0, const double *U, const double *xg, const double *u_ref,
                              const double *Q, const double *R, const double *Qf, const double *w,
                              unsigned wrap_mask, int central, double *J, int *T_star, int *status)
{
    hopo_job j; memset(&j, 0, sizeof j);
    j.kind = 0; j.sys = sys; j.p = p; j.N = N; j.T_min = T_min; j.T_max = T_max; j.x0 = x0; j.U = U; j.xg = xg;
    j.u_ref = u_ref; j.Q = Q; j.R = R; j.Qf = Qf; j.w = w; j.wrap_mask = wrap_mask; j.central = central;
    j.J = J; j.T_star = T_star; j.status = status;
    return hopo_fan_out(nthreads, Bsz, &j);
}

int hopo_select_from_x0_batch_ex(int nthreads, int Bsz, int sys, const double *p, int N, int T_min, int T_max,
                                 const double *x0, const double *U, const double *xg, const double *u_ref,
                                 const double *Q, const double *R, const double *Qf, const double *w,
                                 unsigned wrap_mask, int central, int use_f80, double *J, int *T_star, int *status)
{
    hopo_job j; memset(&j, 0, sizeof j);
    j.kind = 0; j.sys = sys; j.p = p; j.N = N; j.T_min = T_min; j.T_max = T_max; j.x0 = x0; j.U = U; j.xg = xg;
    j.u_ref = u_ref; j.Q = Q; j.R = R; j.Qf = Qf; j.w = w; j.wrap_mask = wrap_mask; j.central = central;
    j.use_f80 = use_f80; j.J = J; j.T_star = T_star; j.status = status;
    return hopo_fan_out(nthreads, Bsz, &j);
}

/* hopo_select_fused over a batch of given linearisations: A [B][N][n][n], B [B][N][n][m], a_resid [B][N][n] or NULL (= 0),
 * X [B][N+1][n], U [B][N][m] (per instance), xg [B][n], w [B]. */
int hopo_select_fused_batch(int nthreads, int Bsz, int n, int m, int N, int T_min, int T_max, const double *A,
                            const double *B, const double *a_resid, const double *X, const double *U,
                            const double *xg, const double *u_ref, const double *Q, const double *R,
                            const double *Qf, const double *w, unsigned wrap_mask, int use_f80, double *J,
                            int *T_star, int *status)
{
    if (!dims_ok(n, m)) return HOP_ERR_ARG;
    hopo_job j; memset(&j, 0, sizeof j);
    j.kind = 3; j.d = n; j.m = m; j.N = N; j.T_min = T_min; j.T_max = T_max; j.A = A; j.B = B; j.a_resid = a_resid;
    j.X = X; j.U = U; j.xg = xg; j.u_ref = u_ref; j.Q = Q; j.R = R; j.Qf = Qf; j.w = w; j.wrap_mask = wrap_mask;
    j.use_f80 = use_f80; j.J = J; j.T_star = T_star; j.status = status;
    return hopo_fan_out(nthreads, Bsz, &j);
}

int hopo_propagator_batch(int nthreads, int Bsz, int N, int T_use, int d, int m, const double *A_aug,
                          const double *B_aug, const double *Q_aug, const double *R_inv, long rinv_stride,
                          const double *z0, const double *QT, double *J, int *status)
{
    if (d < 1 || d > HOP_MAXD || m < 1 || m > HOP_MAXD || T_use > N) return HOP_ERR_ARG;
    if (rinv_stride != 0 && rinv_stride != (long)m * m) return HOP_ERR_ARG;
    hopo_job j; memset(&j, 0, sizeof j);
    j.kind = 1; j.N = N; j.T_use = T_use; j.d = d; j.m = m; j.A_aug = A_aug; j.B_aug = B_aug; j.Q_aug = Q_aug;
    j.R_inv = R_inv; j.rinv_stride = rinv_stride; j.z0 = z0; j.QT = QT; j.J = J; j.status = status;
    return hopo_fan_out(nthreads, Bsz, &j);
}

int hopo_ilqr_timeopt_batch(int nthreads, int Bsz, int sys, const double *p, int N, int T_min, int T_max,
                            const double *x0, const double *U_init, const double *xg, const double *u_ref,
                            const double *Q, const double *R, const double *Qf, const double *w,
                            unsigned wrap_mask, const hopo_ilqr_opts *opts, double *X_out, double *U_out,
                            double *J_hist, int *T_hist, int *n_hist, double *J_curve, int *T_star,
                            int *status)
{
    hopo_job j; memset(&j, 0, sizeof j);
    j.kind = 2; j.sys = sys; j.p = p; j.N = N; j.T_min = T_min; j.T_max = T_max; j.x0 = x0; j.U = U_init; j.xg = xg;
    j.u_ref = u_ref; j.Q = Q; j.R = R; j.Qf = Qf; j.w = w; j.wrap_mask = wrap_mask; j.opts = opts;
    j.X_out = X_out; j.U_out = U_out; j.J_hist = J_hist; j.T_hist = T_hist; j.n_hist = n_hist; j.J = J_curve;
    j.T_star = T_star; j.status = status;
    return hopo_fan_out(nthreads, Bsz, &j);
}
