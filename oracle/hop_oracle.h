/* hop_oracle.h -- CPU ORACLE for the HOP horizon-selection hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline /
 * `--impl reference` legs may load this library; the product path (time-opt-ilqr_b200/) never
 * does and has no CPU fallback.
 *
 * Plain-C restatement of the reference numpy algorithm (dmmsjtu-umich/time-opt-ilqr); each
 * function cites the reference file:line it follows (see hop_oracle.c / hop_la.inc).
 * Parity pin: the .npz files under tests/golden are produced by tests/golden/make_golden.py, which imports the
 * real reference from /root/reference and records its inputs/outputs; tests/test_oracle.py checks
 * this oracle against them.  The reference itself ships no tests or golden vectors (SURVEY.md s.4).
 *
 * Conventions: fp64, row-major, per-instance layouts [N][r][c]; `wrap_mask` bit i set <=> state
 * index i is in the reference's wrap_idx list; `Qf` is as_terminal_weight(alpha, n) (utils.py:49-62)
 * materialised by the caller.
 */
#ifndef HOP_ORACLE_H
#define HOP_ORACLE_H

#ifdef __cplusplus
extern "C" {
#endif

enum {
    HOP_OK = 0,
    HOP_ERR_NONFINITE = 1, /* reference raises FloatingPointError (utils.py:40-42) */
    HOP_ERR_LINALG = 2,    /* reference raises np.linalg.LinAlgError              */
    HOP_ERR_ALLOC = 3,
    HOP_ERR_ARG = 4
};

enum { HOP_SYS_DOUBLE_INTEGRATOR = 0, HOP_SYS_CARTPOLE = 1, HOP_SYS_QUADROTOR = 2, HOP_SYS_SEGWAY = 3 };

/* ---- utils.py ---- */
int hopo_chol_inv(int d, const double *A, double *X, double jitter, int max_tries, int *info);
int hopo_chol_solve(int d, int c, const double *A, const double *B, double *X, double jitter, int max_tries);
double hopo_angle_normalize(double a);
void hopo_wrap_error(int n, double *e, unsigned wrap_mask);

/* ---- systems.py ---- */
int hopo_sys_dims(int sys, int *n, int *m);
void hopo_dynamics(int sys, const double *p, const double *x, const double *u, double *xn);

/* ---- solver.py primitives ----
 * Every entry point below that takes the state / control dimensions n, m (not a system id) needs
 * 1 <= n <= 15 and 1 <= m <= 16 and returns HOP_ERR_ARG otherwise (hopo_cost_timeopt_true: NaN). */
void hopo_rollout(int sys, const double *p, int N, const double *x0, const double *U, double *X,
                  double max_state_norm);
double hopo_cost_timeopt_true(int n, int m, const double *X, const double *U, const double *xg,
                              const double *u_ref, const double *Q, const double *R, const double *Qf,
                              double w, int T_star, unsigned wrap_mask);
int hopo_backward_pass(int n, int m, const double *A, const double *B, const double *X, const double *U,
                       const double *xg, const double *u_ref, const double *Q, const double *R,
                       const double *Qf, int T_star, double lm_lambda, unsigned wrap_mask,
                       double *k_out, double *K_out, int *ok);
int hopo_forward_linesearch(int sys, const double *p, int N, const double *X, const double *U,
                            const double *xg, const double *u_ref, const double *Q, const double *R,
                            const double *Qf, double w, int T_star, const double *k_list,
                            const double *K_list, unsigned wrap_mask, double *X_new, double *U_new,
                            double *J_out, int *accepted);
int hopo_bruteforce_all_Jt(int n, int m, const double *A, const double *B, const double *X, const double *U,
                           const double *xg, const double *u_ref, const double *Q, const double *R,
                           const double *Qf, double w, int T_max, double lm_lambda, unsigned wrap_mask,
                           double *J);

/* ---- linearization.py ---- */
void hopo_linearize(int sys, const double *p, int N, const double *X, const double *U, int central,
                    double epsx, double epsu, double relx, double relu, double *A, double *B);
void hopo_affine_residuals(int sys, const double *p, int N, const double *X, const double *U, double *a);

/* ---- augmented.py ---- */
int hopo_build_augmented(int n, int m, int N, const double *A, const double *B, const double *a,
                         const double *X, const double *U, const double *xg, const double *u_ref,
                         const double *Q, const double *R, double w, unsigned wrap_mask, double q_reg,
                         double rho_reg, double *A_aug, double *B_aug, double *Q_aug, double *R_inv);
int hopo_build_terminal(int n, int N, const double *X, const double *xg, const double *Qf,
                        unsigned wrap_mask, double rho_reg, double *QT);

/* ---- horizon_selection.py ----
 * R_inv is [m][m] (rinv_stride = 0: the R_inv_cached argument) or [N][m][m] (rinv_stride = m*m: chol_inv(R_list[k])
 * per step, horizon_selection.py:60-61); hopo_propagator_batch: [B][m][m] or [B][N][m][m]. */
int hopo_propagator_all_Jt_f64(int T_use, int d, int m, const double *A_aug, const double *B_aug,
                               const double *Q_aug, const double *R_inv, long rinv_stride, const double *z0,
                               const double *QT, double *J, double jitter, int max_tries, long *retries);
int hopo_propagator_all_Jt_f80(int T_use, int d, int m, const double *A_aug, const double *B_aug,
                               const double *Q_aug, const double *R_inv, long rinv_stride, const double *z0,
                               const double *QT, double *J, double jitter, int max_tries, long *retries);
/* solver.py:522,590: int(np.argmin(J[T_min-1:T_max]) + T_min)  (first minimum; NaN wins) */
int hopo_argmin_window(const double *J, int T_min, int T_max);

/* ---- composed paths (what bench.py's CPU legs time) ---- */
/* a6+a8+a9+a10..a13 for one instance: (A,B,X,U) -> J[T_max], T*.  a_resid may be NULL (=> computed
 * from the dynamics when sys >= 0, else taken as zero). */
int hopo_select_fused(int sys, const double *p, int n, int m, int N, int T_min, int T_max,
                      const double *A, const double *B, const double *a_resid, const double *X,
                      const double *U, const double *xg, const double *u_ref, const double *Q,
                      const double *R, const double *Qf, double w, unsigned wrap_mask, int use_f80,
                      double *J, int *T_star);
/* rollout + FD linearisation + hopo_select_fused from x0 (S1 workload, SURVEY.md s.8d). */
int hopo_select_from_x0(int sys, const double *p, int N, int T_min, int T_max, const double *x0,
                        const double *U, const double *xg, const double *u_ref, const double *Q,
                        const double *R, const double *Qf, double w, unsigned wrap_mask, int central,
                        double *J, int *T_star);
/* pthread fan-out of the two calls above over a batch (per-instance x0/xg/w; shared case constants) */
int hopo_select_from_x0_batch(int nthreads, int Bsz, int sys, const double *p, int N, int T_min, int T_max,
                              const double *x0, const double *U, const double *xg, const double *u_ref,
                              const double *Q, const double *R, const double *Qf, const double *w,
                              unsigned wrap_mask, int central, double *J, int *T_star, int *status);
/* same with the selection sweep optionally in x87 extended precision (use_f80; noise accounting only) */
int hopo_select_from_x0_batch_ex(int nthreads, int Bsz, int sys, const double *p, int N, int T_min, int T_max,
                                 const double *x0, const double *U, const double *xg, const double *u_ref,
                                 const double *Q, const double *R, const double *Qf, const double *w,
                                 unsigned wrap_mask, int central, int use_f80, double *J, int *T_star, int *status);
/* hopo_select_fused over a batch of GIVEN linearisations (per-instance A, B, a_resid or NULL, X, U, xg, w) */
int hopo_select_fused_batch(int nthreads, int Bsz, int n, int m, int N, int T_min, int T_max, const double *A,
                            const double *B, const double *a_resid, const double *X, const double *U,
                            const double *xg, const double *u_ref, const double *Q, const double *R,
                            const double *Qf, const double *w, unsigned wrap_mask, int use_f80, double *J,
                            int *T_star, int *status);
int hopo_propagator_batch(int nthreads, int Bsz, int N, int T_use, int d, int m, const double *A_aug,
                          const double *B_aug, const double *Q_aug, const double *R_inv, long rinv_stride,
                          const double *z0, const double *QT, double *J, int *status);

/* solver.py:449-765  ilqr_timeopt(method="propagator") */
typedef struct {
    int max_iter;
    double lm_init;
    int use_central_diff;
    int use_f80_select; /* 0: fp64 selection (the reference's arithmetic) */
} hopo_ilqr_opts;
int hopo_ilqr_timeopt(int sys, const double *p, int N, int T_min, int T_max, const double *x0,
                      const double *U_init, const double *xg, const double *u_ref, const double *Q,
                      const double *R, const double *Qf, double w, unsigned wrap_mask,
                      const hopo_ilqr_opts *opts, double *X_out, double *U_out, double *J_hist,
                      int *T_hist, int *n_hist, double *J_curve, int *T_star, int *n_outer);
int hopo_ilqr_timeopt_batch(int nthreads, int Bsz, int sys, const double *p, int N, int T_min, int T_max,
                            const double *x0, const double *U_init, const double *xg, const double *u_ref,
                            const double *Q, const double *R, const double *Qf, const double *w,
                            unsigned wrap_mask, const hopo_ilqr_opts *opts, double *X_out, double *U_out,
                            double *J_hist, int *T_hist, int *n_hist, double *J_curve, int *T_star,
                            int *status);

const char *hopo_version(void);

#ifdef __cplusplus
}
#endif
#endif
