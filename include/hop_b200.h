/* hop_b200.h -- C-ABI of libhop_b200.so: the B200-native HOP horizon-selection hot path.
 *
 * The reference (dmmsjtu-umich/time-opt-ilqr) is pure Python and has no FFI; its boundary for this
 * path is the Python function API.  Each entry point below names the reference function(s) it
 * replaces (file:line).  The host-side mirror of those Python signatures lives in
 * time-opt-ilqr_b200/dropin/ and calls these symbols through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - fp64, row-major, batch-major: [B][N][rows][cols].  Unless an entry point says "host", every
 *     pointer is a DEVICE pointer owned by the caller; nothing is retained after the call returns.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are asynchronous
 *     with respect to the host except the *_host_* variants, which synchronise before returning.
 *   - Return value: 0 on success, otherwise a cudaError_t value or HOP_E_* (< 0); the message is
 *     available from hop_last_error_string().  Kernels never trap: per-instance numerical outcomes
 *     are reported in `status[b]`:
 *         low byte  0 = ok, 1 = non-finite input to a chol_inv (reference: FloatingPointError,
 *                   utils.py:40-42,75), 2 = singular LU fallback (reference: LinAlgError, utils.py:93)
 *         bit 8     some Cholesky attempt failed and the jitter ladder was climbed (utils.py:81-88)
 *         bit 9     the LU fallback of utils.py:90-93 was taken
 *         bit 10    HOP_MODE_VERIFIED only: the instance was re-evaluated in HOP_MODE_EXACT (see below)
 *   - wrap_mask bit i  <=>  state index i is in the reference's wrap_idx list (utils.py:131-137).
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef HOP_B200_H
#define HOP_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define HOP_ABI_VERSION 1

enum { HOP_E_BADARG = -1, HOP_E_UNSUPPORTED_DIMS = -2, HOP_E_NO_DEVICE = -3, HOP_E_WORKSPACE = -4 };

/* status word */
enum { HOP_ST_OK = 0, HOP_ST_NONFINITE = 1, HOP_ST_LINALG = 2, HOP_ST_ERRMASK = 0xff,
       HOP_ST_FLAG_RETRY = 0x100, HOP_ST_FLAG_LU = 0x200, HOP_ST_FLAG_REEVALUATED = 0x400 };

/* selection variants (all compute the reference's function J(T), T*; see DESIGN.md s.4)
 *   EXACT: the PARITY mode.  The reference's operation order with individually rounded IEEE operations: Cholesky in
 *          LAPACK dpotf2 order -> two substitutions for the inverse (utils.py:83-85), numpy's left-to-right products,
 *          _sym exactly where the reference has it, no FMA contraction.  On identical inputs J(T) is bit-identical to
 *          the plain-C restatement in oracle/ (asserted by the tests), hence T* too.  One warp per problem, blocks in
 *          shared memory, any 1 <= d, m <= 16.  ~5x slower than FAST.
 *   FAST : the throughput mode (bench default).  Fused entry points with n = 12: closed-form block inverses for E_k
 *          and X_t, pivot-only evaluation of J(t) = 0.5 / pivot_n(X0), software-pipelined Gauss-Jordan sweeps in DMMA
 *          register fragments.  Elsewhere identical to GJ.  Differs from EXACT by rounding only: <= 1e-9 relative on
 *          well-conditioned problems (S2), ~1e-7 on the J(T) window of the rank-deficient augmented problems, where
 *          the reference itself is only reproducible to ~5e-8 across BLAS builds (SURVEY.md s.9).
 *   GJ   : every augmented block materialised (in registers) and inverted by an in-place Gauss-Jordan sweep with FMA
 *          (same jitter-ladder decisions as Cholesky: the sweep pivots are the squared Cholesky pivots).  The cold path
 *          of FAST and the kernels behind hop_select_f64 in FAST mode; instantiated (d, m) only.
 *   SCAN : hop_select_f64 and hop_select_fused_f64, (d, m) = (12,4) / (13,4): the prefix composition as a chunked parallel scan over the
 *          horizon (one CTA of 8 warps per problem; latency 2T/8 + 7 instead of T steps for ~2x the prefix work) --
 *          for SMALL batches.  Re-association changes the rounding (<= 1e-9 on well-conditioned problems; unsafe on
 *          ill-conditioned ones such as the cartpole embedding, SURVEY.md s.9), so it is opt-in.
 *   FP32 : hop_select_f64 only: the EXACT sweep in IEEE single precision (inputs converted on load, J written as double).
 *          Tolerance on S2 (well conditioned): J within 1e-4 relative, T* reproduced on >= 99 % of instances (the
 *          mismatches are argmin gaps below the fp32 noise; measured in tests/ and DESIGN.md).  Not for the augmented
 *          problems: their 1e-9 jitter and 1e-12 regularisation are below fp32 resolution.
 *   VERIFIED: fused entry points and hop_ilqr_timeopt_f64 (hop_select_f64 refuses it: at the LQR boundary the caller gives
 *          the tolerance, hop_select_verified_f64): FAST, then every instance whose
 *          T* could depend on the implementation is recomputed in EXACT.  Per instance:
 *            1. the FAST selection, unchanged (same kernels, same routing, same bits);
 *            2. near-tie scan of the curve FAST returned (J_out, the curve the kernel minimised): with J1 = J(T*) and
 *               gap = (min over t != T* in [T_min, T_max] of J(t) - J1) / |J1|  (oracle/census.py argmin_gap), the instance
 *               is marked when  gap < tol  (the tie tolerance of the state dimension n, below),  or the window holds a
 *               NaN or +-Inf,  or status != 0,  or the scan's own argmin (first minimum, first NaN, as np.argmin)
 *               differs from Tstar_out (defensive; never seen); instances masked by the HOP-DDP `done` word are not scanned;
 *            3. every marked instance is recomputed by the EXACT kernel, which overwrites its whole J_out row, Tstar_out,
 *               Jstar_out and status, and then sets HOP_ST_FLAG_REEVALUATED in status.
 *          So re-evaluated instances carry EXACT's outputs bit for bit plus bit 10, all others FAST's outputs unchanged with
 *          status 0.  T* and the low byte of status equal EXACT's on EVERY instance PROVIDED FAST's relative distance to
 *          EXACT at the competing horizons stays below tol / 2: an unmarked instance then has the same
 *          argmin in both curves.  That is a tolerance argument backed by measurement (below), not a proof.  The outputs
 *          are deterministic: the order in which marked instances are collected changes no bit.  Scratch (B + 1 ints) is
 *          allocated stream-ordered on the caller's stream; the host never waits for the device.
 *          HOP_VERIFY_TIE_TOL is calibrated on the quadrotor embedding (n = 12): over the 65 536 S1 instances FAST is at
 *          most 5.5e-9 relative from EXACT at T* (DESIGN.md s.6), an 18x margin on tol / 2; the reference's own argmin gap is
 *          below 1e-7 on 2.4 % of its 4 096 golden instances.  Measured on a B200 (1000 W) over the S1 batch: FAST within
 *          6.0e-9 of EXACT at its two best horizons and at EXACT's T*, 2.9 % of the instances re-evaluated, smallest ratio of
 *          FAST's gap to that distance over the other instances 28.9 (tools/verified_ab.py, profiles/r3_verified_ab.jsonl).
 *          Per state dimension n of the fused forms (calibrated on the same card; FAST's distance to EXACT at its two best
 *          horizons and at EXACT's T*, over 300 / 900 / 3 000 instances, i.e. every FAST routing branch):
 *            n = 12 (quadrotor)          HOP_VERIFY_TIE_TOL = 1e-7 (above).
 *            n = 2  (double integrator)  HOP_VERIFY_TIE_TOL_N2 = 1e-6: distance <= 4.6e-8, so 1e-7 would leave a margin of
 *                                        only 1.1x on tol / 2; 1e-6 re-evaluates 0 - 0.2 % of the instances.
 *            n = 4  refused (HOP_E_UNSUPPORTED_DIMS): the dimension is shared by the Segway and the cartpole embeddings.  The
 *                                        cartpole embedding (ill-conditioned, SURVEY.md s.9) has FAST-vs-EXACT T* differences
 *                                        on 11 - 14 % of its instances with FAST gaps up to 2.3e-4; a tolerance of 1e-4 already
 *                                        re-evaluates 80 % and still misses some.  (Segway alone: differences on <= 0.5 %,
 *                                        FAST gaps up to 7.6e-7.)  Use HOP_MODE_EXACT there. */
enum { HOP_MODE_EXACT = 0, HOP_MODE_FAST = 1, HOP_MODE_SCAN = 2, HOP_MODE_GJ = 3, HOP_MODE_FP32 = 4, HOP_MODE_VERIFIED = 5 };
#define HOP_VERIFY_TIE_TOL 1e-7
#define HOP_VERIFY_TIE_TOL_N2 1e-6

/* device dynamics registry (systems.py closures cannot run on the GPU) */
enum { HOP_SYS_DOUBLE_INTEGRATOR = 0, /* systems.py:28-50   params [dt]                               */
       HOP_SYS_CARTPOLE = 1,          /* systems.py:57-112  params [dt,g,m_pole,length,total_mass,pml] */
       HOP_SYS_QUADROTOR = 2,         /* systems.py:119-230 params [dt,m,g,Ix,Iy,Iz,1/Ix,1/Iy,1/Iz,kv,kw,cos_min,omg_max,norm_max] */
       HOP_SYS_SEGWAY = 3 };          /* systems.py:303-349 params [dt,A_tau,A_th,B_tau,B_th]           */
#define HOP_NPARAMS 16

int hop_abi_version(void);
const char *hop_version(void);
const char *hop_last_error_string(void);
/* number of visible CUDA devices (0 => every compute call returns HOP_E_NO_DEVICE) */
int hop_device_count(void);
/* 1 if (d, m) is an instantiated augmented-dimension / control-dimension pair of the FAST / GJ / SCAN kernels
 * ((3,1) (4,2) (5,1) (12,4) (13,4)); HOP_MODE_EXACT and HOP_MODE_FP32 take any 1 <= d, m <= 16 */
int hop_select_supported(int d, int m);
/* same question for a given mode (HOP_MODE_VERIFIED: the FAST pairs whose state dimension n = d - 1 has a calibrated tie
 * tolerance, i.e. (3,1) and (13,4), for the fused forms; hop_select_verified_f64 takes every FAST pair) */
int hop_select_supported_mode(int d, int m, int mode);

/* horizon_selection.py:36-86 propagator_all_Jt_aug (+ solver.py:522,590 argmin), batched.
 *   A_aug [B][N][d][d], B_aug [B][N][d][m], Q_aug [B][N][d][d], QT [B][N][d][d] (QT[t-1] = terminal block
 *   of horizon t), R_inv [B][m][m] (the R_inv_cached argument; rinv_step_stride = 0) or [B][N][m][m]
 *   (chol_inv(R_list[k]) per step; rinv_step_stride = m*m), z0 [B][d].
 *   w_explicit: NULL, or [B] -- argmin is then taken over J(t) + w*t (SURVEY.md s.8d "S2"); J_out is
 *   always the raw curve the reference returns.
 *   Outputs: J_out [B][T_max] (index t-1), Tstar_out [B] = argmin over t in [T_min, T_max] (first
 *   minimum, NaN wins, as np.argmin), Jstar_out [B], status [B]. */
int hop_select_f64(int B, int N, int d, int m, int T_min, int T_max,
                   const double *A_aug, const double *B_aug, const double *Q_aug, const double *R_inv,
                   long rinv_step_stride, const double *z0, const double *QT, const double *w_explicit, int mode,
                   double *J_out, int *Tstar_out, double *Jstar_out, int *status, void *stream);

/* HOP_MODE_VERIFIED at the LQR boundary, with a tie tolerance the CALLER chooses.  Arguments and outputs are those of
 * hop_select_f64; `mode` is replaced by `tie_tol` (finite, > 0).  (d, m): the FAST pairs of hop_select_supported, else
 * HOP_E_UNSUPPORTED_DIMS.  Argument errors are reported before any device is needed.  Per instance:
 *   1. the FAST selection of hop_select_f64, unchanged (same routing and kernels, same bits);
 *   2. the near-tie scan of HOP_MODE_VERIFIED on the curve the kernel minimised: v(t) = J(t) + w t, evaluated as
 *      add_rn(J, mul_rn(w, t)) like the EXACT body, when w_explicit is given, J(t) otherwise; marked when the relative gap
 *      is below tie_tol, when the window holds a NaN or +-Inf, when status != 0, or when the scan's argmin differs from
 *      Tstar_out.  The pipelined FAST kernels (d = 12, 13) may contract J + w t into an FMA, so the last check also fires
 *      on some last-bit differences of v: that only adds re-evaluations, it never hides a tie;
 *   3. every marked instance is recomputed by the EXACT kernel (whole J_out row, Tstar_out, Jstar_out, status) and gets
 *      HOP_ST_FLAG_REEVALUATED.
 * T* and the low byte of status then equal HOP_MODE_EXACT's on every instance PROVIDED FAST stays within tie_tol / 2 of EXACT
 * (relative, on v) at the competing horizons of the caller's input family.  The conditioning of LQR-boundary inputs belongs to
 * the caller, so the library cannot fix one tolerance: choosing it is the caller's responsibility.  Deterministic; scratch of
 * B + 1 ints, stream-ordered on `stream`; the host never waits.  Measured guidance (B200, tools/verified_ab.py,
 * profiles/r4_verified_lqr_ab.jsonl; FAST's largest relative distance to EXACT on v at its two best horizons and at EXACT's T*):
 *   S2 (tests/run_configs.py configuration 5: d = 4, 12, 13, N = 128, with w_explicit): distance <= 2.7e-14, so tie_tol = 1e-12
 *     leaves an 18x margin on tie_tol / 2; at 1e-10 none of 262 144 (d = 4) / 65 536 (d = 12, 13) instances is re-evaluated and
 *     VERIFIED takes FAST's time (d = 13: 51.4 ms against EXACT's 674 ms); 1e-7 would re-evaluate 0.02 %.
 *   Quadrotor embedding built at the boundary (hop_build_augmented_f64 / hop_build_terminal_f64 on S1 linearisations, 16 384
 *     instances): distance <= 4.7e-9; tie_tol = 1e-7 (10.7x margin) re-evaluates 2.8 %: FAST 16.2 ms, VERIFIED 34.3 ms,
 *     EXACT 196 ms.  1e-8 would leave a margin of 1.07x.
 *   Other families (ill-conditioned embeddings such as the cartpole's, see HOP_MODE_VERIFIED above): not measured;
 *     measure FAST against EXACT on a sample of the family before choosing the tolerance. */
int hop_select_verified_f64(int B, int N, int d, int m, int T_min, int T_max,
                            const double *A_aug, const double *B_aug, const double *Q_aug, const double *R_inv,
                            long rinv_step_stride, const double *z0, const double *QT, const double *w_explicit,
                            double tie_tol, double *J_out, int *Tstar_out, double *Jstar_out, int *status, void *stream);

/* Fused form: augmented.py:10-60 build_augmented_sequence_QR + augmented.py:63-87
 * build_terminal_aug_list + horizon_selection.py:36-86 + argmin in one kernel; the (n+1)^2 blocks are
 * built in shared memory and never written to HBM.
 *   A [B][N][n][n], Bm [B][N][n][m] (linearisation), a_resid [B][N][n] or NULL (= 0, which is what
 *   linearization.py:269-270 yields on a consistent rollout), X [B][N+1][n], U [B][N][m]
 *   (u_batch_stride = N*m) or one shared U [N][m] (u_batch_stride = 0), xg [B][n], w [B]; shared case constants u_ref [m], Q [n][n], R [m][m], Qf [n][n] (=
 *   as_terminal_weight(alpha), utils.py:49-62). */
int hop_select_fused_f64(int B, int N, int n, int m, int T_min, int T_max,
                         const double *A, const double *Bm, const double *a_resid, const double *X,
                         const double *U, long u_batch_stride, const double *xg, const double *w, const double *u_ref,
                         const double *Q, const double *R, const double *Qf, unsigned wrap_mask,
                         double q_reg, double rho_reg, int mode,
                         double *J_out, int *Tstar_out, double *Jstar_out, int *status, void *stream);

/* solver.py:42-62 rollout, batched: X [B][N+1][n] from x0 [B][n], U [B][N][m]
 * (u_batch_stride = N*m for per-instance controls, 0 when all instances share one U [N][m]).
 * params: HOP_NPARAMS doubles on the HOST. */
int hop_rollout_f64(int B, int sys, const double *params_host, int N, const double *x0, const double *U,
                    long u_batch_stride, double max_state_norm, double *X, void *stream);

/* linearization.py:216-262 (central = 0) / :177-211 (central = 1), batched: A [B][N][n][n], Bm [B][N][n][m]. */
int hop_linearize_f64(int B, int sys, const double *params_host, int N, const double *X, const double *U,
                      long u_batch_stride, int central, double epsx, double epsu, double relx, double relu,
                      double *A, double *Bm, void *stream);

/* Whole selection from initial states (SURVEY.md s.8d workload "S1"): rollout -> forward/central FD
 * linearisation -> fused selection.  `workspace` must hold hop_select_from_x0_workspace_bytes(...). */
unsigned long long hop_select_from_x0_workspace_bytes(int B, int N, int n, int m);
int hop_select_from_x0_f64(int B, int sys, const double *params_host, int N, int T_min, int T_max,
                           const double *x0, const double *U, long u_batch_stride, const double *xg,
                           const double *w, const double *u_ref, const double *Q, const double *R,
                           const double *Qf, unsigned wrap_mask, int central, int mode,
                           void *workspace, unsigned long long workspace_bytes,
                           double *J_out, int *Tstar_out, double *Jstar_out, int *status, void *stream);

/* Same, HOST buffers in and out (x0, U, xg, w and the outputs live in host memory; the case
 * constants too).  Copies, kernels and the final device->host read are issued on one internal
 * stream and the call returns after they complete.  J_out may be NULL (only T*, J* wanted). */
int hop_select_from_x0_host_f64(int B, int sys, const double *params_host, int N, int T_min, int T_max,
                                const double *x0, const double *U, long u_batch_stride, const double *xg,
                                const double *w, const double *u_ref, const double *Q, const double *R,
                                const double *Qf, unsigned wrap_mask, int central, int mode,
                                double *J_out, int *Tstar_out, double *Jstar_out, int *status);

/* utils.py:69-93 chol_inv / utils.py:96-120 chol_solve over a batch of d x d matrices (d <= 16), one thread
 * per matrix, through the same Cholesky route as the reference (L, L^-1, L^-T L^-1; jitter ladder; LU
 * fallback for the inverse, none for the solve).  status as above. */
int hop_chol_inv_f64(int B, int d, const double *A, double *X, double jitter, int max_tries, int *status, void *stream);
int hop_chol_solve_f64(int B, int d, int c, const double *A, const double *Bm, double *X, double jitter, int max_tries,
                       int *status, void *stream);

/* linearization.py:269-270 compute_affine_residuals: a_out [B][N][n] = F(X_k, U_k) - X_{k+1}. */
int hop_affine_residuals_f64(int B, int sys, const double *params_host, int N, const double *X, const double *U,
                             long u_batch_stride, double *a_out, void *stream);

/* augmented.py:10-60 build_augmented_sequence_QR (blocks materialised in HBM: A_aug [B][N][d][d],
 * B_aug [B][N][d][m], Q_aug [B][N][d][d]; R_inv is hop_chol_inv_f64 of sym(R)) and augmented.py:63-87
 * build_terminal_aug_list (QT [B][N][d][d], QT[t-1] from X[t]).  a_resid may be NULL (= 0). */
int hop_build_augmented_f64(int B, int N, int n, int m, const double *A, const double *Bm, const double *a_resid,
                            const double *X, const double *U, long u_batch_stride, const double *xg, const double *w,
                            const double *u_ref, const double *Q, unsigned wrap_mask, double q_reg, double rho_reg,
                            double *A_aug, double *B_aug, double *Q_aug, void *stream);
int hop_build_terminal_f64(int B, int N, int n, const double *X, const double *xg, const double *Qf, unsigned wrap_mask,
                           double rho_reg, double *QT, void *stream);

/* solver.py:65-105 cost_timeopt_true, batched: J_out[b] at the per-instance horizon T_star[b] (device int).
 * In this and the two entry points below a T_star[b] > N is clamped to N on the device (the trajectories hold N steps);
 * T_star[b] <= 0 behaves as in the reference (cost = inf; backward pass: ok = 0). */
int hop_cost_f64(int B, int N, int n, int m, const double *X, const double *U, const double *xg, const double *w,
                 const double *u_ref, const double *Q, const double *R, const double *Qf, unsigned wrap_mask,
                 const int *T_star, double *J_out, void *stream);

/* solver.py:293-358 bruteforce_all_Jt_backward_expansion, batched: J_out [B][T_max], J_out[b][T-1] = V0[0] of a full
 * Riccati sweep T -> 0 (it already contains w T).  One warp per (instance, T): O(T_max^2 n^3) per instance -- the
 * reference's baseline-1 curve, kept as an independent on-device check of the propagator.  status [B]: 0, or the
 * chol_solve failure of some horizon (1 FloatingPointError, 2 LinAlgError; that horizon's J is NaN). */
int hop_bruteforce_jt_f64(int B, int N, int n, int m, int T_max, const double *A, const double *Bm, const double *X,
                          const double *U, long u_batch_stride, const double *xg, const double *w, const double *u_ref,
                          const double *Q, const double *R, const double *Qf, unsigned wrap_mask, double lm_lambda,
                          double *J_out, int *status, void *stream);

/* solver.py:156-230 backward_pass_truncated followed by solver.py:233-286 forward_linesearch_fixedT, batched,
 * at per-instance horizons T_star[b] and Levenberg-Marquardt weights lm[b].
 *   k_out [B][N][m], K_out [B][N][m][n] (rows >= T_star[b] untouched), ok_out [B] (0 = the reference's
 *   `return None, None, False`), err_out [B] (non-zero = chol_solve raised: 1 FloatingPointError, 2 LinAlgError),
 *   X_new [B][N+1][n], U_new [B][N][m], J_new [B], accepted [B]. */
int hop_backward_linesearch_f64(int B, int sys, const double *params_host, int N, const double *A, const double *Bm,
                                const double *X, const double *U, const double *xg, const double *w, const double *u_ref,
                                const double *Q, const double *R, const double *Qf, unsigned wrap_mask, const int *T_star,
                                const double *lm, double *k_out, double *K_out, int *ok_out, int *err_out, double *X_new,
                                double *U_new, double *J_new, int *accepted, void *stream);

/* solver.py:233-286 forward_linesearch_fixedT alone, with caller-provided gains k_list [B][N][m],
 * K_list [B][N][m][n] (rows >= T_star[b] ignored); ok [B] or NULL masks instances to skip: a skipped instance gets
 * accepted[b] = 0 and keeps X_new, U_new and J_new as the caller left them. */
int hop_linesearch_f64(int B, int sys, const double *params_host, int N, const double *X, const double *U, const double *xg,
                       const double *w, const double *u_ref, const double *Q, const double *R, const double *Qf,
                       unsigned wrap_mask, const int *T_star, const double *k_list, const double *K_list, const int *ok,
                       double *X_new, double *U_new, double *J_new, int *accepted, void *stream);

/* solver.py:449-765 ilqr_timeopt(method="propagator"), batched over instances (x0, xg, w); the whole
 * per-instance state machine (warm start, accept/reject, LM schedule, stop rule) runs on the device.
 *   U_init [B][N][m] or NULL (= tile(u_ref), solver.py:480-481).
 *   Outputs: X [B][N+1][n], U [B][N][m] (final trajectories), J_hist/T_hist [B][max_iter+1] with n_hist [B]
 *   valid entries, J_curve [B][T_max] (last selection curve), T_star [B] (= T_hist[-1] or T_bar), status [B]
 *   (low byte != 0: the reference would have raised -> run_suite "crash"), *iters_run_host (host int, may be NULL),
 *   timers_host (host double[4] or NULL): device seconds spent in linearize / select / backward / forward, the
 *   keys of the reference's `timers` dict (solver.py:497).
 *   The call returns after the stream has drained.  Inside, the host never waits for the device between outer iterations:
 *   the early exit (every instance stopped) is decided one iteration late on an asynchronously copied counter. */
unsigned long long hop_ilqr_workspace_bytes(int B, int N, int n, int m);
int hop_ilqr_timeopt_f64(int B, int sys, const double *params_host, int N, int T_min, int T_max, const double *x0,
                         const double *U_init, const double *xg, const double *w, const double *u_ref, const double *Q,
                         const double *R, const double *Qf, unsigned wrap_mask, int max_iter, double lm_init, int central,
                         int mode, void *workspace, unsigned long long workspace_bytes, double *X, double *U,
                         double *J_hist, int *T_hist, int *n_hist, double *J_curve, int *T_star, int *status,
                         int *iters_run_host, double *timers_host, void *stream);

/* Test hook: selects the quadrotor finite-difference kernel (0 = thread per step [default], 2 = the generic kernel; any
 * other value is ignored); returns the previous value.  Both produce identical bits (tests/test_gpu_parity.py). */
int hop_test_set_linearize_variant(int variant);
/* Test hook: smallest batch hop_select_f64 routes to the thread-per-problem kernel (d <= 5).  -1 = the built-in defaults
 * (d <= 4: every batch; d = 5: B >= 16384), >= 0 = that threshold for every d (0 = always),
 * < -1 = query only.  Below the threshold the lane-group kernel runs; the two produce identical bits.  Returns the
 * previous value. */
long hop_test_set_tpp_min_batch(long min_batch);
/* Test hook: hop_select_f64 for d in {12, 13}: 1 = the input-only inversions E_k = chol_inv(Q_k), X_t = chol_inv(QT_t) run
 * in a parallel pre-pass (k_preinvert), 0 = inside the sequential kernel, -1 = pre-pass for B <= 1024 only [default]; identical
 * bits.  Returns the previous value. */
int hop_test_set_generic_pre(int on);
/* Test hook: hop_select_f64 for d in {12, 13}: 1 [default] = DIAGONAL input blocks Q_k / QT_t are inverted element-wise (what the
 * Gauss-Jordan sweep of a diagonal matrix computes anyway), 0 = by the sweep like any other block; identical bits.  Returns the
 * previous value. */
int hop_test_set_generic_diag(int on);
/* Test hook: fused selection kernel of the small systems (n <= 4).  0 [default] = by batch size: up to 592 instances one
 * problem per CTA as a warp-specialised pipeline (stage / prefix / query warps, one matrix element per lane), up to 1024
 * one warp per problem (one element per lane), a lane group per problem above; 1 = lane group,
 * 2 = pipeline, 3 = one warp per problem.  All three perform the same IEEE operations per element: identical bits.  Returns the
 * previous value. */
int hop_test_set_fused_small_variant(int variant);
/* Test hook: line-search kernel, 0 = the five step sizes side by side, six threads per problem [default], 1 = one thread
 * per problem trying them in turn; identical bits.  Returns the previous value. */
int hop_test_set_linesearch_variant(int variant);
/* Test hook: backward-pass kernel.  0 [default] = matrix products on the FP64 tensor pipe for n > 8 (quadrotor) in FAST / GJ
 * solves of at least 4 096 instances, one warp per problem with the reference's summation order otherwise (small systems, HOP_MODE_EXACT solves, the
 * stand-alone entry point); 1 = one thread per problem; 2 = one warp per problem, ordered sums (1 and 2: identical bits);
 * 3 = tensor-pipe kernel wherever it is instantiated (gains within 1e-12 relative of 2).  Returns the previous value. */
int hop_test_set_backward_variant(int variant);

/* Measures the FP64 FMA throughput of the current device with a register-resident DFMA chain
 * (8 independent accumulators per thread, 2048 threads per SM), timed with CUDA events.  This is
 * the roofline denominator bench.py reports against (MEASURED_PEAKS.json holds no FP64 figure). */
int hop_probe_fp64_tflops(int iters, double *tflops_out, double *ms_out);

#ifdef __cplusplus
}
#endif
#endif
