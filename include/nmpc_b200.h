/*
 * nmpc_b200.h -- C ABI of the B200-native batched NMPC solver (libnmpc_b200.so).
 *
 * Drop-in boundary for ONE path of devsonni/MPC-Implementation: the per-step NLP solve
 *     sol = solver(x0=, lbx=, ubx=, lbg=, ubg=, p=)            Python/NMPC_TT.py:358-365
 * of the CasADi `Function` built by  ca.nlpsol('solver','ipopt',nlp_prob,opts)  (:250-267), plus
 * the plant/target/warm-start shift around it (shift_timestep, :13-30) and the FOV-centre
 * bookkeeping (:399-402).  Everything the reference derives symbolically from its SX graph
 * (dynamics :139-148, rollout :160-167, cost :193-221, constraint rows :234-244) is compiled into
 * the kernels; what the scripts edit in source (T, N, obstacles, weights) is the `nmpc_spec`.
 *
 * Conventions
 *   - All vectors use CasADi's layouts: w = vec(U) column-major, w[6k+i] = U[i,k] (:247-248,:294);
 *     g stage-major, rows [z, theta, X5, X6, X7, obs_1..obs_n] per stage k=0..N (:235-243);
 *     p = [x(8); x_t; y_t; theta_t] (:350-353).
 *   - Batches are instance-major: field[b][i].  Each field is its own array (structure of arrays
 *     at field level); one warp solves one instance and reads its row with coalesced loads.
 *   - FP64 throughout.  +-inf (or |b| >= 1e19) in lbg/ubg/lbx/ubx means "no bound" (:280-282).
 *   - Every function returns 0 on success, non-zero on error (message via nmpc_last_error()).
 *     Per-instance solver outcomes are DATA (status[], iters[]), never error returns -- the
 *     reference never inspects IPOPT's status either (:358-367).
 *   - Device pointers unless the name says _host.  Calls are asynchronous on `cuda_stream`
 *     (a cudaStream_t cast to void*; NULL = default stream); the caller synchronises.
 *   - One handle per (device, stream); calls on one handle are not re-entrant.
 *   - There is no CPU fallback: nmpc_create fails if no sm_100 device is present.
 */
#ifndef NMPC_B200_H
#define NMPC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NMPC_NX 8
#define NMPC_NU 6
#define NMPC_NP 11
#define NMPC_MAX_STAGES 32   /* N + 1 <= 32: one horizon stage per warp lane */
#define NMPC_MAX_OBS 16

/* per-instance return status (mirrors IPOPT's ApplicationReturnStatus names where one exists) */
enum {
  NMPC_SOLVE_SUCCEEDED = 0,
  NMPC_MAXITER_EXCEEDED = 1,
  NMPC_RESTORATION_FAILED = 2,   /* IPOPT "Restoration_Failed": the restoration phase was called at an (almost) feasible point,
                                    or converged to a feasible point that the original filter does not accept */
  NMPC_STEP_TOO_SMALL = 3,       /* "Search_Direction_Becomes_Too_Small" */
  NMPC_INVALID_NUMBER = 4,
  NMPC_ERROR_IN_STEP_COMPUTATION = 5,
  NMPC_INFEASIBLE_PROBLEM = 6    /* "Infeasible_Problem_Detected": the restoration phase converged to a point of local infeasibility */
};

/* What the reference scripts hard-code in source.  Replaces the SX dict {'f','x','g','p'} and the
 * opts dict handed to ca.nlpsol (NMPC_TT.py:250-267). */
typedef struct nmpc_spec {
  double T;            /* Euler step                           NMPC_TT.py:57   */
  int32_t N;           /* horizon, N + 1 <= NMPC_MAX_STAGES    NMPC_TT.py:58   */
  int32_t n_obs;       /* obstacle rows per stage              NMPC_TT.py:241-243 */
  double w1, w2;       /* cost weights                         NMPC_TT.py:204-205 */
  double vfov, hfov;   /* field of view                        NMPC_TT.py:201-202 */
  /* IPOPT options the scripts set (NMPC_TT.py:257-265) or leave at default */
  int32_t max_iter;    /* 100 */
  int32_t scaling;     /* 1 = gradient-based NLP scaling (IPOPT default) */
  double tol;          /* 1e-8 */
  int32_t max_batch;   /* largest B any call will pass */
  int32_t fill;        /* scheduling hint, 0 or 1 = default: a batch smaller than the machine is spread over as many SMs as it
                          has instances; k > 1 packs it onto fewer SMs, k instances per resident warp (refilled from the
                          queue), which leaves SMs to the concurrent solves of other handles (pipelined sub-batches) */
  int32_t model;       /* NMPC_MODEL_GIMBAL (0, every Python script) or NMPC_MODEL_GIMBAL_LESS (1) */
} nmpc_spec;

/* Model variants (SURVEY.md 8f-4).
 *   NMPC_MODEL_GIMBAL       8 states [x y z theta psi phi_g shi_g theta_g], 6 controls, p[11], rows [z theta X5 X6 X7 obstacles]
 *                           per stage, cost = w1 * distance + w2 * FOV ellipse          Python/NMPC_TT.py:105-154, :193-244
 *   NMPC_MODEL_GIMBAL_LESS  5 states [x y z theta psi], 3 controls [v omega_2 omega_3], p[8] = [state(5); x_t y_t theta_t], rows
 *                           [z theta obstacles] per stage, cost = distance only (w1, w2, vfov, hfov ignored)
 *                                                                   MATLAB/Dynamic Obstacles/NMPC_TT.m:25-37, :100-111
 * Every array below has the model's own sizes: n_w = nmpc_n_w(spec) controls, n_g = nmpc_n_g(spec) rows, nmpc_n_p(spec)
 * parameters per instance (6N / (5 + n_obs)(N + 1) / 11 for model 0, 3N / (2 + n_obs)(N + 1) / 8 for model 1). */
#define NMPC_MODEL_GIMBAL 0
#define NMPC_MODEL_GIMBAL_LESS 1

typedef struct nmpc_handle nmpc_handle;

/* ca.nlpsol(...)  (NMPC_TT.py:267): allocate the per-device workspace. */
int nmpc_create(const nmpc_spec* spec, int device, nmpc_handle** out);
int nmpc_destroy(nmpc_handle* h);

/* flags for nmpc_solve */
#define NMPC_OBS_PER_INSTANCE 1u   /* obst is [B][n_obs][3] instead of [n_obs][3] */
#define NMPC_PREDICT_TARGET 2u     /* nmpc_solve_and_step / nmpc_run_closed_loop only: every solve uses the target's own Euler
                                      prediction over the horizon instead of the frozen target p[8:10] -- stage k of instance b
                                      sees  th_k = th_t + (T om) k,  s_k = (T v)(cos th_k, sin th_k),  (x, y)_k = (x_t, y_t) +
                                      (s_0 + ... + s_{k-1})  with (x_t, y_t, th_t) the target block of p and (v, om) this step's
                                      target input (target_vw or the schedule), computed in the kernel, no host work per step.
                                      Refused by the calls that have no (v, om) (nmpc_solve, nmpc_solve_host(_async), nmpc_eval,
                                      nmpc_lam_p) and while a target trajectory is set (nmpc_set_target_trajectory). */
#define NMPC_KEEP_BARRIER 4u       /* nmpc_solve, nmpc_solve_host, nmpc_solve_host_async only: the solve also keeps the barrier data
                                      of its final iterate (the Sigma_x and Sigma_g of the sensitivity system below) in buffers the
                                      handle owns, for nmpc_sensitivity.  The results of the solve are bit-identical with and
                                      without it.  Refused by nmpc_solve_and_step and nmpc_run_closed_loop. */

/* solver(x0,lbx,ubx,lbg,ubg,p)  (NMPC_TT.py:358-365), B instances at once.
 *   p    [B][11]   x0  [B][6N]                       inputs
 *   lbx, ubx [6N]; lbg, ubg [n_g]                    shared by the batch (as in every script)
 *   obst [n_obs][3] = {cx, cy, r_uav + r_obs}        (x_o_j, y_o_j, UAV_r+obs_r of :224-243)
 *   x [B][6N], f [B], g [B][n_g], lam_x [B][6N], lam_g [B][n_g]   outputs; g/lam_* may be NULL
 *   status [B], iters [B]                            per-instance outcome (may be NULL)          */
int nmpc_solve(nmpc_handle* h, int32_t B,
               const double* p, const double* x0,
               const double* lbx, const double* ubx, const double* lbg, const double* ubg,
               const double* obst, uint32_t flags,
               double* x, double* f, double* g, double* lam_x, double* lam_g,
               int32_t* status, int32_t* iters, void* cuda_stream);

/* Same call with HOST buffers (what a CasADi-DM caller holds): H2D copies, solve, D2H copies and a
 * stream synchronise happen inside. */
int nmpc_solve_host(nmpc_handle* h, int32_t B,
                    const double* p, const double* x0,
                    const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                    const double* obst, uint32_t flags,
                    double* x, double* f, double* g, double* lam_x, double* lam_g,
                    int32_t* status, int32_t* iters);

/* The same, asynchronous: the copies and the solve are enqueued on the handle's own stream and the call returns.
 * The host buffers should be page-locked (cudaHostAlloc, torch pin_memory) -- pageable memory makes the copies
 * synchronous -- and must not be read or written until nmpc_synchronize(h) has returned.  Several handles driven this
 * way overlap: while one sub-batch waits for its stragglers, the next one's copies and solve proceed. */
int nmpc_solve_host_async(nmpc_handle* h, int32_t B,
                          const double* p, const double* x0,
                          const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                          const double* obst, uint32_t flags,
                          double* x, double* f, double* g, double* lam_x, double* lam_g,
                          int32_t* status, int32_t* iters);
int nmpc_synchronize(nmpc_handle* h);   /* waits for the handle's own stream */
int nmpc_query(nmpc_handle* h, int32_t* busy);   /* *busy = 1 while an asynchronous host call is still in flight; never blocks */

/* Function-level evaluation (what CasADi's generated nlp_f / nlp_g / nlp_grad_f / nlp_hess_l
 * compute for IPOPT): at w [B][6N], p [B][11]
 *   f [B], g [B][n_g], grad_f [B][6N],
 *   jtv [B][6N]  = J(w)^T lam          (lam [B][n_g])
 *   hv  [B][6N]  = Hess_w(sigma f + lam^T g) v          (v [B][6N])
 * Any output may be NULL. */
int nmpc_eval(nmpc_handle* h, int32_t B, const double* w, const double* p, const double* obst, uint32_t flags,
              double sigma, const double* lam, const double* v,
              double* f, double* g, double* grad_f, double* jtv, double* hv, void* cuda_stream);

/* sol['lam_p'] of CasADi's result dict (NMPC_TT.py:358-365 returns it with x, f, g, lam_x, lam_g; no script reads it): the
 * multipliers of the parameters, lam_p = -(d/dp)(f + lam_g^T g) at the returned point [3P: CasADi's sign convention, the one
 * that makes grad_x (f + lam_g^T g) + lam_x = 0 for lam_x].  x_sol [B][n_w], p [B][n_p], lam_g [B][n_g] as returned by
 * nmpc_solve; lam_p [B][n_p].  With a per-stage target prediction (nmpc_set_target_trajectory) the target entries of p do not
 * enter the NLP and their multipliers are 0. */
int nmpc_lam_p(nmpc_handle* h, int32_t B, const double* x_sol, const double* p, const double* obst, uint32_t flags,
               const double* lam_g, double* lam_p, void* cuda_stream);

/* Solution sensitivities of the last solve on this handle, which must have passed NMPC_KEEP_BARRIER with the same B: CasADi's
 * jac:x:p (and sIPOPT's), and the derivative with respect to the cost weights.  For each instance it is the implicit-function
 * derivative of the barrier KKT system at the solve's final iterate, with no inertia correction (delta_w = 0):
 *     K dx/dth = -(grad2_{x th} L + J^T Sigma_g J_th),     K = grad2_{xx} L + Sigma_x + J^T Sigma_g J,     L = f + lam_g^T g,
 * with J = dg/dx, J_th = dg/dth, Sigma_x = z_L / (x - l) + z_U / (u - x) from the solve's own bound multipliers and distances to
 * its relaxed bounds, and Sigma_g the same for the row slacks, all in the unscaled units of lam_x / lam_g (DESIGN.md section 1).
 * It is computed from those kept Sigmas, not from lam_x / lam_g and g(x): x is clipped to the original bounds and g(x) differs
 * from the solve's slacks by up to the tolerance, which for an active row is more than the slack's distance to its bound.
 *   x_sol [B][n_w], p [B][n_p], lam_g [B][n_g]: as that solve returned them (and given to it);  obst / flags as for nmpc_solve
 *   dx_dp [B][n_w][n_p] = dx/dp.  The theta_t column is exactly 0 (theta_t does not enter the NLP), and so are the target columns
 *     while a target trajectory is set (nmpc_set_target_trajectory), as in nmpc_lam_p
 *   dx_dw [B][n_w][2] = dx/d(w1, w2) (may be NULL; model 0 only): with per-instance weights (nmpc_set_weights), each instance's own
 *   sens_status [B] (may be NULL): 0, or 1 when the reduced Hessian is not positive definite at delta_w = 0 -- the sensitivity is
 *     then undefined and the instance's columns are NaN
 * The weights and the target trajectory set on the handle are read as by the solve: they must be the solve's.  The columns are
 * computed for every instance; only those of converged instances (status NMPC_SOLVE_SUCCEEDED) are a sensitivity of a solution.
 * Refused when the last solve did not keep its barrier data, when B differs from its B, and when dx_dw is given for model 1.
 * cuda_stream may differ from the solve's (e.g. after nmpc_solve_host, which runs on the handle's own stream): the launch waits
 * for the keeping solve, and the next solve on the handle waits for the launch (they share the handle's Riccati scratch). */
int nmpc_sensitivity(nmpc_handle* h, int32_t B, const double* x_sol, const double* p, const double* lam_g, const double* obst,
                     uint32_t flags, double* dx_dp, double* dx_dw, int32_t* sens_status, void* cuda_stream);
/* The obstacle columns of the same sensitivity: dx_dobst [B][n_w][n_obs][3] = dx/d(cx_j, cy_j, r_j) of every obstacle row j,
 * r_j = r_uav + r_obs as in the obstacle table.  The other arguments, the conditions and the stream ordering are those of
 * nmpc_sensitivity: obst / flags must be the positions the solve used (one shared table or NMPC_OBS_PER_INSTANCE), and with a
 * shared table each instance's columns are its own x* with respect to the shared entries.  sens_status as for nmpc_sensitivity
 * (the same factorisation: the same value).  Also refused for a problem without obstacle rows (n_obs = 0). */
int nmpc_sensitivity_obstacles(nmpc_handle* h, int32_t B, const double* x_sol, const double* p, const double* lam_g,
                               const double* obst, uint32_t flags, double* dx_dobst, int32_t* sens_status, void* cuda_stream);
/* The barrier data nmpc_sensitivity uses: sig_x [B][n_w], sig_g [B][n_g] (device pointers, either may be NULL) <- the Sigma_x and
 * Sigma_g kept by the last solve, B its batch size.  Lets a caller check the sensitivity system or form other right-hand sides.
 * Refused when the last solve did not keep them.  (An addition to the sensitivity call: the tests build the sensitivity system
 * from these Sigmas.)  The copies wait for the keeping solve. */
int nmpc_barrier_data(nmpc_handle* h, double* sig_x, double* sig_g, void* cuda_stream);

/* shift_timestep (NMPC_TT.py:13-30) + FOV centre (:399-402) for B instances, in place on the
 * parameter block the next solve reads:
 *   p [B][11]: p[0:8] <- x + T f_u(x, u[:,0]);  p[8:11] <- target + T [v cos th, v sin th, om]
 *   u_warm [B][6N] <- x_sol shifted by one stage, last stage repeated (may alias x_sol)
 *   target_vw [B][2] = (v, om) of the target for this step (the scripts' con_t, keyed on mpc_iter); nmpc_solve_and_step
 *   also takes NULL here when a device-side schedule is set (nmpc_set_schedule)
 *   fov_centre [B][2] (may be NULL) = (X_E, Y_E) of the NEW state
 *   err_accum [B] (may be NULL; needs fov_centre) += || FOV centre of the NEW state - target of THIS step ||, the
 *   per-step term of the scripts' final metric (NMPC_TT.py:433-440). */
int nmpc_step(nmpc_handle* h, int32_t B, const double* x_sol, double* p,
              double* u_warm, const double* target_vw, double* fov_centre, double* err_accum, void* cuda_stream);

/* nmpc_solve and nmpc_step in ONE launch (SURVEY 8f-1: "fused into the solve kernel's epilogue"): the warp that solved
 * instance b applies the shift to it right away -- p[b] and u_warm[b] (which is also the warm start x0 of the solve)
 * are updated in place, fov_centre / err_accum as in nmpc_step.  x (may be NULL) receives the un-shifted solution and
 * must not alias u_warm.  g / lam_* are not produced by this entry point. */
int nmpc_solve_and_step(nmpc_handle* h, int32_t B, double* p, double* u_warm,
                        const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                        const double* obst, uint32_t flags, const double* target_vw,
                        double* x, double* f, double* fov_centre, double* err_accum,
                        int32_t* status, int32_t* iters, void* cuda_stream);

/* The scripts' main loop `while mpc_iter < sim_time / T` (NMPC_TT.py:346-402) on the device: every one of the B instances
 * advances `steps` closed-loop steps (solve :358-365 + shift_timestep :382 + FOV centre / error :399-402, :435) in ONE launch.
 * The closed loops are independent, so there is no batch-wide barrier between the steps: the warp that has finished step k of
 * an instance goes straight on with its step k + 1 (the epilogue has written p and the warm start in place), and the SMs never
 * wait for the slowest solve of a step.  Per instance the arithmetic is exactly that of `steps` consecutive
 * nmpc_solve_and_step calls -- results are bit-identical (tests) -- only the schedule differs.
 *   p [B][n_p], u_warm [B][n_w] in/out;  target_vw [B][2] constant per instance, or NULL with nmpc_set_schedule (the table is read
 *   at mpc_iter, mpc_iter + 1, ...; the step counter advances by `steps`)
 *   x [B][n_w], f [B]: solution of the LAST step (may be NULL);  fov_centre [B][2], err_accum [B] (+=) as in nmpc_step
 *   status_log, iters_log [steps][B]: outcome of every solve (may be NULL);  converged [B]: += number of converged solves (may be NULL)
 * Every option of nmpc_solve_and_step applies to every step: the target prediction (flags |= NMPC_PREDICT_TARGET) is made from
 * each step's own target, and moving obstacles (nmpc_set_obstacle_motion) move after each step.  Not available with a
 * caller-given target trajectory (nmpc_set_target_trajectory), which would hold for one step only. */
int nmpc_run_closed_loop(nmpc_handle* h, int32_t B, int32_t steps, double* p, double* u_warm,
                         const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                         const double* obst, uint32_t flags, const double* target_vw,
                         double* x, double* f, double* fov_centre, double* err_accum,
                         int32_t* status_log, int32_t* iters_log, int32_t* converged, void* cuda_stream);

/* Target schedule on the device.  The reference's shift_timestep reads the target's (v, omega) for this step from an
 * if-chain keyed on the global step counter (`con_t`, T_Trajectory.py:24-57, Plus Trajectory.py:25-69, Race Track 2.py:28-36).
 * dev_table [n_rows][len][2] holds (v, omega) per step for n_rows schedules (a step index beyond len - 1 uses the last
 * entry); instance b follows row dev_row_of_instance[b] (NULL: row 0) starting at step dev_phase[b] (NULL: 0).  After
 * this call nmpc_solve_and_step accepts target_vw == NULL, looks the pair up in its epilogue with
 * step = mpc_iter + phase[b], and advances mpc_iter by one per call -- no per-step host work at any batch size.
 * dev_table == NULL removes the schedule.  All arrays stay owned by the caller and must outlive their use. */
int nmpc_set_schedule(nmpc_handle* h, const double* dev_table, int32_t n_rows, int32_t len,
                      const int32_t* dev_row_of_instance, const int32_t* dev_phase, int32_t mpc_iter);

/* statistics of the last nmpc_solve on this handle (device work counters, host copy) */
typedef struct nmpc_stats {
  int64_t kernel_launches;     /* kernels launched by the last call */
  int64_t factorizations;      /* Riccati factorisations summed over the batch */
  int64_t ls_trials;           /* line-search trial points summed over the batch */
  int64_t soc_accepted;
  int64_t resto_calls;         /* restoration phases entered */
  int64_t resto_iters;         /* iterations spent inside restoration phases */
  int64_t watchdog_starts;
  int64_t soft_resto_steps;    /* steps accepted by the soft restoration phase's primal-dual error test */
  int64_t filter_resets;
  int64_t trial_passes;        /* trial-point evaluations: ls_trials - trial_passes trials came from a paired pass's second point */
} nmpc_stats;
int nmpc_get_stats(nmpc_handle* h, nmpc_stats* out);   /* synchronises the handle's last stream */

/* Scheduling.  The persistent kernel fetches instances from a queue; the step ends when the last straggler does, so
 * long solves should start first.  By default the library orders the queue itself: when a call has the same B as
 * the previous call on this handle (a closed loop), instances are fetched by the previous call's iteration counts,
 * longest first (a counting sort done by the previous launch's last warp; NMPC_B200_AUTO_ORDER=0 in the environment
 * disables it).
 * nmpc_set_order overrides this for the NEXT nmpc_solve only: dev_order [B] is a permutation of 0..B-1.
 * Results never depend on the order (instances are independent); only the tail of the batch step does. */
int nmpc_set_order(nmpc_handle* h, const int32_t* dev_order);

/* Per-instance cost weights (w1, w2) for the weight sweeps of the reference's outer loops (MATLAB/Race Track 1/MPC.m:1,:90;
 * the dead tables at NMPC_TT.py:178-188): dev_weights [B][2] is read by every subsequent nmpc_solve / nmpc_solve_host /
 * nmpc_eval on this handle (it must stay allocated and hold at least B rows); NULL restores spec.w1 / spec.w2. */
int nmpc_set_weights(nmpc_handle* h, const double* dev_weights);

/* Predicted target trajectory (north star: "p = [UAV state; predicted target trajectory]"; SURVEY 8f-2).  The reference
 * holds the target at p[8:10] over the whole horizon (NMPC_TT.py:219-220); with dev_targets [B][N][2] = (x_t, y_t) of
 * stage k = 0..N-1 every stage cost uses its own prediction instead.  Read by every subsequent nmpc_solve /
 * nmpc_solve_host / nmpc_eval / nmpc_solve_and_step on this handle (must stay allocated, at least B rows); NULL restores
 * p[8:10].  A closed loop that wants the target's own Euler prediction every step passes NMPC_PREDICT_TARGET instead,
 * which computes it in the kernel (and works in nmpc_run_closed_loop); the two exclude each other. */
int nmpc_set_target_trajectory(nmpc_handle* h, const double* dev_targets);

/* Moving obstacles (MATLAB/Dynamic Obstacles: obstacle positions are parameters that move every step; SURVEY 8f-2).
 * dev_obst [B][n_obs][3] = (cx, cy, r_uav + r_obs) is the writable per-instance obstacle field that the following
 * nmpc_solve_and_step / nmpc_run_closed_loop calls pass as `obst` (with NMPC_OBS_PER_INSTANCE when B > 1); dev_vel
 * [B][n_obs][2] holds the obstacle velocities.  After each solve those calls advance the centres in place,
 * cx += T vx, cy += T vy (rounded as o + (T v)); the constraint rows of that solve use the positions before the move.
 * They fail if `obst` is not dev_obst, or is a shared table while B > 1.  The other calls neither check nor move.
 * NULL, NULL removes the motion.  Both arrays stay owned by the caller and must outlive their use. */
int nmpc_set_obstacle_motion(nmpc_handle* h, double* dev_obst, const double* dev_vel);

/* NON-REFERENCE fast mode (SURVEY.md 8f-4): warm start of the multipliers -- CasADi's lam_x0 / lam_g0 inputs with
 * ipopt.warm_start_init_point = "yes".  No reference script uses it (they pass neither, NMPC_TT.py:358-365), and it changes
 * the iterates, so it is OFF unless this call enables it.  dev_lam_x0 [B][n_w], dev_lam_g0 [B][n_g] (sign convention of the
 * lam_x / lam_g outputs) are read by every subsequent nmpc_solve on this handle; nmpc_solve_and_step additionally
 * OVERWRITES them with the multipliers of its own solve shifted by one stage (the dual counterpart of the primal warm
 * start, NMPC_TT.py:20-23).  A NaN in dev_lam_x0[b][0] cold-starts instance b (IPOPT's default multiplier start, mu_init
 * 0.1); the fused shift stores that marker after a solve that did not converge.  NULL, NULL restores the cold start.
 * opts NULL or fields <= 0: IPOPT's defaults (1e-3 pushes) and mu_init 1e-4.
 * Measured (tests/probes/warm_start_probe.py): a re-solve from (x*, lam*) drops from 19 to 6..9 iterations; in the closed
 * loop the shifted guesses do NOT reduce the iteration count (the active set of the shifted problem differs). */
typedef struct nmpc_warm_opts {
  double mu_init;             /* barrier parameter a warm-started solve begins with */
  double bound_push, bound_frac, slack_bound_push, slack_bound_frac;   /* warm_start_(slack_)bound_push / _frac */
  double mult_bound_push;     /* warm_start_mult_bound_push */
} nmpc_warm_opts;
int nmpc_set_warm_start(nmpc_handle* h, double* dev_lam_x0, double* dev_lam_g0, const nmpc_warm_opts* opts);

/* Test hook: per-iteration log of every instance of subsequent nmpc_solve calls,
 * dev_buf [B][rows][10] = {mu, f, inf_pr, inf_du, delta_w, alpha_pr, alpha_du, ls_trials, step tag (IPOPT's alpha_primal_char),
 * 1 inside the restoration phase}; NULL disables. */
int nmpc_set_debug_log(nmpc_handle* h, double* dev_buf, int32_t rows);

/* Measurement aid: FP64 FMA peak of `device` in TFLOP/s (register-resident DFMA loop on every SM).
 * MEASURED_PEAKS.json carries HBM and bf16 peaks only; this is the denominator of the FP64 roofline. */
int nmpc_measure_fp64_peak(int device, double* tflops);

/* sizes implied by a spec */
int32_t nmpc_n_w(const nmpc_spec* spec);   /* 6 N                 (model 1: 3 N) */
int32_t nmpc_n_g(const nmpc_spec* spec);   /* (5 + n_obs)(N + 1)  (model 1: (2 + n_obs)(N + 1)) */
int32_t nmpc_n_p(const nmpc_spec* spec);   /* 11                  (model 1: 8) */

const char* nmpc_last_error(void);   /* thread-local */
const char* nmpc_version(void);

#ifdef __cplusplus
}
#endif
#endif
