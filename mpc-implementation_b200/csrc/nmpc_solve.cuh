// nmpc_solve.cuh -- one-warp-per-instance primal-dual interior-point solve (the hot path).
//
// Replaces  sol = solver(x0,lbx,ubx,lbg,ubg,p)  (Python/NMPC_TT.py:358-365; CasADi -> IPOPT -> MUMPS) for the
// reference's UAV target-tracking NLP.  Algorithm = IPOPT's (Waechter & Biegler 2006) with the scripts'
// options (NMPC_TT.py:257-265): slack form g(w) - s = 0, relaxed bounds, gradient-based scaling,
// monotone barrier, fraction-to-boundary, inertia correction, filter line search with second-order
// correction, watchdog, soft restoration phase and the restoration phase proper (min ||c||_1 with a proximity
// term, solved by the same algorithm -- `RS = true` instantiations of the phases), scaled optimality-error
// termination.  The whole iteration loop runs inside the kernel.
//
// Structure: the iterate lives in the warp's slice of shared memory at compile-time offsets (Lay<N, NOBS>); every
// phase is a __noinline__ function template that loads its operands, works in registers and stores back, so each
// heavy code sequence exists exactly once and every workspace access is an LDS/STS with an immediate offset.  A block
// holds Lay::WPB warps (8 at N = 15, n_obs = 3) that start every IPM iteration together (align_warps) so that they
// share instruction-cache lines.  One launch is one whole closed-loop step when asked (nmpc_solve_and_step: the shift
// runs in ph_output) and also prepares the next call on the handle (queue / counters, longest-first fetch order).
// Rare events (watchdog, soft restoration, restoration) keep their extra state in a per-warp global scratch (`cold`).
#pragma once
#include "nmpc_device.cuh"
#include "nmpc_riccati.cuh"

namespace nmpc {

struct Opt {
  int max_iter; int scaling; double tol;
  double dual_inf_tol = 1.0, constr_viol_tol = 1e-4, compl_inf_tol = 1e-4;
  double bound_relax = 1e-8, bound_push = 1e-2, bound_frac = 1e-2;
  double mu_init = 0.1, kappa_mu = 0.2, theta_mu = 1.5, kappa_eps = 10.0, tau_min = 0.99;
  double kappa_d = 1e-4, kappa_sigma = 1e10, s_max = 100.0;
  double max_grad = 100.0, scal_min = 1e-8;
  double constr_mult_init_max = 1e3;
  double dw_init = 1e-4, dw_min = 1e-20, dw_max = 1e20, dw_inc_first = 100.0, dw_inc = 8.0, dw_dec = 1.0 / 3.0;
  double gamma_theta = 1e-5, gamma_phi = 1e-8, eta_phi = 1e-8, s_theta = 1.1, s_phi = 2.3, delta = 1.0;
  double alpha_min_frac = 0.05, alpha_red = 0.5; int max_soc = 4; double kappa_soc = 0.99;
  double theta_max_fact = 1e4, theta_min_fact = 1e-4;
  double tiny_step_tol = 10.0 * 2.220446049250313e-16, tiny_step_y_tol = 1e-2;
  double obj_max_inc = 5.0; int max_filter_resets = 5, filter_reset_trigger = 5;
  int watchdog_trigger = 10, watchdog_trial_max = 3;
  int max_soft_resto = 10; double soft_resto_red = 1.0 - 1e-4;
  double resto_rho = 1000.0, resto_eta_factor = 1.0, kappa_resto = 0.9;
  double bound_mult_reset_threshold = 1e3;
  double resto_theta_max_fact = 1e8;
  // NON-REFERENCE warm start of the multipliers (nmpc_set_warm_start; IPOPT's WarmStartIterateInitializer [3P])
  double ws_mu_init = 1e-4, ws_bound_push = 1e-3, ws_bound_frac = 1e-3, ws_slack_push = 1e-3, ws_slack_frac = 1e-3;
  double ws_mult_push = 1e-3, ws_mult_init_max = 1e6;
};

struct SolveArgs {
  Prob pr; Opt o;
  int B;
  const double *p, *x0, *lbx, *ubx, *lbg, *ubg, *obs;
  int obs_per_instance;
  double *x, *f, *g, *lam_x, *lam_g;
  int32_t *status, *iters;
  const double* weights;             // optional per-instance cost weights [B][2] = (w1, w2); NULL = spec weights
  const double* tgt;                 // optional per-instance, per-stage predicted target [B][N][2]; NULL = p[8:10]
  // fused closed-loop shift (nmpc_solve_and_step): when step_p != NULL the warp that solved instance b also applies
  // shift_timestep to it -- p[b] and u_warm[b] in place, FOV centre, error term -- and no nmpc_step launch is needed
  double *step_p, *step_u; const double* step_vw; double *step_fov, *step_err;
  // multiplier guesses lam_x0 [B][n_w], lam_g0 [B][n_g] (NULL = IPOPT's cold multiplier start, as every reference script;
  // a NaN in lam_x0[b][0] cold-starts instance b); with ws_shift the fused closed-loop epilogue overwrites them with
  // this solve's multipliers shifted by one stage (NaN marker after a failed solve)
  double *lam_x0, *lam_g0; int ws_shift;
  // free-running closed loop (nmpc_run_closed_loop): every instance advances run_steps closed-loop steps back to back in the
  // warp that fetched it; optional per-step logs [run_steps][B], per-instance count of converged solves
  int run_steps; int32_t *status_log, *iters_log, *conv_count;
  // target schedule on the device (nmpc_set_schedule): when step_vw == NULL the target's (v, omega) of this step is
  // sched_table[sched_id[b]][min(sched_iter + sched_phase[b], sched_len - 1)]  -- the scripts' `con_t` keyed on mpc_iter
  const double* sched_table; const int32_t *sched_id, *sched_phase; int sched_len, sched_iter;
  // target prediction on the device (NMPC_PREDICT_TARGET, fused calls only): ph_predict writes the target's own Euler prediction
  // over the horizon from p's target block and this step's (v, omega) to tgt_pred [B][N][2], which is then also `tgt`
  double* tgt_pred;
  // obstacle motion (nmpc_set_obstacle_motion, fused calls only): after the shift the epilogue advances the per-instance table
  // obs_move [B][n_obs][3] (the same array as `obs`) by T * obs_vel [B][n_obs][2]
  double* obs_move; const double* obs_vel;
  int32_t* iters_keep;              // handle-owned copy of iters[] (drives the next call's fetch order)
  const int32_t* order;              // optional processing order (longest-first scheduling); NULL = 0..B-1
  int* counter;                      // work queue of THIS call
  // Bookkeeping for the NEXT call on the same handle is done by this launch, so that a solve is ONE launch: the first
  // thread resets the next call's queue / done / work counters (calls on a handle are stream-ordered), and the warp that
  // finishes the last instance writes the next call's longest-first fetch order from this call's iteration counts.
  int *counter_next, *done, *done_next;
  unsigned long long* stats_next;
  int32_t* order_out;                // may be NULL (no automatic ordering)
  unsigned long long* stats;         // [9]: factorizations, ls trials, soc accepted, restoration calls, restoration iterations,
                                     //      watchdog starts, soft restoration steps, filter resets, trial passes
  double* ric; int ric_stride;       // L2-resident Riccati scratch, one slice per resident warp
  double* cold; int cold_stride;     // per-warp scratch of the rare paths (Lay::COLD_TOTAL)
  const unsigned* ricmap;            // per-lane ownership maps of the factorisation (nmpc_riccati.cuh: ric_map_build)
  double* dbg; int dbg_rows;         // optional per-iteration log [B][dbg_rows][10] (tests only)
  int pair_trials;                   // layouts with Lay::PAIR: each backtracking trial pass also evaluates the next trial point
  // barrier data of the final iterate (NMPC_KEEP_BARRIER: non-NULL launches the KEEP instantiation of the kernel, whose
  // ph_output writes them), in the unscaled units of lam_x / lam_g: sig_x [B][n_w] = z_L / (w - l~) + z_U / (u~ - w),
  // sig_g [B][n_g] the same for the row slacks.  The sensitivity kernel (nmpc_sens.cuh) reads them, with x / lam_g as inputs.
  double *sig_x, *sig_g;
  double *dx_dp, *dx_dw; int32_t* sens_status;     // nmpc_sensitivity: [B][n_w][n_p], [B][n_w][2] (may be NULL), [B]
  double* dx_do;                     // nmpc_sensitivity_obstacles: [B][n_w][3 n_obs], column 3 j + (0, 1, 2) = (cx_j, cy_j, r_j)
};
constexpr int NSTAT = 9;
constexpr int DBG_COLS = 10;

constexpr double EPSM = 2.220446049250313e-16;
__device__ __forceinline__ bool cmp_le(double lhs, double rhs, double bas) { return lhs - rhs <= 10.0 * EPSM * fabs(bas); }

__device__ __forceinline__ double push_in(double v, double lo, double hi, bool hl, bool hu, double k1, double k2) {
  if (hl && hu) {
    const double pl = fmin(k1 * fmax(1.0, fabs(lo)), k2 * (hi - lo));
    const double pu = fmin(k1 * fmax(1.0, fabs(hi)), k2 * (hi - lo));
    v = fmax(v, lo + pl); v = fmin(v, hi - pu);
  } else if (hl) v = fmax(v, lo + k1 * fmax(1.0, fabs(lo)));
  else if (hu) v = fmin(v, hi - k1 * fmax(1.0, fabs(hi)));
  return v;
}

struct Bnd { double lo, hi; bool hl, hu; };
// Relaxed bounds of control i of stage k (NMPC_TT.py:294-306) and of the scaled row r of stage k (:275-291).
// NOTE: these are inlined into several phase functions; the explicit round-to-nearest intrinsics keep the compiler
// from contracting the expressions into FMAs differently per copy.  A bound that differs by one ulp between the
// function that builds the Newton system and the one that updates the multipliers is a 1e-6 RELATIVE error of a
// 1e-10 slack, i.e. a 1e-5 error in a multiplier -- enough to stall the end game (seen with v2, DESIGN.md section 5).
__device__ __forceinline__ double relaxed_lo(double lo, double relax) { return lo > -1e19 ? __dsub_rn(lo, __dmul_rn(relax, fmax(1.0, fabs(lo)))) : -CUDART_INF; }
__device__ __forceinline__ double relaxed_hi(double hi, double relax) { return hi < 1e19 ? __dadd_rn(hi, __dmul_rn(relax, fmax(1.0, fabs(hi)))) : CUDART_INF; }
template <class L>
__device__ __forceinline__ Bnd ctl_bounds(const SolveArgs& A, int k, int i) {
  Bnd b;
  if (i >= L::NUA) { b.lo = -CUDART_INF; b.hi = CUDART_INF; b.hl = false; b.hu = false; return b; }     // absent control (model 1)
  b.lo = relaxed_lo(__ldg(A.lbx + L::NUA * k + i), A.o.bound_relax); b.hi = relaxed_hi(__ldg(A.ubx + L::NUA * k + i), A.o.bound_relax);
  b.hl = b.lo > -CUDART_INF; b.hu = b.hi < CUDART_INF;
  return b;
}
template <class L>
__device__ __forceinline__ Bnd row_bounds(const SolveArgs& A, int k, int r, double dc) {
  const double lo = __ldg(A.lbg + k * L::R + r), hi = __ldg(A.ubg + k * L::R + r);
  Bnd b;
  b.lo = relaxed_lo(lo > -1e19 ? __dmul_rn(dc, lo) : lo, A.o.bound_relax);
  b.hi = relaxed_hi(hi < 1e19 ? __dmul_rn(dc, hi) : hi, A.o.bound_relax);
  b.hl = b.lo > -CUDART_INF; b.hu = b.hi < CUDART_INF;
  return b;
}

// Warp alignment (DESIGN.md section 2): all Lay::WPB warps of a block meet at named barrier 1 at the start of every
// IPM iteration, and once more at named barrier 2 after the inertia-correction retries.  Both barriers count every
// thread of the block; barrier 0 is __syncthreads'.
//
// Alignment barrier (named barrier 1), OR-reducing `working` over the block.  Every warp calls it the same number of
// times: working warps once per IPM iteration, warps that ran out of work in a loop until the reduction says nobody is
// working -- the exit decision comes out of the barrier itself, so no warp can leave while another still waits.
template <class L>
__device__ __forceinline__ int align_warps(int working) {
  unsigned out;
  asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %1, 0;\n\tbar.red.or.pred q, 1, %2, p;\n\tselp.u32 %0, 1, 0, q;\n\t}"
               : "=r"(out) : "r"((unsigned)working), "n"(32 * L::WPB) : "memory");
  return (int)out;
}

// Retry point (named barrier 2).  Between two calls of align_warps every warp passes it exactly once: it waits there
// after the inertia-correction retries (retry_sync), and every path that skips that place -- an exit from the
// iteration loop, a `continue`, the least-squares multiplier start, a warp out of work -- arrives without waiting
// (retry_arrive).  A warp that did neither would leave the others waiting at bar.sync for ever; one that passed twice
// would complete a round that another warp has not reached.
template <class L>
__device__ __forceinline__ void retry_sync() { asm volatile("bar.sync 2, %0;" :: "n"(32 * L::WPB) : "memory"); }
template <class L>
__device__ __forceinline__ void retry_arrive() { asm volatile("bar.arrive 2, %0;" :: "n"(32 * L::WPB) : "memory"); }

#define LV(e) smem[L::LV0 + (e) * L::S + lane]
#define RW(arr, r) smem[L::rw(arr, r) + lane]
// lower-bound arrays exist for the box rows only (nmpc_device.cuh: RowArr)
#define VL_(r) ((r) < L::NB ? RW(A_VL, r) : 0.0)
#define IL_(r) ((r) < L::NB ? RW(A_IL, r) : 0.0)
#define LQ(e) smem[L::LQ0 + (e) * L::S + lane]
#define SOC(e) smem[L::soc(e) + lane]
#define RES(i) smem[L::RES0 + (i)]
#define PAR(i) smem[L::PAR0 + (i)]
#define SOC_DUS 0
#define SOC_Q2 6
// restoration row arrays in the cold scratch: (arr * R + r) * S + lane
#define RG(arr, r) cold[((arr) * L::R + (r)) * L::S + lane]
#define UREF(i) cold[L::CG_UR + (i) * L::S + lane]
enum RgArr { G_N = 0, G_P, G_ZN, G_ZP, G_DN, G_DP, G_DY, G_DN2, G_DP2, G_DY2, G_DS2, G_CSOC, G_CT };     // the last three: SOC step in s, SOC residual, residual of the last trial point

// T-scaled non-zeros of the dynamics Jacobian A_k - I of this lane's stage
struct Dyn { double e03, e13, e23, e04, e14; };
__device__ __forceinline__ Dyn dyn_entries(const Stage& s, double tv) {
  Dyn d; d.e03 = -tv * s.cps * s.sth; d.e13 = -tv * s.sps * s.sth; d.e23 = tv * s.cth;
  d.e04 = -tv * s.sps * s.cth; d.e14 = tv * s.cps * s.cth;
  return d;
}
// adjoint recursion lam_k = a_k + A_k^T lam_{k+1} by suffix scans; returns lam_{k+1} in lamn
template <int W = 32>
__device__ __forceinline__ void adjoint(const double* a, const Dyn& d, bool act, int lane, double* lamn) {
  double v[6] = {act ? a[0] : 0.0, act ? a[1] : 0.0, act ? a[2] : 0.0, act ? a[5] : 0.0, act ? a[6] : 0.0, act ? a[7] : 0.0};
  rscan_incl<6, W>(v, lane);
  lamn[0] = shfl_next(v[0], lane); lamn[1] = shfl_next(v[1], lane); lamn[2] = shfl_next(v[2], lane);
  lamn[5] = shfl_next(v[3], lane); lamn[6] = shfl_next(v[4], lane); lamn[7] = shfl_next(v[5], lane);
  double w[2] = {(act ? a[3] : 0.0) + d.e03 * lamn[0] + d.e13 * lamn[1] + d.e23 * lamn[2],
                 (act ? a[4] : 0.0) + d.e04 * lamn[0] + d.e14 * lamn[1]};
  rscan_incl<2, W>(w, lane);
  lamn[3] = shfl_next(w[0], lane); lamn[4] = shfl_next(w[1], lane);
}

// obstacle row jn of this lane's stage: value (r_u + r_o) - ||(x,y) - c_j||, unit normal, 1/distance   NMPC_TT.py:241-243
template <class L>
__device__ __forceinline__ double obs_value(const double* X, int jn, double& nx, double& ny, double& iD) {
  const double dx_ = X[0] - smem[L::OBS0 + 3 * jn], dy_ = X[1] - smem[L::OBS0 + 3 * jn + 1];
  const double d2 = __fma_rn(dx_, dx_, __dmul_rn(dy_, dy_));
  const double D = sqrt(d2);
  iD = rcp(D); nx = dx_ * iD; ny = dy_ * iD;
  return smem[L::OBS0 + 3 * jn + 2] - D;
}
// Per-lane scratch of a phase: 8 doubles per lane of the Riccati staging area, which is live only inside the riccati_*
// calls.  The rolled row and control loops below keep there what they would otherwise index dynamically in registers
// (which would put the array in local memory).
template <class L>
__device__ __forceinline__ double& stash(int i, int lane) { return smem[L::STG0 + i * 32 + lane]; }
static_assert(8 * 32 <= STG_N, "stash must fit the Riccati staging area");
// the states a box row reads, stashed for a FOR_ROWS over states held in registers
template <class L>
__device__ __forceinline__ void stash_box_states(const double* X, int lane) {
#pragma unroll
  for (int i = 2; i < 8; ++i) stash<L>(i, lane) = X[i];
}

// Visit the rows of this lane's stage: the box rows and the obstacle rows each in a rolled loop (one copy of the body
// per kind of row: the phases that visit rows are what bounds the instruction cache, DESIGN.md section 2).
// body(r, box, si, gu, nx, ny, iD) with gu the unscaled row value; si is the (run-time) state index of a box row, whose
// value XB(si) reads from shared memory; X holds the states x, y of the obstacle rows.
#define FOR_ROWS(XB, X, body)                                                                       \
  do {                                                                                              \
    _Pragma("unroll 1") for (int r_ = 0; r_ < L::NB; ++r_) {                                        \
      const int si_ = box_state(r_);                                                                \
      body(r_, true, si_, XB(si_), 0.0, 0.0, 0.0);                                                  \
    }                                                                                               \
    _Pragma("unroll 1") for (int jn_ = 0; jn_ < L::NOBS; ++jn_) {                                   \
      double nx_, ny_, iD_;                                                                         \
      const double gu_ = obs_value<L>((X), jn_, nx_, ny_, iD_);                                     \
      body(L::NB + jn_, false, 0, gu_, nx_, ny_, iD_);                                              \
    }                                                                                               \
  } while (0)

// target position seen by this lane's stage: the reference keeps (x_t, y_t) = p[8:10] over the horizon
// (NMPC_TT.py:219-220); with a predicted trajectory (nmpc_set_target_trajectory, NMPC_PREDICT_TARGET) stage k has its own.
// Coherent loads: with NMPC_PREDICT_TARGET the kernel itself has written the trajectory (ph_predict).
template <class L>
__device__ __forceinline__ double2 stage_target(const SolveArgs& A, int lane) {
  if (!A.tgt || lane >= L::N) return make_double2(PAR(8), PAR(9));
  const double* t = A.tgt + ((size_t)PAR(NPAR + 2) * L::N + lane) * 2;
  return make_double2(__ldcg(t), __ldcg(t + 1));
}

// the target's (v, omega) of closed-loop step `step` of this call (fused calls): the caller's target_vw, or the device
// schedule sched_table[row][min(sched_iter + step + phase, len - 1)] -- the scripts' `con_t` keyed on mpc_iter
__device__ __forceinline__ double2 target_input(const SolveArgs& A, int b, int step) {
  if (A.step_vw) return make_double2(__ldg(A.step_vw + 2 * (size_t)b), __ldg(A.step_vw + 2 * (size_t)b + 1));
  const int row = A.sched_id ? __ldg(A.sched_id + b) : 0, ph = A.sched_phase ? __ldg(A.sched_phase + b) : 0;
  const int at = min(A.sched_iter + step + ph, A.sched_len - 1);
  const double* e = A.sched_table + ((size_t)row * A.sched_len + at) * 2;
  return make_double2(__ldg(e), __ldg(e + 1));
}

// stage cost of this lane's stage (value / value + gradient + Hessian over (x, y, z, X5, X6, X7)) for the model of the layout
template <class L>
__device__ __forceinline__ double cost_val(const SolveArgs& A, const double* X, int lane) {
  const double2 t = stage_target<L>(A, lane);
  if (L::MODEL) return stage_cost_dist(X, t.x, t.y);
  return stage_cost(with_weights(A.pr, PAR(NPAR), PAR(NPAR + 1)), X, t.x, t.y);
}
template <class L>
__device__ __forceinline__ double cost_d2(const SolveArgs& A, const double* X, int lane, double* gl, double* Hl) {
  const double2 t = stage_target<L>(A, lane);
  if (L::MODEL) return stage_cost_dist_d2(X, t.x, t.y, gl, Hl);
  return stage_cost_d2(with_weights(A.pr, PAR(NPAR), PAR(NPAR + 1)), X, t.x, t.y, gl, Hl);
}

// Row quantities of the restoration problem's condensed Newton system (AugRestoSystemSolver).  With the slack s and the
// elastic variables n, p of row  d(x) + n - p - s = 0  eliminated,
//     dy = Om (G dx + chat),   Om = 1 / (1/D + 1/Dn + 1/Dp),   chat = c + rs/D + rp/Dp - rn/Dn,
//     ds = (dy - rs)/D,   dn = -(dy + rn)/Dn,   dp = (dy - rp)/Dp.
struct RestoRow { double D, Dn, Dp, Om, rs, rn, rp, n, p, zn, zp; };
template <class L>
__device__ __forceinline__ RestoRow resto_row(const SolveArgs& A, const double* cold, int lane, int r, double sig_s, double beta, double y,
                                              double mu, double dw) {
  RestoRow q;
  q.zn = RG(G_ZN, r); q.zp = RG(G_ZP, r);
  q.n = (RG(G_N, r)); q.p = (RG(G_P, r));
  const double in_ = rcp(q.n), ip_ = rcp(q.p), kdm = A.o.kappa_d * mu;
  q.D = sig_s + dw; q.Dn = q.zn * in_ + dw; q.Dp = q.zp * ip_ + dw;
  q.rs = mu * beta - y;
  q.rn = A.o.resto_rho + y - mu * in_ + kdm;
  q.rp = A.o.resto_rho - y - mu * ip_ + kdm;
  q.Om = rcp(rcp(q.D) + rcp(q.Dn) + rcp(q.Dp));
  return q;
}

// NMPC_PREDICT_TARGET (end of ph_load): the target's own Euler prediction over the horizon from the target
// block (x_t, y_t, th_t) of p and this step's (v, omega) into A.tgt_pred, in exactly the arithmetic of
// ClosedLoop.target_prediction() (bit-identical; no FMA contraction, sin and cos called separately):
//   th_k = th_t + (T w) k,   s_k = (T v) (cos th_k, sin th_k),   pos_k = (x_t, y_t) + (((0 + s_0) + s_1) + ... + s_{k-1})
// The prefix sum runs left to right, as torch's cumsum over a non-innermost dimension does.  A function of its own: inlined,
// the trigonometric reduction would add to ph_load's registers.
template <class L>
__device__ __noinline__ void ph_predict(const SolveArgs& A, int b, int lane, int step) {
  const double* pt = A.p + (size_t)b * L::NPA + L::NPA - 3;     // (L2 path: a free-running call re-reads what its own epilogue wrote)
  const double xt = __ldcg(pt), yt = __ldcg(pt + 1), tht = __ldcg(pt + 2);
  const double2 vw = target_input(A, b, step);
  const double Tv = __dmul_rn(A.pr.T, vw.x), Tw = __dmul_rn(A.pr.T, vw.y);
  const double th = __dadd_rn(tht, __dmul_rn(Tw, (double)lane));
  const double sx = __dmul_rn(Tv, cos(th)), sy = __dmul_rn(Tv, sin(th));
  double ax = 0.0, ay = 0.0;
#pragma unroll 1
  for (int j = 0; j < L::N - 1; ++j) {
    const double qx = __shfl_sync(FULL, sx, j), qy = __shfl_sync(FULL, sy, j);
    if (j < lane) { ax = __dadd_rn(ax, qx); ay = __dadd_rn(ay, qy); }
  }
  if (lane < L::N) {
    double* t = A.tgt_pred + ((size_t)b * L::N + lane) * 2;
    t[0] = __dadd_rn(xt, ax); t[1] = __dadd_rn(yt, ay);
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------
// load one instance: p -> PAR, warm start -> LV_U, obstacle table, unit scaling; the target prediction of step `step`
template <class L>
__device__ __noinline__ void ph_load(const SolveArgs& A, int b, int lane, int step) {
  if (L::MODEL) {      // p = [state(5); target(3)]: the camera states are zero
    if (lane < NPAR) PAR(lane) = lane < 5 ? __ldcg(A.p + (size_t)b * L::NPA + lane) : (lane < 8 ? 0.0 : __ldcg(A.p + (size_t)b * L::NPA + lane - 3));
  } else if (lane < NPAR) PAR(lane) = __ldcg(A.p + (size_t)b * NPAR + lane);      // (L2 path: a free-running call re-reads what its own epilogue wrote)
  if (lane == NPAR) PAR(NPAR) = A.weights ? A.weights[2 * (size_t)b] : A.pr.w1;
  if (lane == NPAR + 1) PAR(NPAR + 1) = A.weights ? A.weights[2 * (size_t)b + 1] : A.pr.w2;
  if (lane == NPAR + 2) PAR(NPAR + 2) = (double)b;      // instance index, for the per-stage target lookup
  const double* ob = A.obs + (A.obs_per_instance ? (size_t)b * 3 * L::NOBS : 0);
  for (int i = lane; i < 3 * L::NOBS; i += 32) smem[L::OBS0 + i] = ob[i];
  if (lane <= L::N) {
    const double* xx = A.x0 + (size_t)b * (L::NUA * L::N) + L::NUA * lane;
#pragma unroll
    for (int i = 0; i < 6; ++i) { LV(LV_U + i) = (lane < L::N && i < L::NUA) ? xx[i] : 0.0; LV(LV_DU + i) = 0.0; }
#pragma unroll 1
    for (int r = 0; r < L::R; ++r) { RW(A_DC, r) = 1.0; RW(A_DS, r) = 0.0; }
  }
  __syncwarp();
  if (A.tgt_pred) ph_predict<L>(A, b, lane, step);
}

// gradient-based scaling at the user's starting point (IPOPT nlp_scaling_method = gradient-based): returns df, sets DC
template <class L>
__device__ __noinline__ double ph_scaling(const SolveArgs& A, int lane) {
  const Prob& pr = A.pr; constexpr int N = L::N; const double T = pr.T;
  const bool act = lane <= N, hasu = lane < N;
  double u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = act ? LV(LV_U + i) : 0.0;
  Stage st; rollout<L::SW>(pr, &PAR(0), u, lane, st);
  const Dyn dy = dyn_entries(st, hasu ? T * u[0] : 0.0);
  double gl[6], Hl[21], a[8], lamn[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 0.0;
  if (hasu && lane >= 1) {
    cost_d2<L>(A, st.X, lane, gl, Hl);
#pragma unroll
    for (int v = 0; v < 6; ++v) a[cost_state(v)] = gl[v];
  }
  adjoint<L::SW>(a, dy, act, lane, lamn);
  double gmax = 0.0;
  if (hasu) {
    gmax = fabs(T * (st.cps * st.cth * lamn[0] + st.sps * st.cth * lamn[1] + st.sth * lamn[2]));
#pragma unroll
    for (int r = 1; r < 6; ++r) gmax = fmax(gmax, fabs(T * lamn[r + 2]));
  }
  gmax = warp_max(gmax);
  // row maxima of the Jacobian: |d g_{k,i} / d u_j| for j < k
  const double d0 = st.cps * st.cth, d1 = st.sps * st.cth, d2 = st.sth;
  double c3[3] = {dy.e03, dy.e13, dy.e23}, c4[2] = {dy.e04, dy.e14};
  scan_excl<3, L::SW>(c3, lane); scan_excl<2, L::SW>(c4, lane);
  double zmax = 0.0;
  // scratch in row arrays that are not live yet (ph_start initialises them): A_Y = row max, A_S / A_IU = obstacle normal
  if (act) {
#pragma unroll 1
    for (int jn = 0; jn < L::NOBS; ++jn) {
      double nx, ny, iD; obs_value<L>(st.X, jn, nx, ny, iD);
      RW(A_Y, L::NB + jn) = 0.0; RW(A_S, L::NB + jn) = nx; RW(A_IU, L::NB + jn) = ny;
    }
  }
#pragma unroll 1
  for (int jj = 0; jj < N; ++jj) {
    const double dj0 = __shfl_sync(FULL, d0, jj), dj1 = __shfl_sync(FULL, d1, jj), dj2 = __shfl_sync(FULL, d2, jj);
    const double a30 = __shfl_sync(FULL, c3[0], jj + 1), a31 = __shfl_sync(FULL, c3[1], jj + 1), a32 = __shfl_sync(FULL, c3[2], jj + 1);
    const double a40 = __shfl_sync(FULL, c4[0], jj + 1), a41 = __shfl_sync(FULL, c4[1], jj + 1);
    if (act && jj < lane) {
      const double pv0 = T * dj0, pv1 = T * dj1, pv2 = T * dj2;
      const double pt0 = T * (c3[0] - a30), pt1 = T * (c3[1] - a31), pt2 = T * (c3[2] - a32);
      const double pp0 = T * (c4[0] - a40), pp1 = T * (c4[1] - a41);
      zmax = fmax(zmax, fmax(fabs(pv2), fabs(pt2)));
#pragma unroll 1
      for (int jn = 0; jn < L::NOBS; ++jn) {
        const double nx = RW(A_S, L::NB + jn), ny = RW(A_IU, L::NB + jn);
        const double m1 = fabs(nx * pv0 + ny * pv1), m2 = fabs(nx * pt0 + ny * pt1), m3 = fabs(nx * pp0 + ny * pp1);
        RW(A_Y, L::NB + jn) = fmax(RW(A_Y, L::NB + jn), fmax(m1, fmax(m2, m3)));
      }
    }
  }
  if (act) {
    const double mg = A.o.max_grad, smin = A.o.scal_min;
    RW(A_DC, 0) = zmax > mg ? fmax(smin, mg / zmax) : 1.0;
    const double lin = lane >= 1 ? T : 0.0, sl = lin > mg ? fmax(smin, mg / lin) : 1.0;
#pragma unroll
    for (int r = 1; r < L::NB; ++r) RW(A_DC, r) = sl;
#pragma unroll 1
    for (int jn = 0; jn < L::NOBS; ++jn) { const double m = RW(A_Y, L::NB + jn); RW(A_DC, L::NB + jn) = m > mg ? fmax(smin, mg / m) : 1.0; }
  }
  __syncwarp();
  return gmax > A.o.max_grad ? fmax(A.o.scal_min, A.o.max_grad / gmax) : 1.0;
}

// starting point: push controls and slacks inside their bounds, unit bound multipliers; returns #finite bounds
// warm (non-reference mode): multipliers from the caller's guesses (unscaled, CasADi's sign convention lam = upper - lower),
// pushed away from zero, smaller pushes of the primal point (WarmStartIterateInitializer)
template <class L>
__device__ __noinline__ int ph_start(const SolveArgs& A, int lane, int b_, double df, bool warm) {
  const Prob& pr = A.pr; constexpr int N = L::N;
  const bool act = lane <= N, hasu = lane < N;
  const double kb1 = warm ? A.o.ws_bound_push : A.o.bound_push, kb2 = warm ? A.o.ws_bound_frac : A.o.bound_frac;
  const double ks1 = warm ? A.o.ws_slack_push : A.o.bound_push, ks2 = warm ? A.o.ws_slack_frac : A.o.bound_frac;
  const double zmin = A.o.ws_mult_push, zcap = A.o.ws_mult_init_max;
  double u[6]; int nz = 0; bool bad_lb = false;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    u[i] = act ? LV(LV_U + i) : 0.0;
    if (hasu) {
      const Bnd b = ctl_bounds<L>(A, lane, i);
      u[i] = push_in(u[i], b.lo, b.hi, b.hl, b.hu, kb1, kb2);
      double zl = b.hl ? 1.0 : 0.0, zu = b.hu ? 1.0 : 0.0;
      if (warm && i < L::NUA) {
        const double lz = fmin(fmax(A.lam_x0[(size_t)b_ * (L::NUA * N) + L::NUA * lane + i] * df, -zcap), zcap);
        zl = b.hl ? fmax(-lz, zmin) : 0.0; zu = b.hu ? fmax(lz, zmin) : 0.0;
      }
      LV(LV_U + i) = u[i]; LV(LV_ZL + i) = zl; LV(LV_ZU + i) = zu;
      nz += (b.hl ? 1 : 0) + (b.hu ? 1 : 0);
    } else if (act) { LV(LV_ZL + i) = 0.0; LV(LV_ZU + i) = 0.0; }
  }
  Stage st; rollout<L::SW>(pr, &PAR(0), u, lane, st);
  if (act) {
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double dc = RW(A_DC, r);
      const double g = __dmul_rn(dc, gu);
      const Bnd b = row_bounds<L>(A, lane, r, dc);
      const double s = push_in(g, b.lo, b.hi, b.hl, b.hu, ks1, ks2);
      double y = 0.0, vl = b.hl ? 1.0 : 0.0, vu = b.hu ? 1.0 : 0.0;
      if (warm) {      // y_d from the caller; v from y_d = v_U - v_L
        y = fmin(fmax(A.lam_g0[(size_t)b_ * (L::R * L::S) + lane * L::R + r] * df / dc, -zcap), zcap);
        vl = b.hl ? fmax(-y, zmin) : 0.0; vu = b.hu ? fmax(y, zmin) : 0.0;
      }
      RW(A_S, r) = s; RW(A_Y, r) = y;
      RW(A_VU, r) = vu; RW(A_IU, r) = b.hu ? rcp(b.hi - s) : 0.0;
      if (box) { RW(A_VL, r) = vl; RW(A_IL, r) = b.hl ? rcp(s - b.lo) : 0.0; }
      else if (b.hl) bad_lb = true;                     // a lower bound on an obstacle row: not this NLP family
      nz += (b.hl ? 1 : 0) + (b.hu ? 1 : 0);
    };
    stash_box_states<L>(st.X, lane);
    auto xb = [&](int si) { return stash<L>(si, lane); };
    FOR_ROWS(xb, st.X, body);
  }
  __syncwarp();
  const int total = __reduce_add_sync(FULL, nz);
  return __any_sync(FULL, bad_lb) ? -1 : total;
}

// ---------------------------------------------------------------------------------------------------
// derivatives at the current point: stage Hessian blocks / gradients of the LQ sub-problem into LQ, optimality
// error ingredients into RES.  ls = least-squares multiplier system (W = 0, Sigma = I, rhs = gradient of L).
// RS (restoration problem): no tracking cost; the objective rho*sum(n+p) + eta/2 ||D_R (u - u_R)||^2 adds eta*D_R^2
// to the control diagonal and its gradient to the control right-hand side; rows enter with the weight Om(dw) instead
// of Sigma_s + dw, so this phase is re-run for every inertia-correction value dw.
template <class L, bool RS>
__device__ __noinline__ void ph_derivs(const SolveArgs& A, int lane, bool ls, double df, double mu, double dw, int flags, double* cold) {
  const Prob& pr = A.pr; constexpr int N = L::N; const double T = pr.T;
  const bool want1 = flags & 1;
  const bool act = lane <= N, hasu = lane < N;
  double u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = act ? LV(LV_U + i) : 0.0;
  Stage st; rollout<L::SW>(pr, &PAR(0), u, lane, st);
  const Dyn dy = dyn_entries(st, hasu ? T * u[0] : 0.0);
  double gl[6], Hl[21];
#pragma unroll
  for (int v = 0; v < 6; ++v) gl[v] = 0.0;
#pragma unroll
  for (int e = 0; e < 21; ++e) Hl[e] = 0.0;
  double l = 0.0;
  if (!RS) {
    if (hasu) l = cost_d2<L>(A, st.X, lane, gl, Hl);
    if (lane == 0) {   // stage 0 is constant in w
#pragma unroll
      for (int v = 0; v < 6; ++v) gl[v] = 0.0;
#pragma unroll
      for (int e = 0; e < 21; ++e) Hl[e] = 0.0;
    }
  }
  const double fsum = RS ? 0.0 : df * warp_sum(l);
  double a[8], qa[8], qb[8], qd[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { a[i] = 0.0; qa[i] = 0.0; qb[i] = 0.0; qd[i] = 0.0; }
  double du_l = 0.0, pr_l = 0.0, sumy = 0.0, sumz = 0.0, viol = 0.0, pmax = 0.0, pmin = CUDART_INF;
  double du1 = 0.0, pr1 = 0.0, co1 = 0.0, oth = 0.0, oinf = 0.0;
  // want1: also the 1-norms the soft restoration phase tests (rare; the hot path skips them)
  auto compl_ = [&](double pz) { pmax = fmax(pmax, pz); pmin = fmin(pmin, pz); if (want1) co1 += fabs(pz - mu); };
  if (act) {
#pragma unroll
    for (int i = 0; i < 8; ++i) LV(LV_X + i) = st.X[i];
#pragma unroll
    for (int v = 0; v < 6; ++v) { gl[v] *= df; LV(LV_GL + v) = gl[v]; a[cost_state(v)] = gl[v]; qa[cost_state(v)] = gl[v]; }
    double q66[21], nn[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int e = 0; e < 21; ++e) q66[e] = ls ? 0.0 : df * Hl[e];
    // The box rows run in a rolled loop, and each touches the entries of its own state si only (the obstacle rows touch
    // x, y only): their entries of a, qa, qb, qd and of the Hessian start in shared memory (a in the stash) and the rows
    // accumulate there.  The explicit fma is what the compiler made of `acc += dc * v` in the unrolled form.
#pragma unroll
    for (int i = 2; i < 8; ++i) {
      stash<L>(i, lane) = a[i]; LQ(LQ_QA + i) = qa[i];
      if (!L::FOLD) { LQ(LQ_QB + i) = 0.0; LQ(LQ_QD + i) = 0.0; }
    }
#pragma unroll
    for (int e = 3; e < 21; ++e) LQ(LQ_Q + e) = q66[e];
    LQ(LQ_Q + 21) = 0.0;
    const double kd = A.o.kappa_d;
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double dc = RW(A_DC, r);
      const double g = __dmul_rn(dc, gu);
      const double s = RW(A_S, r), y = RW(A_Y, r), vl = box ? RW(A_VL, r) : 0.0, vu = RW(A_VU, r), il = box ? RW(A_IL, r) : 0.0, iu = RW(A_IU, r);
      const bool hl = il > 0.0, hu = iu > 0.0;
      double c = g - s;
      const double sig = ls ? 1.0 : vl * il + vu * iu;
      double beta = iu - il;                              // barrier gradient per unit mu (with damping)
      if (hl && !hu) beta += kd;
      if (hu && !hl) beta -= kd;
      double ya, wk, yad;                                 // ya: delta_w- and mu-free part of y-hat; yad: seed of the adjoint; dc^2 wk: row weight
      if (RS) {
        oth += fabs(c); oinf = fmax(oinf, fabs(c));
        const RestoRow q = resto_row<L>(A, cold, lane, r, sig, beta, y, mu, dw);
        c += RG(G_N, r) - RG(G_P, r);
        const double chat = c + q.rs * rcp(q.D) + q.rp * rcp(q.Dp) - q.rn * rcp(q.Dn);
        ya = y + q.Om * chat; wk = q.Om; yad = y;
        // n / p parts of the optimality error
        const double gn = A.o.resto_rho + y - q.zn, gp = A.o.resto_rho - y - q.zp;
        du_l = fmax(du_l, fmax(fabs(gn), fabs(gp))); if (want1) du1 += fabs(gn) + fabs(gp);
        sumz += q.zn + q.zp;
        compl_(q.n * q.zn); compl_(q.p * q.zp);
      } else if (L::FOLD && !ls) {      // mu and delta_w folded in: Q gets G^T (Sigma_s + dw) G, q gets G^T ((Sigma_s + dw) c + mu beta)
        ya = (sig + dw) * c + mu * beta; wk = sig + dw; yad = y;
      } else {
        ya = ls ? (vu - vl) : sig * c; wk = sig; yad = y;
      }
      if (box) {
        stash<L>(si, lane) = __fma_rn(dc, yad, stash<L>(si, lane)); LQ(LQ_QA + si) = __fma_rn(dc, ya, LQ(LQ_QA + si));
        if (!RS && !L::FOLD) {
          LQ(LQ_QB + si) = ls ? 0.0 : __fma_rn(dc, beta, LQ(LQ_QB + si)); LQ(LQ_QD + si) = ls ? 0.0 : __fma_rn(dc, c, LQ(LQ_QD + si));
        }
        const int qi = si == 3 ? 21 : tri(si < 3 ? si : si - 2, si < 3 ? si : si - 2);
        LQ(LQ_Q + qi) = __fma_rn(dc * dc, wk, LQ(LQ_Q + qi));
        if (!L::FOLD) LQ(LQ_DG + r) = RS ? 0.0 : dc * dc;
      } else {
        const double w = dc * dc * wk;
        const double cur = ls ? 0.0 : -y * dc * iD;        // y * d2h,  d2h = -(I - n n^T)/D
        q66[0] += w * nx * nx + cur * (1.0 - nx * nx);
        q66[1] += w * nx * ny - cur * nx * ny;
        q66[2] += w * ny * ny + cur * (1.0 - ny * ny);
        if (!RS && !L::FOLD) { nn[0] += dc * dc * nx * nx; nn[1] += dc * dc * nx * ny; nn[2] += dc * dc * ny * ny; }
        const double gy = -dc * yad, ga = -dc * ya;
        a[0] += gy * nx; a[1] += gy * ny; qa[0] += ga * nx; qa[1] += ga * ny;
        if (!RS && !L::FOLD) {
          const double gb = -dc * beta, gd = -dc * c;
          qb[0] += gb * nx; qb[1] += gb * ny; qd[0] += gd * nx; qd[1] += gd * ny;
        }
      }
      // optimality-error ingredients
      const double gs = fabs(-y - vl + vu);
      du_l = fmax(du_l, gs); pr_l = fmax(pr_l, fabs(c)); sumy += fabs(y); sumz += vl + vu;
      if (want1) { du1 += gs; pr1 += fabs(c); }
      const Bnd b = row_bounds<L>(A, lane, r, dc);
      if (b.hl) compl_((s - b.lo) * vl);
      if (b.hu) compl_((b.hi - s) * vu);
      const double lo_o = __ldg(A.lbg + lane * L::R + r), hi_o = __ldg(A.ubg + lane * L::R + r);
      if (lo_o > -1e19) viol = fmax(viol, lo_o - gu);
      if (hi_o < 1e19) viol = fmax(viol, gu - hi_o);
    };
    auto xb = [&](int si) { return LV(LV_X + si); };
    FOR_ROWS(xb, st.X, body);
#pragma unroll
    for (int i = 2; i < 8; ++i) a[i] = stash<L>(i, lane);
#pragma unroll
    for (int e = 0; e < 3; ++e) LQ(LQ_Q + e) = q66[e];
    LQ(LQ_ZERO) = 0.0;
    LQ(LQ_QA + 0) = qa[0]; LQ(LQ_QA + 1) = qa[1];
    if (!L::FOLD) {
      LQ(LQ_NN + 0) = nn[0]; LQ(LQ_NN + 1) = nn[1]; LQ(LQ_NN + 2) = nn[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) { LQ(LQ_QB + i) = ls ? 0.0 : qb[i]; LQ(LQ_QD + i) = ls ? 0.0 : qd[i]; }
    }
    if (!L::FOLD && L::NB < 5) {      // rows that do not exist in this model
#pragma unroll
      for (int r = L::NB; r < 5; ++r) LQ(LQ_DG + r) = 0.0;
    }
    LQ(LQ_DD + 0) = st.cps * st.cth; LQ(LQ_DD + 1) = st.sps * st.cth; LQ(LQ_DD + 2) = st.sth;
    LQ(LQ_EE + 0) = dy.e03; LQ(LQ_EE + 1) = dy.e13; LQ(LQ_EE + 2) = dy.e23; LQ(LQ_EE + 3) = dy.e04; LQ(LQ_EE + 4) = dy.e14;
  }
  double lamn[8];
  adjoint<L::SW>(a, dy, act, lane, lamn);
  if (act) {
    double svt = 0.0, svp = 0.0, q33 = 0.0, q34 = 0.0, q44 = 0.0;
    if (hasu && !ls) {
      // curvature of T*v*d(theta,psi) weighted by the next-stage adjoint
      const double L0 = T * lamn[0], L1 = T * lamn[1], L2 = T * lamn[2], v = u[0];
      const double cc = st.cps * st.cth, sc = st.sps * st.cth, cs = st.cps * st.sth, ss = st.sps * st.sth;
      q33 = -v * (L0 * cc + L1 * sc + L2 * st.sth);
      q44 = -v * (L0 * cc + L1 * sc);
      q34 = v * (L0 * ss - L1 * cs);
      svt = -L0 * cs - L1 * ss + L2 * st.cth;
      svp = -L0 * sc + L1 * cc;
    }
    LQ(LQ_Q + 21) += q33; LQ(LQ_Q + 22) = q34; LQ(LQ_Q + 23) = q44;
    LQ(LQ_SV + 0) = svt; LQ(LQ_SV + 1) = svp;
    // controls: Sigma_x, gradient per unit mu, dual infeasibility, complementarity products
    // (the gradient glx goes through the stash to the rolled control loop)
    stash<L>(0, lane) = T * (st.cps * st.cth * lamn[0] + st.sps * st.cth * lamn[1] + st.sth * lamn[2]);
#pragma unroll
    for (int r = 1; r < 6; ++r) stash<L>(r, lane) = T * lamn[r + 2];
    const double eta = RS ? A.o.resto_eta_factor * sqrt(mu) : 0.0;
#pragma unroll 1
    for (int i = 0; i < 6; ++i) {
      double sig = 1.0, rb = 0.0;       // absent controls (model 1) keep the unit diagonal and a zero right-hand side
      if (hasu && i < L::NUA) {
        const Bnd b = ctl_bounds<L>(A, lane, i);
        const double ui = LV(LV_U + i), zl = LV(LV_ZL + i), zu = LV(LV_ZU + i);
        const double sl = (ui - b.lo), su = (b.hi - ui);
        double gli = stash<L>(i, lane), gR = 0.0;
        if (RS) { const double ur = UREF(i), d = rcp(fmax(1.0, fabs(ur))); gR = eta * d * d * (ui - ur); gli += gR; }
        if (ls) rb = zu - zl;
        else {
          const double il = b.hl ? rcp(sl) : 0.0, iu = b.hu ? rcp(su) : 0.0;
          sig = zl * il + zu * iu; rb = iu - il;
          if (b.hl && !b.hu) rb += A.o.kappa_d;
          if (b.hu && !b.hl) rb -= A.o.kappa_d;
          if (RS) { const double ur = UREF(i), d = rcp(fmax(1.0, fabs(ur))); sig += eta * d * d; rb += gR / mu; }
        }
        const double gx = fabs(gli - zl + zu);
        du_l = fmax(du_l, gx); if (want1) du1 += gx;
        sumz += zl + zu;
        if (b.hl) compl_(sl * zl);
        if (b.hu) compl_(su * zu);
      }
      LQ(LQ_RD + i) = sig; LQ(LQ_RB + i) = rb;
    }
  }
  du_l = warp_max(du_l); pr_l = warp_max(pr_l); sumy = warp_sum(sumy); sumz = warp_sum(sumz);
  viol = warp_max(viol); pmax = warp_max(pmax); pmin = warp_min(pmin);
  if (want1) { du1 = warp_sum(du1); pr1 = warp_sum(pr1); co1 = warp_sum(co1); }
  if (RS) { oth = warp_sum(oth); oinf = warp_max(oinf); }
  if (lane == 0) {
    RES(R_F) = fsum; RES(R_DU) = du_l; RES(R_PR) = pr_l; RES(R_SUMY) = sumy; RES(R_SUMZ) = sumz;
    RES(R_VIOL) = viol; RES(R_PMAX) = pmax; RES(R_PMIN) = pmin;
    if (want1) { RES(R_DU1) = du1; RES(R_THETA) = pr1; RES(R_CO1) = co1; }
    if (RS) { RES(R_OTH) = oth; RES(R_OINF) = oinf; }
  }
  __syncwarp();
}

// least-squares multipliers from the solved LS system: y = G dx + (v_U - v_L); zero if too large
template <class L>
__device__ __noinline__ void ph_lsy(const SolveArgs& A, int lane, bool ok) {
  const bool act = lane <= L::N;
  double ymax = 0.0;
  if (act && ok) {
    double X[8], dx[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { X[i] = LV(LV_X + i); dx[i] = LV(LV_DX + i); }
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double dc = RW(A_DC, r);
      const double gd = box ? dc * LV(LV_DX + si) : -dc * (nx * dx[0] + ny * dx[1]);
      const double yv = gd + (RW(A_VU, r) - (box ? RW(A_VL, r) : 0.0));
      RW(A_Y, r) = yv; ymax = fmax(ymax, fabs(yv));
    };
    auto xb = [&](int si) { return LV(LV_X + si); };
    FOR_ROWS(xb, X, body);
  }
  ymax = warp_max(ymax);
  if (!ok || !(ymax <= A.o.constr_mult_init_max)) {
    if (act) {
#pragma unroll 1
      for (int r = 0; r < L::R; ++r) RW(A_Y, r) = 0.0;
    }
  }
  __syncwarp();
}

// step in the slacks (and in n, p for RS), fraction-to-the-boundary limits, directional derivative of the barrier
// function, max |dy|.  soc: second-order-correction direction (residual CSOC, controls DUS, output DS2).
template <class L, bool RS>
__device__ __noinline__ void ph_dir(const SolveArgs& A, int lane, double mu, double tau, bool soc, double dw, double* cold) {
  const bool act = lane <= L::N, hasu = lane < L::N;
  double tp = 0.0, dnum = 0.0, dden = 1.0, gbd = 0.0, theta = 0.0, dymax = 0.0; bool nottiny = false;
  const double tt = A.o.tiny_step_tol, kd = A.o.kappa_d;
  auto dual_frac = [&](double z, double dz) {   // track max of -dz/z over dz < 0 as a fraction
    if (dz < 0.0 && -dz * dden > dnum * z) { dnum = -dz; dden = z; }
  };
  if (act) {
    double X[8], dx[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { X[i] = LV(LV_X + i); dx[i] = LV(LV_DX + i); }
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double dc = RW(A_DC, r), s = RW(A_S, r), il = box ? RW(A_IL, r) : 0.0, iu = RW(A_IU, r), vl = box ? RW(A_VL, r) : 0.0, vu = RW(A_VU, r);
      const bool hl = il > 0.0, hu = iu > 0.0;
      double beta = iu - il;
      if (hl && !hu) beta += kd;
      if (hu && !hl) beta -= kd;
      const double gd = box ? dc * LV(LV_DX + si) : -dc * (nx * dx[0] + ny * dx[1]);
      double c, ds;
      if (RS) {
        const double y = RW(A_Y, r);
        const RestoRow q = resto_row<L>(A, cold, lane, r, vl * il + vu * iu, beta, y, mu, dw);
        c = soc ? RG(G_CSOC, r) : __dmul_rn(dc, gu) + RG(G_N, r) - RG(G_P, r) - s;
        const double chat = c + q.rs * rcp(q.D) + q.rp * rcp(q.Dp) - q.rn * rcp(q.Dn);
        const double dyv = q.Om * (gd + chat);
        // dy first, then ds, dn, dp from their own dual equations: exact dual consistency whatever the rounding of the D's
        const double dn = -(dyv + q.rn) * rcp(q.Dn), dp = (dyv - q.rp) * rcp(q.Dp);
        ds = (dyv - q.rs) * rcp(q.D);
        if (soc) { RG(G_DN2, r) = dn; RG(G_DP2, r) = dp; RG(G_DY2, r) = dyv; } else { RG(G_DN, r) = dn; RG(G_DP, r) = dp; RG(G_DY, r) = dyv; }
        const double in_ = rcp(q.n), ip_ = rcp(q.p);
        tp = fmax(tp, fmax(-dn * in_, -dp * ip_));
        dual_frac(q.zn, (mu - q.zn * dn) * in_ - q.zn);
        dual_frac(q.zp, (mu - q.zp * dp) * ip_ - q.zp);
        gbd += (A.o.resto_rho - mu * in_ + kd * mu) * dn + (A.o.resto_rho - mu * ip_ + kd * mu) * dp;
        nottiny = nottiny || (fabs(dn) > tt * (1.0 + fabs(q.n))) || (fabs(dp) > tt * (1.0 + fabs(q.p)));
        dymax = fmax(dymax, fabs(dyv));
      } else {
        c = soc ? RG(G_CSOC, r) : __dmul_rn(dc, gu) - s;
        ds = gd + c;
        dymax = fmax(dymax, fabs((vl * il + vu * iu + dw) * ds + (mu * beta - RW(A_Y, r))));
      }
      if (soc) RG(G_DS2, r) = ds; else RW(A_DS, r) = ds;
      tp = fmax(tp, fmax(-ds * il, ds * iu));
      if (hl) dual_frac(vl, (mu - vl * ds) * il - vl);
      if (hu) dual_frac(vu, (mu + vu * ds) * iu - vu);
      gbd += mu * beta * ds; theta += fabs(c);
      nottiny = nottiny || (fabs(ds) > tt * (1.0 + fabs(s)));
    };
    auto xb = [&](int si) { return LV(LV_X + si); };
    FOR_ROWS(xb, X, body);
    if (hasu) {
      const double eta = RS ? A.o.resto_eta_factor * sqrt(mu) : 0.0;
#pragma unroll 1
      for (int i = 0; i < 6; ++i) {
        const Bnd b = ctl_bounds<L>(A, lane, i);
        const double u = LV(LV_U + i), du = soc ? SOC(SOC_DUS + i) : LV(LV_DU + i), zl = LV(LV_ZL + i), zu = LV(LV_ZU + i);
        const double il = b.hl ? rcp((u - b.lo)) : 0.0, iu = b.hu ? rcp((b.hi - u)) : 0.0;
        tp = fmax(tp, fmax(-du * il, du * iu));
        if (b.hl) dual_frac(zl, (mu - zl * du) * il - zl);
        if (b.hu) dual_frac(zu, (mu + zu * du) * iu - zu);
        double beta = iu - il;
        if (b.hl && !b.hu) beta += kd;
        if (b.hu && !b.hl) beta -= kd;
        gbd += mu * beta * du;
        if (RS) { const double ur = UREF(i), d = rcp(fmax(1.0, fabs(ur))); gbd += eta * d * d * (u - ur) * du; }
        nottiny = nottiny || (fabs(du) > tt * (1.0 + fabs(u)));
      }
      if (!RS) {
#pragma unroll
        for (int v = 0; v < 6; ++v) gbd += LV(LV_GL + v) * dx[cost_state(v)];
      }
    }
  }
  tp = warp_max(tp);
  const double td = warp_max(dnum / dden);
  gbd = warp_sum(gbd); theta = warp_sum(theta); dymax = warp_max(dymax);
  const bool any_nt = __any_sync(FULL, nottiny);
  if (lane == 0) {
    RES(R_APR) = tp > tau ? tau / tp : 1.0;             // alpha = min(1, tau / max ratio)
    RES(R_ADU) = td > tau ? tau / td : 1.0;
    if (!soc) { RES(R_GBD) = gbd; RES(R_THETA) = theta; RES(R_TINY) = any_nt ? 0.0 : 1.0; RES(R_DYMAX) = dymax; }
  }
  __syncwarp();
}

// trial point u + alpha*du, s + alpha*ds (n, p for RS): objective, constraint violation, barrier pieces; residual into CT.
// pair (Lay::PAIR layouts only): lanes SW .. 2 SW - 1 evaluate the point at alpha * alpha_red -- the trial that follows a
// plain rejection -- in the same instructions, stage k on lane SW + k, into R_FT2 .. R_DTT2.  The lower half computes
// exactly what it computes without pairing; the upper half does not store CT (only ph_socrhs reads it, after the trial at
// alpha_max, which is never a precomputed one).
template <class L, bool RS>
__device__ __noinline__ void ph_trial(const SolveArgs& A, int lane_, double alpha_, bool soc, double df, double mu, double* cold, bool pair) {
  const Prob& pr = A.pr;
  pair = L::PAIR && pair;
  const bool hi = pair && lane_ >= L::SW;
  const int lane = pair ? lane_ & (L::SW - 1) : lane_;      // stage index: every lane-indexed access below uses it
  const double alpha = hi ? alpha_ * A.o.alpha_red : alpha_;
  const bool act = lane <= L::N, hasu = lane < L::N;
  double ut[6], lb = 0.0, dt = 0.0, fr = 0.0;
  double prod = 1.0; int cnt = 0;
  // the trial controls go through the stash (physical lane: with pairing both halves use it) to the rollout
#pragma unroll 1
  for (int i = 0; i < 6; ++i) {
    double uti = 0.0;
    if (hasu) {
      uti = fma(alpha, soc ? SOC(SOC_DUS + i) : LV(LV_DU + i), LV(LV_U + i));   // same expression as ph_accept
      const Bnd b = ctl_bounds<L>(A, lane, i);
      if (b.hl) prod *= (uti - b.lo);
      if (b.hu) prod *= (b.hi - uti);
      if (b.hl && !b.hu) dt += uti - b.lo;
      if (b.hu && !b.hl) dt += b.hi - uti;
      if (i == 2 || i == 5) { lb += n_log(prod); prod = 1.0; }
      if (RS) { const double ur = UREF(i), d = rcp(fmax(1.0, fabs(ur))), e = d * (uti - ur); fr += e * e; }
    }
    stash<L>(i, lane_) = uti;
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) ut[i] = stash<L>(i, lane_);
  Stage st; rollout<L::SW>(pr, &PAR(0), ut, lane, st);
  double l = 0.0;
  if (!RS) l = hasu ? cost_val<L>(A, st.X, lane) : 0.0;
  else l = 0.5 * A.o.resto_eta_factor * sqrt(mu) * fr;
  double th = 0.0;
  if (act) {
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double dc = RW(A_DC, r);
      const double g = __dmul_rn(dc, gu);
      const double sv = fma(alpha, soc ? RG(G_DS2, r) : RW(A_DS, r), RW(A_S, r));
      double ct = g - sv;
      if (RS) {
        const double nt = fma(alpha, soc ? RG(G_DN2, r) : RG(G_DN, r), RG(G_N, r));
        const double pt = fma(alpha, soc ? RG(G_DP2, r) : RG(G_DP, r), RG(G_P, r));
        ct += nt - pt;
        const double ns = (nt), ps = (pt);
        prod *= ns * ps; cnt += 2; dt += ns + ps; l += A.o.resto_rho * (nt + pt);
      }
      if (!hi) RG(G_CT, r) = ct;      // (only the second-order correction reads it back)
      th += fabs(ct);
      const Bnd b = row_bounds<L>(A, lane, r, dc);
      if (b.hl) { prod *= (sv - b.lo); ++cnt; }
      if (b.hu) { prod *= (b.hi - sv); ++cnt; }
      if (b.hl && !b.hu) dt += sv - b.lo;
      if (b.hu && !b.hl) dt += b.hi - sv;
      if (cnt >= 4) { lb += n_log(prod); prod = 1.0; cnt = 0; }
    };
    stash_box_states<L>(st.X, lane_);
    auto xb = [&](int si) { return stash<L>(si, lane_); };
    FOR_ROWS(xb, st.X, body);
    if (cnt) lb += n_log(prod);
  }
  // per half-warp sums where pairing is possible (the lanes >= SW hold zeros when unpaired: lane 0's sums are warp_sum's)
  auto sum = [](double v) { if constexpr (L::PAIR) return seg_sum<L::SW>(v); else return warp_sum(v); };
  const double fs = (RS ? 1.0 : df) * sum(l);
  th = sum(th); lb = sum(lb); dt = sum(dt);
  if (lane_ == 0) { RES(R_FT) = fs; RES(R_THT) = th; RES(R_LBT) = lb; RES(R_DTT) = dt; }
  if (pair && lane_ == L::SW) { RES(R_FT2) = fs; RES(R_THT2) = th; RES(R_LBT2) = lb; RES(R_DTT2) = dt; }
  __syncwarp();
}

// SOC right-hand side: c_soc <- a_soc * c_soc + c(trial);  q' = grad l + G^T((Sigma_s + dw) c_soc + mu beta)
// (RS: q' = G^T (y + Om chat(c_soc)))
template <class L, bool RS>
__device__ __noinline__ void ph_socrhs(const SolveArgs& A, int lane, double a_soc, double mu, double dw, bool first, double* cold) {
  if (lane <= L::N) {
    double X[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { X[i] = LV(LV_X + i); q[i] = 0.0; }
    if (!RS) {
#pragma unroll
      for (int v = 0; v < 6; ++v) q[cost_state(v)] = LV(LV_GL + v);
    }
    const double kd = A.o.kappa_d;
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double dc = RW(A_DC, r), il = box ? RW(A_IL, r) : 0.0, iu = RW(A_IU, r);
      const bool hl = il > 0.0, hu = iu > 0.0;
      double c0 = __dmul_rn(dc, gu) - RW(A_S, r);
      if (RS) c0 += RG(G_N, r) - RG(G_P, r);
      const double cprev = first ? c0 : RG(G_CSOC, r);
      const double cs = a_soc * cprev + RG(G_CT, r);
      RG(G_CSOC, r) = cs;
      double beta = iu - il;
      if (hl && !hu) beta += kd;
      if (hu && !hl) beta -= kd;
      const double sig = (box ? RW(A_VL, r) : 0.0) * il + RW(A_VU, r) * iu;
      double yh;
      if (RS) {
        const double y = RW(A_Y, r);
        const RestoRow w = resto_row<L>(A, cold, lane, r, sig, beta, y, mu, dw);
        yh = y + w.Om * (cs + w.rs * rcp(w.D) + w.rp * rcp(w.Dp) - w.rn * rcp(w.Dn));
      } else yh = (sig + dw) * cs + mu * beta;
      if (box) SOC(SOC_Q2 + si) = __fma_rn(dc, yh, SOC(SOC_Q2 + si)); else { q[0] -= dc * yh * nx; q[1] -= dc * yh * ny; }
    };
#pragma unroll
    for (int i = 2; i < 8; ++i) SOC(SOC_Q2 + i) = q[i];      // box entries: accumulated in place by the rolled box rows
    auto xb = [&](int si) { return LV(LV_X + si); };
    FOR_ROWS(xb, X, body);
    SOC(SOC_Q2 + 0) = q[0]; SOC(SOC_Q2 + 1) = q[1];
  }
  __syncwarp();
}

// Slack safeguard (rare): repair the primal values whose slack fell below smin after a step, then give their
// multipliers the kappa_Sigma reset against the repaired slack (ph_accept left them un-reset) and refresh the
// reciprocal row slacks.
template <class L, bool RS>
__device__ __noinline__ void ph_repair(const SolveArgs& A, int lane, double mu, bool reset, double* cold) {
  const double ks = A.o.kappa_sigma, iks = 1.0 / A.o.kappa_sigma, smin = EPSM * fmin(1.0, mu);
  auto clampz = [&](double z, double sl) { const double i2 = rcp(sl); return reset ? fmax(fmin(z, ks * mu * i2), mu * i2 * iks) : z; };
  if (lane < L::N) {
#pragma unroll 1
    for (int i = 0; i < 6; ++i) {
      const Bnd b = ctl_bounds<L>(A, lane, i);
      double u = LV(LV_U + i);
      if (b.hl && u - b.lo < smin) { const double t = safe_value(u - b.lo, b.lo); u = b.lo + t; LV(LV_ZL + i) = clampz(LV(LV_ZL + i), t); }
      if (b.hu && b.hi - u < smin) { const double t = safe_value(b.hi - u, b.hi); u = b.hi - t; LV(LV_ZU + i) = clampz(LV(LV_ZU + i), t); }
      LV(LV_U + i) = u;
    }
  }
  if (lane <= L::N) {
#pragma unroll 1
    for (int r = 0; r < L::R; ++r) {
      const Bnd b = row_bounds<L>(A, lane, r, RW(A_DC, r));
      double s = RW(A_S, r);
      if (r < L::NB && b.hl && s - b.lo < smin) { const double t = safe_value(s - b.lo, b.lo); s = b.lo + t; RW(A_VL, r) = clampz(RW(A_VL, r), t); RW(A_IL, r) = rcp(t); }
      if (b.hu && b.hi - s < smin) { const double t = safe_value(b.hi - s, b.hi); s = b.hi - t; RW(A_VU, r) = clampz(RW(A_VU, r), t); RW(A_IU, r) = rcp(t); }
      RW(A_S, r) = s;
      if (RS) {
        double n = RG(G_N, r), p = RG(G_P, r);
        if (n < smin) { n = safe_value(n, 0.0); RG(G_N, r) = n; RG(G_ZN, r) = clampz(RG(G_ZN, r), n); }
        if (p < smin) { p = safe_value(p, 0.0); RG(G_P, r) = p; RG(G_ZP, r) = clampz(RG(G_ZP, r), p); }
      }
    }
  }
  __syncwarp();
}

// accept the trial point: primal step alpha, dual step a_du, kappa_Sigma reset (reset), new reciprocal slacks.
// Straight-line: a slack that comes out below smin only raises a flag (its multiplier is left un-reset) and the rare
// ph_repair fixes it up afterwards.
template <class L, bool RS>
__device__ __noinline__ void ph_accept(const SolveArgs& A, int lane, double alpha, double a_du, double mu, double dw, bool soc, bool reset,
                                       double* cold) {
  const bool act = lane <= L::N, hasu = lane < L::N;
  const double ks = A.o.kappa_sigma, kd = A.o.kappa_d, iks = 1.0 / A.o.kappa_sigma;
  const double smin = EPSM * fmin(1.0, mu);
  bool bad = false;
  if (hasu) {
#pragma unroll 1
    for (int i = 0; i < 6; ++i) {
      const Bnd b = ctl_bounds<L>(A, lane, i);
      const double u = LV(LV_U + i), du = soc ? SOC(SOC_DUS + i) : LV(LV_DU + i);
      double zl = LV(LV_ZL + i), zu = LV(LV_ZU + i);
      if (b.hl) zl += a_du * ((mu - zl * du) * rcp(u - b.lo) - zl);
      if (b.hu) zu += a_du * ((mu + zu * du) * rcp(b.hi - u) - zu);
      const double un = fma(alpha, du, u);
      if (b.hl) { const double sl = un - b.lo, i2 = rcp(sl); const bool un_ = sl < smin; bad = bad || un_; if (reset && !un_) zl = fmax(fmin(zl, ks * mu * i2), mu * i2 * iks); }
      if (b.hu) { const double sl = b.hi - un, i2 = rcp(sl); const bool un_ = sl < smin; bad = bad || un_; if (reset && !un_) zu = fmax(fmin(zu, ks * mu * i2), mu * i2 * iks); }
      LV(LV_U + i) = un; LV(LV_ZL + i) = zl; LV(LV_ZU + i) = zu;
    }
  }
  if (act) {
#pragma unroll 1
    for (int r = 0; r < L::R; ++r) {
      const double dc = RW(A_DC, r), s = RW(A_S, r), il = IL_(r), iu = RW(A_IU, r), y = RW(A_Y, r);
      const double ds = soc ? RG(G_DS2, r) : RW(A_DS, r);
      const bool hl = il > 0.0, hu = iu > 0.0;
      double vl = VL_(r), vu = RW(A_VU, r);
      double beta = iu - il;
      if (hl && !hu) beta += kd;
      if (hu && !hl) beta -= kd;
      const double dy = RS ? (soc ? RG(G_DY2, r) : RG(G_DY, r)) : (vl * il + vu * iu + dw) * ds + (mu * beta - y);
      RW(A_Y, r) = y + alpha * dy;
      if (hl) vl += a_du * ((mu - vl * ds) * il - vl);
      if (hu) vu += a_du * ((mu + vu * ds) * iu - vu);
      const double sn = fma(alpha, ds, s);
      const Bnd b = row_bounds<L>(A, lane, r, dc);
      double il2 = 0.0, iu2 = 0.0;
      if (hl) { const double sl = sn - b.lo; il2 = rcp(sl); const bool un_ = sl < smin; bad = bad || un_; if (reset && !un_) vl = fmax(fmin(vl, ks * mu * il2), mu * il2 * iks); }
      if (hu) { const double sl = b.hi - sn; iu2 = rcp(sl); const bool un_ = sl < smin; bad = bad || un_; if (reset && !un_) vu = fmax(fmin(vu, ks * mu * iu2), mu * iu2 * iks); }
      RW(A_S, r) = sn; RW(A_VU, r) = vu; RW(A_IU, r) = iu2;
      if (r < L::NB) { RW(A_VL, r) = vl; RW(A_IL, r) = il2; }
      if (RS) {
        const double n0 = RG(G_N, r), p0 = RG(G_P, r), zn0 = RG(G_ZN, r), zp0 = RG(G_ZP, r);
        const double dn = soc ? RG(G_DN2, r) : RG(G_DN, r), dp = soc ? RG(G_DP2, r) : RG(G_DP, r);
        double zn = zn0 + a_du * ((mu - zn0 * dn) * rcp(n0) - zn0);
        double zp = zp0 + a_du * ((mu - zp0 * dp) * rcp(p0) - zp0);
        const double nn_ = fma(alpha, dn, n0), pn_ = fma(alpha, dp, p0);
        const bool un1 = nn_ < smin, un2 = pn_ < smin;
        bad = bad || un1 || un2;
        if (reset && !un1) { const double i1 = rcp(nn_); zn = fmax(fmin(zn, ks * mu * i1), mu * i1 * iks); }
        if (reset && !un2) { const double i2 = rcp(pn_); zp = fmax(fmin(zp, ks * mu * i2), mu * i2 * iks); }
        RG(G_N, r) = nn_; RG(G_P, r) = pn_; RG(G_ZN, r) = zn; RG(G_ZP, r) = zp;
      }
    }
  }
  __syncwarp();
  if (__any_sync(FULL, bad)) ph_repair<L, RS>(A, lane, mu, reset, cold);
}

// ---- rare paths --------------------------------------------------------------------------------------------------
// save / restore the iterate (and the primal step) in a slot of the cold scratch
template <class L>
__device__ __noinline__ void ph_slot(double* cold, int slot, bool save, bool with_resto, int lane) {
  constexpr int S = L::S, RSZ = L::RSZ;
  double* sl = cold + L::CG_SLOT + slot * L::SLOT_N;
  auto cp = [&](int sm0, int off, int n) {
    for (int i = lane; i < n; i += 32) { if (save) sl[off + i] = smem[sm0 + i]; else smem[sm0 + i] = sl[off + i]; }
  };
  cp(L::LV0, 0, 18 * S);                                   // U, ZL, ZU
  cp(L::LV0 + LV_DX * S, 18 * S, 14 * S);                  // DX, DU
  cp(L::rw(A_S, 0), 32 * S, 3 * RSZ);                      // S, Y, VU
  cp(L::rw(A_IU, 0), 32 * S + 3 * RSZ, RSZ);               // IU
  cp(L::rw(A_VL, 0), 32 * S + 4 * RSZ, 2 * L::NB * S);      // VL, IL (box rows)
  constexpr int R0 = 32 * S + 4 * RSZ + 2 * L::NB * S;
  if (with_resto)
    for (int i = lane; i < 4 * RSZ; i += 32) { if (save) sl[R0 + i] = cold[i]; else cold[i] = sl[R0 + i]; }
  __syncwarp();
}

// RestoIterateInitializer: elastic variables from the closed-form minimiser, their multipliers mu / value, bound
// multipliers min(rho, .), y = 0, reference point x_R = current controls.  LV_X holds the states of the current point.
template <class L>
__device__ __noinline__ void ph_resto_init(const SolveArgs& A, int lane, double mu, double* cold) {
  const double rho = A.o.resto_rho, h = mu / (2.0 * rho);
  if (lane <= L::N) {
    double X[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) X[i] = LV(LV_X + i);
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double c = __dmul_rn(RW(A_DC, r), gu) - RW(A_S, r);
      const double a = h - 0.5 * c, nv = a + sqrt(a * a + c * h), pv = c + nv;
      RG(G_N, r) = nv; RG(G_P, r) = pv; RG(G_ZN, r) = mu / nv; RG(G_ZP, r) = mu / pv;
      if (box) RW(A_VL, r) = fmin(rho, RW(A_VL, r));
      RW(A_VU, r) = fmin(rho, RW(A_VU, r)); RW(A_Y, r) = 0.0;
    };
    auto xb = [&](int si) { return LV(LV_X + si); };
    FOR_ROWS(xb, X, body);
#pragma unroll
    for (int i = 0; i < 6; ++i) { UREF(i) = LV(LV_U + i); LV(LV_ZL + i) = fmin(rho, LV(LV_ZL + i)); LV(LV_ZU + i) = fmin(rho, LV(LV_ZU + i)); }
  }
  __syncwarp();
}
// RestoRestorationPhase (restoration inside the restoration phase): recompute n, p for the current x, s
template <class L>
__device__ __noinline__ void ph_resto_np(const SolveArgs& A, int lane, double mu, double* cold) {
  const double rho = A.o.resto_rho, h = mu / (2.0 * rho);
  if (lane <= L::N) {
    double X[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) X[i] = LV(LV_X + i);
    auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) {
      const double c = __dmul_rn(RW(A_DC, r), gu) - RW(A_S, r);
      const double a = h - 0.5 * c, nv = a + sqrt(a * a + c * h);
      RG(G_N, r) = nv; RG(G_P, r) = c + nv; RG(G_DN, r) = 0.0; RG(G_DP, r) = 0.0; RG(G_DY, r) = 0.0;
    };
    auto xb = [&](int si) { return LV(LV_X + si); };
    FOR_ROWS(xb, X, body);
  }
  __syncwarp();
}
// MinC_1NrmRestorationPhase, after a successful restoration: bound multipliers of the original problem as if the
// whole phase had been one primal-dual step from the iterate saved in slot `slot`; y = 0.  Two passes: pass 0 returns
// the largest -dz/z over decreasing multipliers (RES(R_ADU) <- step), pass 1 applies the step and returns max z.
template <class L>
__device__ __noinline__ double ph_resto_finish(const SolveArgs& A, int lane, double mu, double tau, double a_du, int pass, double* cold, int slot) {
  constexpr int S = L::S;
  const double* sl = cold + L::CG_SLOT + slot * L::SLOT_N;
  double dnum = 0.0, dden = 1.0, zmax = 0.0;
  auto upd = [&](double z0, double sl0, double sl1, double& znew) {
    const double dz = (mu + z0 * (sl0 - sl1)) * rcp(sl0) - z0;
    if (pass == 0) { if (dz < 0.0 && -dz * dden > dnum * z0) { dnum = -dz; dden = z0; } }
    else { znew = z0 + a_du * dz; zmax = fmax(zmax, znew); }
  };
  if (lane < L::N) {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const Bnd b = ctl_bounds<L>(A, lane, i);
      const double u0 = sl[(LV_U + i) * S + lane], zl0 = sl[(LV_ZL + i) * S + lane], zu0 = sl[(LV_ZU + i) * S + lane], u1 = LV(LV_U + i);
      double zl = 0.0, zu = 0.0;
      if (b.hl) upd(zl0, (u0 - b.lo), (u1 - b.lo), zl);
      if (b.hu) upd(zu0, (b.hi - u0), (b.hi - u1), zu);
      if (pass == 1) { LV(LV_ZL + i) = zl; LV(LV_ZU + i) = zu; }
    }
  }
  if (lane <= L::N) {
#pragma unroll 1
    for (int r = 0; r < L::R; ++r) {
      const double dc = RW(A_DC, r);
      const Bnd b = row_bounds<L>(A, lane, r, dc);
      const double s0 = sl[32 * S + (A_S * L::R + r) * S + lane], vu0 = sl[32 * S + (A_VU * L::R + r) * S + lane];
      const double vl0 = r < L::NB ? sl[32 * S + 4 * L::RSZ + r * S + lane] : 0.0;
      const double s1 = RW(A_S, r);
      double vl = 0.0, vu = 0.0;
      if (b.hl && r < L::NB) upd(vl0, (s0 - b.lo), (s1 - b.lo), vl);
      if (b.hu) upd(vu0, (b.hi - s0), (b.hi - s1), vu);
      if (pass == 1) { if (r < L::NB) RW(A_VL, r) = vl; RW(A_VU, r) = vu; RW(A_Y, r) = 0.0; RW(A_DS, r) = 0.0; }
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) if (pass == 1) LV(LV_DU + i) = 0.0;
  }
  __syncwarp();
  if (pass == 0) { const double td = warp_max(dnum / dden); return td > tau ? tau / td : 1.0; }
  return warp_max(zmax);
}
// all bound multipliers <- 1 (bound_mult_reset_threshold exceeded after the restoration phase)
template <class L>
__device__ __noinline__ void ph_unit_mults(const SolveArgs& A, int lane) {
  if (lane < L::N) {
#pragma unroll
    for (int i = 0; i < 6; ++i) { const Bnd b = ctl_bounds<L>(A, lane, i); LV(LV_ZL + i) = b.hl ? 1.0 : 0.0; LV(LV_ZU + i) = b.hu ? 1.0 : 0.0; }
  }
  if (lane <= L::N) {
#pragma unroll 1
    for (int r = 0; r < L::R; ++r) { if (r < L::NB) RW(A_VL, r) = RW(A_IL, r) > 0.0 ? 1.0 : 0.0; RW(A_VU, r) = RW(A_IU, r) > 0.0 ? 1.0 : 0.0; }
  }
  __syncwarp();
}

// outputs: honour the original bounds, unscale multipliers, f and g at the returned point; KEEP (the kernel instantiation
// that NMPC_KEEP_BARRIER selects): also the barrier data sig_x / sig_g
template <class L, bool KEEP = false>
__device__ __noinline__ void ph_output(const SolveArgs& A, int b, int lane, double df, int status, int iter, int step) {
  const Prob& pr = A.pr; constexpr int N = L::N, R = L::R, S = L::S;
  const bool act = lane <= N, hasu = lane < N;
  constexpr int nw = L::NUA * N, ng = R * S;
  double u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = 0.0;
  if (hasu) {
#pragma unroll
    for (int i = 0; i < L::NUA; ++i) u[i] = fmin(fmax(LV(LV_U + i), __ldg(A.lbx + L::NUA * lane + i)), __ldg(A.ubx + L::NUA * lane + i));
    if (A.x) {
      double* xo = A.x + (size_t)b * nw + L::NUA * lane;
#pragma unroll
      for (int i = 0; i < L::NUA; ++i) xo[i] = u[i];
    }
    if (A.lam_x) {
      double* lo = A.lam_x + (size_t)b * nw + L::NUA * lane;
      const double idf = 1.0 / df;
#pragma unroll
      for (int i = 0; i < L::NUA; ++i) lo[i] = (LV(LV_ZU + i) - LV(LV_ZL + i)) * idf;
    }
    if (KEEP) {      // Sigma_x of the final iterate as ph_derivs forms it, unscaled (the objective scaling df divides out)
      double* so = A.sig_x + (size_t)b * nw + L::NUA * lane;
      const double idf = 1.0 / df;
#pragma unroll 1
      for (int i = 0; i < L::NUA; ++i) {
        const Bnd c = ctl_bounds<L>(A, lane, i);
        const double ui = LV(LV_U + i), il = c.hl ? rcp(ui - c.lo) : 0.0, iu = c.hu ? rcp(c.hi - ui) : 0.0;
        so[i] = (LV(LV_ZL + i) * il + LV(LV_ZU + i) * iu) * idf;
      }
    }
  }
  Stage st; rollout<L::SW>(pr, &PAR(0), u, lane, st);
  const double l = hasu ? cost_val<L>(A, st.X, lane) : 0.0;
  const double fu = warp_sum(l);
  if (lane == 0) {
    if (A.f) A.f[b] = fu;
    if (A.status) A.status[b] = status;
    if (A.iters) A.iters[b] = iter;
    if (A.iters_keep) {      // drives the next call's longest-first order: the mean over the steps of a free-running call
      const int acc = (step == 0 ? 0 : A.iters_keep[b]) + iter;
      A.iters_keep[b] = (A.run_steps > 1 && step == A.run_steps - 1) ? acc / A.run_steps : acc;
    }
    if (A.status_log) A.status_log[(size_t)step * A.B + b] = status;
    if (A.iters_log) A.iters_log[(size_t)step * A.B + b] = iter;
    if (A.conv_count && status == NMPC_SOLVE_SUCCEEDED) A.conv_count[b] += 1;
  }
  if (act) {
    if (A.g) {
      double* go = A.g + (size_t)b * ng + lane * R;
      auto body = [&](const int r, const bool box, const int si, const double gu, double nx, double ny, double iD) { go[r] = gu; };
      stash_box_states<L>(st.X, lane);
      auto xb = [&](int si) { return stash<L>(si, lane); };
      FOR_ROWS(xb, st.X, body);
    }
    if (A.lam_g) {
      double* lo = A.lam_g + (size_t)b * ng + lane * R;
      const double idf = 1.0 / df;
#pragma unroll 1
      for (int r = 0; r < R; ++r) lo[r] = RW(A_Y, r) * RW(A_DC, r) * idf;
    }
    if (KEEP) {      // Sigma_s of the final iterate, unscaled: the scaled row weight enters the Newton matrix as dc^2 Sigma_s / df
      double* so = A.sig_g + (size_t)b * ng + lane * R;
      const double idf = 1.0 / df;
#pragma unroll 1
      for (int r = 0; r < R; ++r) { const double dc = RW(A_DC, r); so[r] = (VL_(r) * IL_(r) + RW(A_VU, r) * RW(A_IU, r)) * (dc * dc) * idf; }
    }
  }
  if (A.step_p) {     // fused closed-loop shift of this instance (NMPC_TT.py:13-30): warm start, plant, target, FOV error
    double* uw = A.step_u + (size_t)b * nw;
#pragma unroll
    for (int i = 0; i < L::NUA; ++i) {
      const double un = __shfl_down_sync(FULL, u[i], 1);          // control of the next stage
      if (lane < N - 1) uw[L::NUA * lane + i] = un;               // drop the first stage ...
      else if (lane == N - 1) uw[L::NUA * lane + i] = u[i];       // ... and repeat the last (:20-23)
    }
    if (A.ws_shift && A.lam_x0) {     // next step's multiplier guesses: this solve's, one stage on (NaN marker after a failed solve)
      const double idf = 1.0 / df;
      double* lx = A.lam_x0 + (size_t)b * nw; double* lg = A.lam_g0 + (size_t)b * ng;
#pragma unroll
      for (int i = 0; i < L::NUA; ++i) {
        const double v = (LV(LV_ZU + i) - LV(LV_ZL + i)) * idf, vn = __shfl_down_sync(FULL, v, 1);
        if (lane < N - 1) lx[L::NUA * lane + i] = vn; else if (lane == N - 1) lx[L::NUA * lane + i] = v;
      }
#pragma unroll 1
      for (int r = 0; r < R; ++r) {
        const double v = act ? RW(A_Y, r) * RW(A_DC, r) * idf : 0.0, vn = __shfl_down_sync(FULL, v, 1);
        if (lane < N) lg[lane * R + r] = vn; else if (lane == N) lg[lane * R + r] = v;
      }
      __syncwarp();
      if (lane == 0 && status != NMPC_SOLVE_SUCCEEDED) lx[0] = CUDART_NAN;
    }
    if (lane == 0) {
      const double2 vw = target_input(A, b, step);
      closed_loop_shift_model(L::MODEL, pr.T, pr.hv, pr.hh, A.step_p + (size_t)b * L::NPA, u, vw.x, vw.y,
                        A.step_fov ? A.step_fov + 2 * (size_t)b : nullptr, A.step_err ? A.step_err + b : nullptr);
    }
    if (A.obs_move) {     // moving obstacles: o += T v from the copy this solve used (the rows g above saw the positions before the move),
                          // rounded as the torch update o + (T v); the lane mapping is ph_load's, so the next step of a free-running
                          // call reads its own write
      const double* vel = A.obs_vel + (size_t)b * 2 * L::NOBS;
      double* om = A.obs_move + (size_t)b * 3 * L::NOBS;
      for (int i = lane; i < 3 * L::NOBS; i += 32) {
        const int j = i / 3, c = i - 3 * j;
        if (c < 2) om[i] = __dadd_rn(smem[L::OBS0 + i], __dmul_rn(pr.T, __ldg(vel + 2 * j + c)));
      }
    }
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------
// State of one run of the algorithm (IpoptAlgorithm + BacktrackingLineSearch + FilterLSAcceptor members) lives in the
// warp's shared-memory slice (Lay::ALG0), as doubles: every lane holds the same value of everything below, so plain
// stores may be issued by all lanes and read-modify-writes go through al_add().  The restoration phase is a second run of
// the same algorithm on the restoration problem; the original run's fields [0, F_NALG) are parked in the cold scratch
// meanwhile.  Keeping this state out of registers keeps the hot loop free of spills across the phase calls, and lets the
// rare paths (watchdog stop, soft restoration, restoration entry / exit) be separate functions.
enum AlgF {
  F_MU = 0, F_TAU, F_DWLAST, F_TOL, F_THMAX, F_THMIN, F_RTH, F_RBARR, F_RGBD,      // barrier parameter, filter reference point
  F_F, F_LB, F_DT,                                  // objective and barrier pieces (sum of logs, damping sum) of the current point
  F_WTH, F_WBARR, F_WGBD, F_WAT, F_WDW,             // watchdog reference
  F_INFPR,                                          // max-norm of g - s where the restoration phase was called
  F_NFILT, F_SUCC, F_NRES, F_WSHORT, F_WTRIAL, F_SOFTC,
  F_LASTREJ, F_INWD, F_INSOFT, F_TINYLAST, F_TINYFLAG, F_FIRST, F_MUST,
  F_PWPHI, F_PWTH,                                  // (-F_RGBD)^s_phi and delta * F_RTH^s_theta of the switching condition, computed once per reference point (< 0: not yet)
  F_NALG,
  F_MODE = F_NALG,                                  // 0 original problem, 1 restoration problem
  F_DW, F_APR, F_ADU, F_GBD, F_THETA, F_PHI,        // this iteration: delta_w, step limits, barrier slope, theta, barrier of the current point
  F_C0,                                             // NSTAT work counters
  F_END = F_C0 + NSTAT
};
static_assert(F_END <= ALG_N, "algorithm state does not fit its shared-memory region");
#define AL(f) smem[L::ALG0 + (f)]

template <class L>
__device__ __forceinline__ double al_add(int f, double d) { const double v = AL(f) + d; __syncwarp(); AL(f) = v; return v; }
template <class L>
__device__ __forceinline__ void al_count(int c, int lane) { if (lane == 0) AL(F_C0 + c) += 1.0; }
template <class L>
__device__ __noinline__ void alg_init(double mu, double tau_min, double tol) {
  __syncwarp();
#pragma unroll 1
  for (int f = 0; f < F_NALG; ++f) AL(f) = 0.0;
  __syncwarp();
  AL(F_MU) = mu; AL(F_TAU) = fmax(tau_min, 1.0 - mu); AL(F_TOL) = tol; AL(F_THMAX) = -1.0; AL(F_THMIN) = -1.0; AL(F_FIRST) = 1.0;
  AL(F_PWPHI) = -1.0;
  __syncwarp();
}

// mode-dispatched phases
template <class L>
__device__ __forceinline__ void do_derivs(const SolveArgs& A, int lane, int mode, double df, double dw, int flags, double* cold) {
  if (mode) ph_derivs<L, true>(A, lane, false, df, AL(F_MU), dw, flags & 1, cold); else ph_derivs<L, false>(A, lane, false, df, AL(F_MU), dw, flags, cold);
}
template <class L>
__device__ __forceinline__ void do_dir(const SolveArgs& A, int lane, int mode, bool soc, double dw, double* cold) {
  if (mode) ph_dir<L, true>(A, lane, AL(F_MU), AL(F_TAU), soc, dw, cold); else ph_dir<L, false>(A, lane, AL(F_MU), AL(F_TAU), soc, dw, cold);
}
// one trial pass (counted as a line-search trial and as a pass); pair: see ph_trial
template <class L>
__device__ __forceinline__ void do_trial(const SolveArgs& A, int lane, int mode, double alpha, bool soc, double df, double* cold, bool pair = false) {
  if (mode) ph_trial<L, true>(A, lane, alpha, soc, df, AL(F_MU), cold, pair); else ph_trial<L, false>(A, lane, alpha, soc, df, AL(F_MU), cold, pair);
  al_count<L>(1, lane); al_count<L>(8, lane);
}
// the trial point the last paired pass evaluated ahead becomes the last trial point (a line-search trial without a pass)
template <class L>
__device__ __forceinline__ void take_ahead(int lane) {
  const double ft = RES(R_FT2), tht = RES(R_THT2), lbt = RES(R_LBT2), dtt = RES(R_DTT2);
  __syncwarp();
  RES(R_FT) = ft; RES(R_THT) = tht; RES(R_LBT) = lbt; RES(R_DTT) = dtt;     // every lane stores the same values
  __syncwarp();
  al_count<L>(1, lane);
}
template <class L>
__device__ __forceinline__ void do_accept(const SolveArgs& A, int lane, int mode, double alpha, double a_du, double dw, bool soc, bool reset, double* cold) {
  if (mode) ph_accept<L, true>(A, lane, alpha, a_du, AL(F_MU), dw, soc, reset, cold); else ph_accept<L, false>(A, lane, alpha, a_du, AL(F_MU), dw, soc, reset, cold);
}
// objective and barrier pieces of the last trial point become those of the current point
template <class L>
__device__ __forceinline__ void take_trial_values() { AL(F_F) = RES(R_FT); AL(F_LB) = RES(R_LBT); AL(F_DT) = RES(R_DTT); }
template <class L>
__device__ __forceinline__ double trial_barrier(const SolveArgs& A) { const double mu = AL(F_MU); return RES(R_FT) - mu * RES(R_LBT) + A.o.kappa_d * mu * RES(R_DTT); }

// ---- FilterLSAcceptor.  filter [FILT_CAP][2] = (barrier, theta) margins, in the cold scratch (a handful of loads per trial)
__device__ __forceinline__ bool filter_ok(const double* filt, int nfilt, double barr, double theta) {
  for (int e = 0; e < nfilt; ++e) {
    const double fb = filt[2 * e], ft = filt[2 * e + 1];
    if (!(cmp_le(barr, fb, fb) || cmp_le(theta, ft, ft))) return false;
  }
  return true;
}
// add (barr, theta), dropping the entries it dominates (and the oldest one if the filter is full); returns the new length
static __device__ __noinline__ int filter_add(double* filt, int nfilt, double barr, double theta, int lane) {
  int n = 0;
  __syncwarp();
  if (lane == 0) {
    for (int e = 0; e < nfilt; ++e) {
      const double fb = filt[2 * e], ft = filt[2 * e + 1];
      if (!(fb >= barr && ft >= theta)) { filt[2 * n] = fb; filt[2 * n + 1] = ft; ++n; }
    }
    if (n >= FILT_CAP) { for (int e = 0; e < 2 * (n - 1); ++e) filt[e] = filt[e + 2]; --n; }
    filt[2 * n] = barr; filt[2 * n + 1] = theta; ++n;
  }
  n = __shfl_sync(FULL, n, 0);
  __syncwarp();
  return n;
}
template <class L>
__device__ __forceinline__ double* filter_of(double* cold, int mode) { return cold + L::CG_FILT + (mode ? 2 * FILT_CAP : 0); }
template <class L>
__device__ __forceinline__ void augment_filter(const SolveArgs& A, double* cold, int mode, int lane) {
  const double rb = AL(F_RBARR), rt = AL(F_RTH);
  const int n = filter_add(filter_of<L>(cold, mode), (int)AL(F_NFILT), rb - A.o.gamma_phi * rt, (1.0 - A.o.gamma_theta) * rt, lane);
  AL(F_NFILT) = (double)n;
}
template <class L>
__device__ __forceinline__ void acceptor_reset() { AL(F_NFILT) = 0.0; AL(F_LASTREJ) = 0.0; AL(F_SUCC) = 0.0; }
template <class L>
__device__ __forceinline__ bool is_ftype(const SolveArgs& A, double at) {
  const double rt = AL(F_RTH), rg = AL(F_RGBD);
  if (rt == 0.0 && rg > 0.0 && rg < 100.0 * EPSM) return true;
  if (!(rg < 0.0)) return false;
  if (AL(F_PWPHI) < 0.0) {      // every lane computes and stores the same two values (the reference point changes once per line search)
    const double a = n_pow(-rg, A.o.s_phi), b = A.o.delta * n_pow(rt, A.o.s_theta);
    __syncwarp();
    AL(F_PWPHI) = a; AL(F_PWTH) = b;
    __syncwarp();
  }
  return at * AL(F_PWPHI) > AL(F_PWTH);
}
template <class L>
__device__ __forceinline__ bool armijo(const SolveArgs& A, double at, double tb) { const double rb = AL(F_RBARR); return cmp_le(tb - rb, A.o.eta_phi * at * AL(F_RGBD), rb); }
__device__ __forceinline__ bool ok_to_current(const Opt& o, double rb, double rt, double tb, double tt, bool from_resto) {
  if (!from_resto && tb > rb) {
    const double basval = fabs(rb) > 10.0 ? log10(fabs(rb)) : 1.0;
    if (log10(tb - rb) > o.obj_max_inc + basval) return false;
  }
  return cmp_le(tt, (1.0 - o.gamma_theta) * rt, rt) || cmp_le(tb - rb, -o.gamma_phi * rt, rb);
}
// FilterLSAcceptor::CheckAcceptabilityOfTrialPoint
template <class L>
__device__ __noinline__ bool check_accept(const SolveArgs& A, double* cold, int mode, double at, double tb, double tt) {
  const Opt& o = A.o;
  if (!isfinite(tb) || !isfinite(tt)) return false;
  const double rt = AL(F_RTH);
  if (AL(F_THMAX) < 0.0) AL(F_THMAX) = (mode ? o.resto_theta_max_fact : o.theta_max_fact) * fmax(1.0, rt);
  if (AL(F_THMIN) < 0.0) AL(F_THMIN) = o.theta_min_fact * fmax(1.0, rt);
  if (AL(F_THMAX) > 0.0 && tt > AL(F_THMAX)) return false;
  bool acc;
  if (at > 0.0 && is_ftype<L>(A, at) && rt <= AL(F_THMIN)) acc = armijo<L>(A, at, tb);
  else acc = ok_to_current(o, AL(F_RBARR), rt, tb, tt, false);
  if (!acc) { AL(F_LASTREJ) = 0.0; return false; }
  acc = filter_ok(filter_of<L>(cold, mode), (int)AL(F_NFILT), tb, tt);
  if (!acc) AL(F_LASTREJ) = 1.0;
  return acc;
}

// ---- watchdog (BacktrackingLineSearch::StartWatchDog / StopWatchDog) -------------------------------------------------
template <class L>
__device__ __noinline__ void wd_start(const SolveArgs& A, double* cold, int lane) {
  al_count<L>(5, lane);
  AL(F_INWD) = 1.0; AL(F_WTRIAL) = 0.0; AL(F_WAT) = AL(F_APR); AL(F_WDW) = AL(F_DW);
  AL(F_WTH) = AL(F_RTH); AL(F_WBARR) = AL(F_RBARR); AL(F_WGBD) = AL(F_RGBD);
  ph_slot<L>(cold, 0, true, AL(F_MODE) != 0.0, lane);
}
// restore the watchdog's reference iterate and its step; everything that belongs to the current point is recomputed
template <class L>
__device__ __noinline__ void wd_stop(const SolveArgs& A, double* cold, int lane, double df) {
  const int mode = (int)AL(F_MODE);
  const double dw = AL(F_WDW);
  AL(F_INWD) = 0.0; AL(F_WSHORT) = 0.0; AL(F_DW) = dw;
  ph_slot<L>(cold, 0, false, mode != 0, lane);
  do_derivs<L>(A, lane, mode, df, dw, false, cold);
  do_dir<L>(A, lane, mode, false, dw, cold);
  AL(F_APR) = RES(R_APR); AL(F_ADU) = RES(R_ADU); AL(F_GBD) = RES(R_GBD); AL(F_THETA) = RES(R_THETA);
  do_trial<L>(A, lane, mode, 0.0, false, df, cold);
  take_trial_values<L>();
  AL(F_PHI) = trial_barrier<L>(A);
  AL(F_RTH) = AL(F_WTH); AL(F_RBARR) = AL(F_WBARR); AL(F_RGBD) = AL(F_WGBD); AL(F_PWPHI) = -1.0;
  __syncwarp();
}

// ---- BacktrackingLineSearch::TrySoftRestoStep with the current step (DU, DS): 0 rejected, 1 accepted by the primal-dual
//      error test (the iterate has already MOVED to the new point, without kappa_Sigma reset), 2 accepted by the original
//      criterion (not moved).  alpha = min(alpha_primal_max, alpha_dual_max) is returned for both step sizes.
template <class L>
__device__ __noinline__ int soft_step(const SolveArgs& A, double* cold, int lane, double df, int nzt, double& alpha) {
  const Opt& o = A.o;
  constexpr int mtot = L::R * L::S, nx_ = L::NUA * L::N;
  const int mode = (int)AL(F_MODE);
  const double dw = AL(F_DW);
  if (o.soft_resto_red == 0.0) return 0;
  const double al = fmin(AL(F_APR), AL(F_ADU));
  do_trial<L>(A, lane, mode, al, false, df, cold);
  const double th_t = RES(R_THT), phi_t = trial_barrier<L>(A);
  if (!isfinite(th_t) || !isfinite(phi_t)) return 0;
  alpha = al;
  if (check_accept<L>(A, cold, mode, 0.0, phi_t, th_t)) return 2;
  const int nz = mode ? nzt + 2 * mtot : nzt;
  const double nvar = (double)(nx_ + mtot + (mode ? 2 * mtot : 0));
  const double ft = RES(R_FT), lbt = RES(R_LBT), dtt = RES(R_DTT);
  do_derivs<L>(A, lane, mode, df, dw, true, cold);                       // 1-norm sums at the current point, current mu
  const double cur_err = RES(R_DU1) / nvar + RES(R_THETA) / (double)mtot + RES(R_CO1) / (double)max(1, nz);
  ph_slot<L>(cold, mode ? 2 : 1, true, mode != 0, lane);
  do_accept<L>(A, lane, mode, al, al, dw, false, false, cold);
  do_derivs<L>(A, lane, mode, df, dw, true, cold);
  const double tr_err = RES(R_DU1) / nvar + RES(R_THETA) / (double)mtot + RES(R_CO1) / (double)max(1, nz);
  __syncwarp();
  if (lane == 0) { RES(R_FT) = ft; RES(R_LBT) = lbt; RES(R_DTT) = dtt; }
  __syncwarp();
  if (tr_err <= o.soft_resto_red * cur_err) { al_count<L>(6, lane); return 1; }
  ph_slot<L>(cold, mode ? 2 : 1, false, mode != 0, lane);
  do_derivs<L>(A, lane, mode, df, dw, false, cold);
  return 0;
}

// ---- restoration phase --------------------------------------------------------------------------------------------------
// MinC_1NrmRestorationPhase::PerformRestoration: park the original algorithm, start a fresh one on the restoration problem
template <class L>
__device__ __noinline__ void resto_enter(const SolveArgs& A, double* cold, int lane, double df) {
  const Opt& o = A.o;
  al_count<L>(3, lane);
  ph_slot<L>(cold, 1, true, false, lane);
  const double infpr = RES(R_PR);                 // max-norm of g - s at the current point (latest ph_derivs)
  AL(F_INFPR) = infpr;
  __syncwarp();
  for (int f = lane; f < F_NALG; f += 32) cold[L::CG_PARK + f] = AL(f);
  const double mu_r = fmax(AL(F_MU), infpr);
  __syncwarp();
  alg_init<L>(mu_r, o.tau_min, o.tol);
  ph_resto_init<L>(A, lane, mu_r, cold);
  AL(F_MODE) = 1.0;
  ph_trial<L, true>(A, lane, 0.0, false, df, mu_r, cold, false);
  take_trial_values<L>();
  __syncwarp();
}
// RestoFilterConvergenceCheck at the current restoration iterate (E0 etc. of the restoration problem are passed in):
// -1 continue, -2 acceptable to the original problem's filter, >= 0 failure status
template <class L>
__device__ __noinline__ int resto_check(const SolveArgs& A, double* cold, int lane, double df, int iter, double E0, double du_inf, double pr_inf, double pmax) {
  const Opt& o = A.o;
  int st = -1;
  if (iter >= o.max_iter) return NMPC_MAXITER_EXCEEDED;
  const double* park = cold + L::CG_PARK;
  const double oth = RES(R_OTH), oinf = RES(R_OINF);
  double infpr_max = fmax(o.kappa_resto * park[F_INFPR], fmin(o.tol, o.constr_viol_tol));
  if (o.kappa_resto == 0.0) infpr_max = 0.0;
  if (AL(F_FIRST) == 0.0 && !(oinf > infpr_max)) {
    const double omu = park[F_MU];
    ph_trial<L, false>(A, lane, 0.0, false, df, omu, cold, false);       // original objective and barrier terms at the restoration iterate
    const double tb = RES(R_FT) - omu * RES(R_LBT) + o.kappa_d * omu * RES(R_DTT);
    if (filter_ok(filter_of<L>(cold, 0), (int)park[F_NFILT], tb, oth) && ok_to_current(o, park[F_RBARR], park[F_RTH], tb, oth, true)) st = -2;
  }
  if (st == -1) {       // is the restoration problem itself solved?  then the original one is (locally) infeasible
    const double tol = AL(F_TOL);
    if (!isfinite(E0)) st = NMPC_INVALID_NUMBER;
    else if (E0 <= tol && du_inf / df <= o.dual_inf_tol && pr_inf <= o.constr_viol_tol && pmax / df <= o.compl_inf_tol) {
      if (oinf <= 1e2 * tol) {
        if (tol > 1e-1 * o.tol) AL(F_TOL) = 1e-2 * tol;       // tighten once: the problem is only very slightly infeasible
        else st = NMPC_RESTORATION_FAILED;                     // converged to a feasible point the original filter does not accept
      } else st = NMPC_INFEASIBLE_PROBLEM;
    }
  }
  AL(F_FIRST) = 0.0;
  return st;
}
// back to the original problem: x, s from the restoration phase, new bound multipliers, y = 0
template <class L>
__device__ __noinline__ void resto_leave(const SolveArgs& A, double* cold, int lane, double df) {
  const Opt& o = A.o;
  __syncwarp();
  for (int f = lane; f < F_NALG; f += 32) AL(f) = cold[L::CG_PARK + f];
  AL(F_MODE) = 0.0;
  __syncwarp();
  const double mu = AL(F_MU), tau = AL(F_TAU);
  const double adu = ph_resto_finish<L>(A, lane, mu, tau, 0.0, 0, cold, 1);
  const double zmax = ph_resto_finish<L>(A, lane, mu, tau, adu, 1, cold, 1);
  if (zmax > o.bound_mult_reset_threshold) ph_unit_mults<L>(A, lane);
  ph_accept<L, false>(A, lane, 0.0, 0.0, mu, 0.0, false, true, cold);      // kappa_Sigma reset (AcceptTrialPoint)
  ph_trial<L, false>(A, lane, 0.0, false, df, mu, cold, false);
  take_trial_values<L>();
  AL(F_INSOFT) = 0.0; AL(F_SOFTC) = 0.0; AL(F_WSHORT) = 0.0;
  __syncwarp();
}
// restoration inside the restoration phase (RestoRestorationPhase): n, p from their closed form, duals unchanged
template <class L>
__device__ __noinline__ void resto_inner(const SolveArgs& A, double* cold, int lane, double df) {
  ph_resto_np<L>(A, lane, AL(F_MU), cold);
  AL(F_INSOFT) = 0.0; AL(F_SOFTC) = 0.0; AL(F_WSHORT) = 0.0;
  if (lane <= L::N) {
    for (int r = 0; r < L::R; ++r) RW(A_DS, r) = 0.0;
    for (int i = 0; i < 6; ++i) LV(LV_DU + i) = 0.0;
  }
  __syncwarp();
  do_trial<L>(A, lane, 1, 0.0, false, df, cold);
}

// MonotoneMuUpdate (with fast decrease).  The error ingredients of the current point are passed by reference because the
// restoration objective depends on mu (eta = sqrt(mu)): they are refreshed when mu changes in restoration mode.
// Returns false when a tiny step can no longer be answered by a smaller mu (TINY_STEP_DETECTED).
template <class L>
__device__ __noinline__ bool update_mu(const SolveArgs& A, double* cold, int lane, double df, int nz, double mu_floor,
                                       double& du_inf, double& pr_inf, double& pmax, double& pmin, double& sd, double& sc) {
  const Opt& o = A.o;
  constexpr int mtot = L::R * L::S;
  const int mode = (int)AL(F_MODE);
  bool tf = AL(F_TINYFLAG) != 0.0;
  AL(F_TINYFLAG) = 0.0;
  if (mode && AL(F_MUST) == 0.0) { AL(F_MUST) = 1.0; return true; }       // first restoration iteration: mu comes from the initializer
  AL(F_MUST) = 1.0;
  double mu = AL(F_MU);
  auto emu = [&](double m) { return fmax(du_inf / sd, fmax(pr_inf, fmax(pmax - m, m - pmin) / sc)); };
  double Emu = emu(mu);
  bool done = false;
  while ((Emu <= o.kappa_eps * mu || tf) && !done) {
    const double nm = fmax(mu_floor, fmin(o.kappa_mu * mu, n_pow(mu, o.theta_mu)));
    const bool changed = nm != mu;
    if (!changed && tf) return false;
    if (!changed) break;
    mu = nm;
    AL(F_MU) = mu; AL(F_TAU) = fmax(o.tau_min, 1.0 - mu);
    if (mode) {
      __syncwarp();
      do_derivs<L>(A, lane, 1, df, 0.0, false, cold);
      du_inf = RES(R_DU); pr_inf = RES(R_PR); pmax = RES(R_PMAX); pmin = RES(R_PMIN);
      const double sumy = RES(R_SUMY), sumz = RES(R_SUMZ);
      sd = fmax(o.s_max, (sumy + sumz) / (double)max(1, mtot + nz)) / o.s_max;
      sc = fmax(o.s_max, sumz / (double)max(1, nz)) / o.s_max;
      ph_trial<L, true>(A, lane, 0.0, false, df, mu, cold, false);
      take_trial_values<L>();
    }
    if (tf) { done = true; tf = false; }
    else { Emu = emu(mu); done = !(Emu <= o.kappa_eps * mu); }
    AL(F_INSOFT) = 0.0; AL(F_SOFTC) = 0.0; acceptor_reset<L>();        // linesearch->Reset()
  }
  return true;
}

template <class L, bool KEEP = false>
__device__ __noinline__ void solve_instance(const SolveArgs& A, double* ric, double* cold, int b, int lane, int step) {
  const Prob& pr = A.pr; const Opt& o = A.o;
  constexpr int S = L::S, R = L::R;
  constexpr int DX0 = L::LV0 + LV_DX * S, DU0 = L::LV0 + LV_DU * S, DUS0 = L::soc(SOC_DUS), Q20 = L::soc(SOC_Q2);
  constexpr int mtot = R * S;
  const double T = pr.T;
  const bool pair = L::PAIR && A.pair_trials;

  ph_load<L>(A, b, lane, step);
  double df = 1.0;
  if (o.scaling) {
    df = ph_scaling<L>(A, lane);
    if (o.scaling == 3) df = 1.0;                                  // debug: constraint scaling only
    if (o.scaling == 2 && lane <= L::N) { for (int r = 0; r < R; ++r) RW(A_DC, r) = 1.0; }   // debug: objective only
    __syncwarp();
  }
  // multiplier guesses for this instance?  (same address for every lane: uniform)
  const bool warm = A.lam_x0 != nullptr && !isnan(A.lam_x0[(size_t)b * (L::NUA * L::N)]);
  const double mu0 = warm ? o.ws_mu_init : o.mu_init;
  const int nzt = ph_start<L>(A, lane, b, df, warm);
  if (nzt < 0) {       // a finite lower bound on an obstacle row (never the case in the reference's NLPs): refused, reported as data
    ph_output<L, KEEP>(A, b, lane, df, NMPC_INVALID_NUMBER, 0, step);
    return;
  }
  alg_init<L>(mu0, o.tau_min, o.tol);
  for (int f = F_NALG + lane; f < F_END; f += 32) AL(f) = 0.0;
  __syncwarp();
  ph_trial<L, false>(A, lane, 0.0, false, df, mu0, cold, false);      // barrier pieces and constraint violation of the start
  take_trial_values<L>();
  const double mu_floor = fmin(o.tol, df * o.compl_inf_tol) / (o.kappa_eps + 1.0);
  int iter = 0, status = NMPC_MAXITER_EXCEEDED;

  bool retry_owed = false;          // this round of the alignment barriers has not passed the retry point yet
  if (!warm) {   // least-squares multiplier start: (I + J^T J) t = -(grad_x L) - J^T (grad_s L),  y = J t + grad_s L
    align_warps<L>(1); retry_arrive<L>();
    ph_derivs<L, false>(A, lane, true, df, o.mu_init, 0.0, false, cold);
    al_count<L>(0, lane);
    const bool ok = riccati_factor<L>(T, ric, A.ricmap, 1.0, 0.0, lane);
    if (ok) riccati_forward<L>(T, ric, false, lane, DX0, DU0);
    ph_lsy<L>(A, lane, ok);
  }
  for (;;) {
    // Alignment point: the warps of a block start every IPM iteration together, so that they walk through the
    // same ~200 KB of phase code at the same time and share instruction-cache lines (unaligned warps thrash it:
    // `no_instruction` was 56 % of all stall cycles in v3).  Pure scheduling; results cannot depend on it.
    if (retry_owed) retry_arrive<L>();
    align_warps<L>(1); retry_owed = true;
    int mode = (int)AL(F_MODE);
    do_derivs<L>(A, lane, mode, df, 0.0, 0, cold);
    // ---- optimality error (scaled) and termination
    double du_inf = RES(R_DU), pr_inf = RES(R_PR), pmax = RES(R_PMAX), pmin = RES(R_PMIN);
    const int nz = mode ? nzt + 2 * mtot : nzt;
    double sd, sc;
    {
      const double sumy = RES(R_SUMY), sumz = RES(R_SUMZ);
      sd = fmax(o.s_max, (sumy + sumz) / (double)max(1, mtot + nz)) / o.s_max;
      sc = fmax(o.s_max, sumz / (double)max(1, nz)) / o.s_max;
    }
    const double E0 = fmax(du_inf / sd, fmax(pr_inf, pmax / sc));
    if (mode == 0) {
      if (!isfinite(E0) || !isfinite(AL(F_F))) { status = NMPC_INVALID_NUMBER; break; }
      if (E0 <= o.tol && du_inf / df <= o.dual_inf_tol && RES(R_VIOL) <= o.constr_viol_tol && pmax / df <= o.compl_inf_tol) {
        status = NMPC_SOLVE_SUCCEEDED; break;
      }
      if (iter >= o.max_iter) { status = NMPC_MAXITER_EXCEEDED; break; }
    } else {
      const int st = resto_check<L>(A, cold, lane, df, iter, E0, du_inf, pr_inf, pmax);
      if (st == -2) { resto_leave<L>(A, cold, lane, df); continue; }
      if (st >= 0) { status = st; break; }
    }
    // ---- barrier parameter
    const double mu_before = AL(F_MU);
    if (!update_mu<L>(A, cold, lane, df, nz, mu_floor, du_inf, pr_inf, pmax, pmin, sd, sc)) {
      if (mode == 0) status = NMPC_STEP_TOO_SMALL;
      else status = RES(R_OINF) <= 1e2 * o.tol ? NMPC_RESTORATION_FAILED : NMPC_INFEASIBLE_PROBLEM;
      break;
    }
    const double mu = AL(F_MU);
    if (L::FOLD && mode == 0 && mu != mu_before) ph_derivs<L, false>(A, lane, false, df, mu, 0.0, false, cold);   // folded layouts: mu is inside q
    // ---- search direction with inertia correction
    const double ls_before = AL(F_C0 + 1);
    double dw = 0.0; bool ok = false;
    {
      const double dw_last = AL(F_DWLAST);
      for (;;) {
        al_count<L>(0, lane);
        ok = riccati_factor<L>(T, ric, A.ricmap, mu, dw, lane);
        if (ok) break;
        if (dw == 0.0) dw = (dw_last == 0.0) ? o.dw_init : fmax(o.dw_min, dw_last * o.dw_dec);
        else dw = (dw_last == 0.0 || 1e5 * dw_last < dw) ? o.dw_inc_first * dw : o.dw_inc * dw;
        if (dw > o.dw_max) break;
        if (mode) ph_derivs<L, true>(A, lane, false, df, mu, dw, false, cold);       // restoration rows enter with Om(dw)
        else if (L::FOLD) ph_derivs<L, false>(A, lane, false, df, mu, dw, false, cold);   // folded layouts: dw is inside Q / q
      }
    }
    bool goto_resto = !ok;                  // step computation failed: fall back to the restoration phase
    retry_sync<L>(); retry_owed = false;    // re-align after the inertia-correction retries (-5 % .. -21 % per iteration)
    if (ok) {
      if (dw > 0.0) AL(F_DWLAST) = dw;
      riccati_forward<L>(T, ric, false, lane, DX0, DU0);
      do_dir<L>(A, lane, mode, false, dw, cold);
    }
    AL(F_DW) = dw; AL(F_APR) = RES(R_APR); AL(F_ADU) = RES(R_ADU); AL(F_GBD) = RES(R_GBD); AL(F_THETA) = RES(R_THETA);
    AL(F_PHI) = AL(F_F) - mu * AL(F_LB) + o.kappa_d * mu * AL(F_DT);
    // ---- BacktrackingLineSearch::FindAcceptableTrialPoint
    // InitThisLineSearch (+ the filter reset heuristic)
    if (AL(F_INWD) == 0.0) {
      if (o.max_filter_resets > 0 && AL(F_NRES) < (double)o.max_filter_resets) {
        if (AL(F_LASTREJ) != 0.0) {
          if (al_add<L>(F_SUCC, 1.0) >= (double)o.filter_reset_trigger) { acceptor_reset<L>(); al_add<L>(F_NRES, 1.0); al_count<L>(7, lane); }
        } else AL(F_SUCC) = 0.0;
      }
      AL(F_LASTREJ) = 0.0;
      AL(F_RTH) = AL(F_THETA); AL(F_RBARR) = AL(F_PHI); AL(F_RGBD) = AL(F_GBD);
    } else { AL(F_RTH) = AL(F_WTH); AL(F_RBARR) = AL(F_WBARR); AL(F_RGBD) = AL(F_WGBD); }
    AL(F_PWPHI) = -1.0;
    bool tiny = !goto_resto && RES(R_TINY) != 0.0 && AL(F_THETA) <= 1e-4;
    if (AL(F_INWD) != 0.0 && (goto_resto || tiny)) { wd_stop<L>(A, cold, lane, df); dw = AL(F_DW); goto_resto = false; tiny = false; }
    if (o.watchdog_trigger > 0 && AL(F_INWD) == 0.0 && !goto_resto && !tiny && AL(F_INSOFT) == 0.0 && AL(F_WSHORT) >= (double)o.watchdog_trigger)
      wd_start<L>(A, cold, lane);
    double alpha = AL(F_APR), a_du = AL(F_ADU), phi_t = 0.0, th_t = 0.0;
    bool accepted = false, used_soc = false, moved = false;     // moved: the iterate already sits at the new point (soft restoration step)
    int n_steps = 0, tag = '?';
    if (tiny) {
      do_trial<L>(A, lane, mode, alpha, false, df, cold);
      if (!isfinite(RES(R_THT)) || !isfinite(trial_barrier<L>(A))) { status = NMPC_INVALID_NUMBER; break; }
      if (AL(F_TINYLAST) != 0.0) { AL(F_TINYFLAG) = 1.0; tag = 'T'; } else tag = 't';
      AL(F_TINYLAST) = RES(R_DYMAX) < o.tiny_step_y_tol ? 1.0 : 0.0;
      accepted = true;
    } else AL(F_TINYLAST) = 0.0;
    if (!goto_resto && !tiny) {
      if (AL(F_INSOFT) != 0.0) {
        if (al_add<L>(F_SOFTC, 1.0) > (double)o.max_soft_resto) accepted = false;
        else {
          const int r = soft_step<L>(A, cold, lane, df, nzt, alpha);
          accepted = r != 0; moved = r == 1; a_du = alpha;
          if (accepted) { tag = 's'; if (r == 2) { AL(F_INSOFT) = 0.0; AL(F_SOFTC) = 0.0; tag = 'S'; } }
        }
      } else {
        bool skip_first = false;
        for (;;) {       // DoBacktrackingLineSearch (repeated once when the watchdog is stopped)
          bool eval_err = false; accepted = false;
          const bool in_wd = AL(F_INWD) != 0.0;
          const double a_max = AL(F_APR), gbd = AL(F_GBD), theta = AL(F_THETA), ref_theta = AL(F_RTH);
          double amin = a_max;
          if (!in_wd) {
            amin = o.gamma_theta;
            if (gbd < 0.0) {
              amin = fmin(o.gamma_theta, o.gamma_phi * theta / (-gbd));
              if (theta <= AL(F_THMIN)) amin = fmin(amin, o.delta * n_pow(theta, o.s_theta) / n_pow(-gbd, o.s_phi));
            }
            amin *= o.alpha_min_frac;
          }
          alpha = a_max; a_du = AL(F_ADU);
          double a_test = in_wd ? AL(F_WAT) : alpha;
          if (skip_first) alpha *= o.alpha_red;
          // alpha of the trial point the last paired pass evaluated ahead (< 0: none).  Between two trials of this loop
          // nothing moves the iterate, the direction, mu or the mode (a second-order correction has arrays of its own),
          // so that result is the one a pass at this alpha would give.
          double ahead = -1.0;
          while (alpha > amin || n_steps == 0) {
            if (pair && alpha == ahead) { take_ahead<L>(lane); ahead = -1.0; }
            else { do_trial<L>(A, lane, mode, alpha, false, df, cold, pair); if (pair) ahead = alpha * o.alpha_red; }
            th_t = RES(R_THT); phi_t = trial_barrier<L>(A);
            const bool okv = isfinite(th_t) && isfinite(phi_t);
            if (!in_wd) a_test = alpha;
            if (okv) accepted = check_accept<L>(A, cold, mode, a_test, phi_t, th_t); else { accepted = false; eval_err = true; }
            if (accepted || in_wd) break;
            if (okv && alpha == a_max && ref_theta <= th_t && o.max_soc > 0) {
              // second-order correction (FilterLSAcceptor::TrySecondOrderCorrection)
              int count = 0; double theta_old = 0.0, theta_trial = th_t, a_soc = alpha; bool first = true;
              while (count < o.max_soc && !accepted && (count == 0 || theta_trial <= o.kappa_soc * theta_old)) {
                theta_old = theta_trial;
                if (mode) ph_socrhs<L, true>(A, lane, a_soc, mu, dw, first, cold); else ph_socrhs<L, false>(A, lane, a_soc, mu, dw, first, cold);
                first = false;
                riccati_resolve<L>(T, Q20, ric, mu, lane);
                riccati_forward<L>(T, ric, true, lane, DX0, DUS0);
                do_dir<L>(A, lane, mode, true, dw, cold);
                a_soc = RES(R_APR);
                do_trial<L>(A, lane, mode, a_soc, true, df, cold);
                th_t = RES(R_THT); phi_t = trial_barrier<L>(A);
                if (!isfinite(th_t) || !isfinite(phi_t)) break;
                accepted = check_accept<L>(A, cold, mode, a_test, phi_t, th_t);
                if (accepted) { alpha = a_soc; a_du = RES(R_ADU); used_soc = true; al_count<L>(2, lane); }
                else { ++count; theta_trial = th_t; }
              }
              if (accepted) break;
            }
            alpha *= o.alpha_red; ++n_steps;
          }
          if (accepted) {      // UpdateForNextIteration
            if (!is_ftype<L>(A, a_test) || !armijo<L>(A, a_test, phi_t)) { augment_filter<L>(A, cold, mode, lane); tag = used_soc ? 'H' : 'h'; }
            else tag = used_soc ? 'F' : 'f';
          } else if (in_wd) tag = 'w';
          if (in_wd) {
            if (accepted) { AL(F_INWD) = 0.0; break; }
            if (eval_err || al_add<L>(F_WTRIAL, 1.0) > (double)o.watchdog_trial_max) { wd_stop<L>(A, cold, lane, df); dw = AL(F_DW); skip_first = true; continue; }
            accepted = true; break;        // take the step without acceptance test
          }
          break;
        }
      }
    }
    bool entered_resto = false;
    if (!accepted) {
      if (AL(F_INSOFT) == 0.0 && !goto_resto) {      // try the current direction as a soft restoration step
        augment_filter<L>(A, cold, mode, lane);       // PrepareRestoPhaseStart
        const int r = soft_step<L>(A, cold, lane, df, nzt, alpha);
        accepted = r != 0; moved = r == 1; a_du = alpha; used_soc = false;
        if (accepted) { if (r == 2) tag = 'S'; else { AL(F_INSOFT) = 1.0; tag = 's'; } }
      }
      if (!accepted) {
        if (AL(F_INSOFT) == 0.0) augment_filter<L>(A, cold, mode, lane);
        if (AL(F_THETA) <= 1e-2 * o.tol) { status = NMPC_RESTORATION_FAILED; break; }    // "... called, but point is almost feasible"
        tag = 'R';
        if (mode) { resto_inner<L>(A, cold, lane, df); alpha = 0.0; a_du = 0.0; moved = false; used_soc = false; accepted = true; }
        else entered_resto = true;
      }
    } else if (AL(F_INSOFT) == 0.0 || tiny) {
      if (n_steps == 0) AL(F_WSHORT) = 0.0; else al_add<L>(F_WSHORT, 1.0);
    }
    if (A.dbg && lane == 0 && iter < A.dbg_rows) {
      double* Lg = A.dbg + ((size_t)b * A.dbg_rows + iter) * DBG_COLS;
      Lg[0] = mu; Lg[1] = mode ? AL(F_F) : AL(F_F) / df; Lg[2] = pr_inf; Lg[3] = du_inf; Lg[4] = dw; Lg[5] = alpha; Lg[6] = a_du;
      Lg[7] = AL(F_C0 + 1) - ls_before; Lg[8] = (double)tag; Lg[9] = (double)mode;
    }
    if (entered_resto) { resto_enter<L>(A, cold, lane, df); ++iter; continue; }
    // ---- accept (IpoptAlgorithm::AcceptTrialPoint)
    if (moved) do_accept<L>(A, lane, mode, 0.0, 0.0, dw, false, true, cold);     // the soft step already moved the iterate: kappa_Sigma reset only
    else do_accept<L>(A, lane, mode, alpha, a_du, dw, used_soc, true, cold);
    take_trial_values<L>();
    if (mode) al_count<L>(4, lane);
    ++iter;
  }
  if (retry_owed) retry_arrive<L>();
  ph_output<L, KEEP>(A, b, lane, df, status, iter, step);
  if (lane == 0 && A.stats) {
#pragma unroll
    for (int c = 0; c < NSTAT; ++c) atomicAdd(&A.stats[c], (unsigned long long)AL(F_C0 + c));
  }
}

// Longest-first fetch order for the NEXT call on this handle from this call's iteration counts: counting sort,
// descending, by the warp that finished the call's last instance (its shared-memory slice is free; the order inside a
// bin is arbitrary -- results do not depend on it).
template <class L>
__device__ __noinline__ void next_order(const SolveArgs& A, int lane) {
  int* bin = reinterpret_cast<int*>(&smem[0]);          // 256 ints
  for (int i = lane; i < 256; i += 32) bin[i] = 0;
  __syncwarp();
  for (int i = lane; i < A.B; i += 32) atomicAdd(&bin[min(max(__ldcg(A.iters_keep + i), 0), 255)], 1);
  __syncwarp();
  if (lane == 0) {
    int acc = 0;
    for (int v = 255; v >= 0; --v) { const int c = bin[v]; bin[v] = acc; acc += c; }
  }
  __syncwarp();
  for (int i = lane; i < A.B; i += 32) A.order_out[atomicAdd(&bin[min(max(__ldcg(A.iters_keep + i), 0), 255)], 1)] = i;
  __syncwarp();
}

// persistent kernel: Lay::WPB warps per block (one block per SM), one instance per warp at a time, instances from
// an atomic work queue (optionally in a caller-given order).  KEEP: the instantiation that also writes the barrier data
// (NMPC_KEEP_BARRIER).  It is a kernel of its own because ptxas compiles a kernel with all its device functions as one unit:
// any code added to ph_output of the production kernel changes the machine code of the per-iteration phases too.
template <int N_, int NOBS_, int MODEL_, bool KEEP = false>
__global__ void __launch_bounds__(32 * Lay<N_, NOBS_, MODEL_>::WPB, 1) nmpc_ipm_kernel(const __grid_constant__ SolveArgs A) {
  using L = Lay<N_, NOBS_, MODEL_>;
  const int lane = threadIdx.x & 31;
  if (blockIdx.x == 0 && threadIdx.x == 0) {      // the next call on this handle starts from clean counters
    *A.counter_next = 0; *A.done_next = 0;
    for (int i = 0; i < NSTAT; ++i) A.stats_next[i] = 0;
  }
  const size_t slot = (size_t)(blockIdx.x * L::WPB + (threadIdx.x >> 5));
  double* ric = A.ric + slot * A.ric_stride;
  double* cold = A.cold + slot * A.cold_stride;
  for (;;) {
    int q = 0;
    if (lane == 0) q = atomicAdd(A.counter, 1);
    q = __shfl_sync(FULL, q, 0);
    if (q >= A.B) break;
    const int b = A.order ? A.order[q] : q;
    // free-running closed loop: the steps of one instance follow each other here (the epilogue of step k has written p and the
    // warm start of step k + 1 in place), with no batch-wide barrier between the steps
    for (int step = 0; step < A.run_steps; ++step) { solve_instance<L, KEEP>(A, ric, cold, b, lane, step); __syncwarp(); }
    __syncwarp();
    int fin = 0;
    if (lane == 0) { __threadfence(); fin = atomicAdd(A.done, 1); }      // this instance's outputs are visible before the count
    fin = __shfl_sync(FULL, fin, 0);
    if (fin == A.B - 1 && A.order_out) next_order<L>(A, lane);           // last instance of the call
  }
  while (align_warps<L>(0)) retry_arrive<L>();   // out of work: keep matching the alignment barriers until the block is done
}

#undef LV
#undef RW
#undef LQ
#undef SOC
#undef RES
#undef PAR
#undef RG
#undef UREF
#undef AL
#undef smem

}  // namespace nmpc
