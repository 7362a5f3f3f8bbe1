// nmpc_b200.cu -- kernels + C ABI (include/nmpc_b200.h) of the B200-native batched NMPC solver.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
//
// Kernels
//   nmpc_ipm_kernel   persistent, one warp per NLP instance, whole IPM loop in-kernel (nmpc_solve.cuh / nmpc_inst.cu);
//                     optionally the closed-loop shift in its epilogue (nmpc_solve_and_step)
//   nmpc_eval_kernel  function-level f / g / grad f / J^T lam / Hess_L v  (one warp per instance)
//   nmpc_step_kernel  closed-loop shift (NMPC_TT.py:13-30) + FOV centre (:399-402), one thread per instance
#include <cuda_runtime.h>
#include <cstdlib>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <new>
#include <string>

#include "../../include/nmpc_b200.h"
#include "nmpc_solve.cuh"

using namespace nmpc;

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
// The IPM kernel (nmpc_solve.cuh) is a template on (N, n_obs); its instantiations live in nmpc_inst.cu objects.
namespace nmpc {
#define NMPC_DECL_INST(N, O, M)                      \
  int ipm_prepare_##N##_##O##_##M(int*, size_t*, int*, int*);  \
  int ipm_ricmap_##N##_##O##_##M(unsigned*, cudaStream_t);     \
  int ipm_launch_##N##_##O##_##M(const SolveArgs&, int, size_t, cudaStream_t);  \
  int ipm_sens_##N##_##O##_##M(const SolveArgs&, int, cudaStream_t);
NMPC_DECL_INST(15, 3, 0) NMPC_DECL_INST(15, 10, 0) NMPC_DECL_INST(30, 10, 0) NMPC_DECL_INST(30, 3, 0) NMPC_DECL_INST(5, 3, 0) NMPC_DECL_INST(15, 7, 0)
NMPC_DECL_INST(15, 0, 1)
}  // namespace nmpc
struct IpmInst {
  int N, n_obs, model;
  int (*prepare)(int*, size_t*, int*, int*); int (*ricmap)(unsigned*, cudaStream_t); int (*launch)(const SolveArgs&, int, size_t, cudaStream_t);
  int (*sens)(const SolveArgs&, int, cudaStream_t);      // nmpc_sensitivity (nmpc_sens.cuh)
};
#define NMPC_INST(N, O, M) {N, O, M, nmpc::ipm_prepare_##N##_##O##_##M, nmpc::ipm_ricmap_##N##_##O##_##M, nmpc::ipm_launch_##N##_##O##_##M, nmpc::ipm_sens_##N##_##O##_##M}
static const IpmInst IPM_INSTS[] = {NMPC_INST(15, 3, 0), NMPC_INST(15, 10, 0), NMPC_INST(30, 10, 0), NMPC_INST(30, 3, 0), NMPC_INST(5, 3, 0),
                                    NMPC_INST(15, 7, 0),      // the 7 obstacle rows of MATLAB/Dynamic Obstacles/Dynamic Obstacle avoidance.m:126-134
                                    NMPC_INST(15, 0, 1)};     // the gimbal-less tracker of MATLAB/Dynamic Obstacles/NMPC_TT.m

struct EvalArgs {
  Prob pr; int B;
  const double *w, *p, *obs; int obs_per_instance;
  const double *weights, *tgt;
  double sigma; const double *lam, *v;
  double *f, *g, *grad, *jtv, *hv;
  double* lamp;      // nmpc_lam_p: -(d/dp)(sigma f + lam^T g), [B][n_p]
};

__global__ void __launch_bounds__(128) nmpc_eval_kernel(const EvalArgs A) {
  const Prob& pr = A.pr;
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= A.B) return;
  const int nu = model_nu(pr.model), nb = model_nb(pr.model), npar = model_np(pr.model);      // model 1: see nmpc_device.cuh
  const int N = pr.N, R = pr.R, S = pr.S, n_obs = pr.n_obs, nw = nu * N, ng = R * S;
  const bool act = lane <= N, hasu = lane < N;
  const double T = pr.T;
  const double* pp = A.p + (size_t)b * npar;
  double X0[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) X0[i] = i < (pr.model ? 5 : 8) ? pp[i] : 0.0;
  const double xt = (A.tgt && hasu) ? A.tgt[((size_t)b * N + lane) * 2] : pp[npar - 3];
  const double yt = (A.tgt && hasu) ? A.tgt[((size_t)b * N + lane) * 2 + 1] : pp[npar - 2];
  double u[6], vv[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    u[i] = (hasu && i < nu) ? A.w[(size_t)b * nw + nu * lane + i] : 0.0; vv[i] = (hasu && A.v && i < nu) ? A.v[(size_t)b * nw + nu * lane + i] : 0.0;
  }
  const double* obs = A.obs + (A.obs_per_instance ? (size_t)b * 3 * n_obs : 0);
  Stage st;
  rollout(pr, X0, u, lane, st);
  const Dyn dyn = dyn_entries(st, hasu ? T * u[0] : 0.0);
  const double e03 = dyn.e03, e13 = dyn.e13, e23 = dyn.e23, e04 = dyn.e04, e14 = dyn.e14;
  auto adjoint = [&](const double* a, double* lamn) { nmpc::adjoint(a, dyn, act, lane, lamn); };
  auto Bt = [&](const double* lamn, double* out) {
    out[0] = T * (st.cps * st.cth * lamn[0] + st.sps * st.cth * lamn[1] + st.sth * lamn[2]);
#pragma unroll
    for (int r = 1; r < 6; ++r) out[r] = T * lamn[r + 2];
  };
  double gl[6], Hl[21];
#pragma unroll
  for (int i = 0; i < 6; ++i) gl[i] = 0.0;
#pragma unroll
  for (int i = 0; i < 21; ++i) Hl[i] = 0.0;
  double l = 0.0;
  if (hasu) l = pr.model ? stage_cost_dist_d2(st.X, xt, yt, gl, Hl)
                         : stage_cost_d2(A.weights ? with_weights(pr, A.weights[2 * (size_t)b], A.weights[2 * (size_t)b + 1]) : pr, st.X, xt, yt, gl, Hl);
  const double fsum = warp_sum(l);
  if (lane == 0 && A.f) A.f[b] = fsum;
  if (act && A.g) {
    double* go = A.g + (size_t)b * ng + lane * R;
    for (int r = 0; r < nb; ++r) go[r] = st.X[box_state(r)];
    for (int jn = 0; jn < n_obs; ++jn) {
      const double dx_ = st.X[0] - obs[3 * jn], dy_ = st.X[1] - obs[3 * jn + 1];
      go[nb + jn] = obs[3 * jn + 2] - sqrt(dx_ * dx_ + dy_ * dy_);
    }
  }
  double a[8], lamn[8], out[6];
  if (A.grad) {
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = 0.0;
#pragma unroll
    for (int v = 0; v < 6; ++v) a[cost_state(v)] = gl[v];
    adjoint(a, lamn); Bt(lamn, out);
    if (hasu) for (int i = 0; i < nu; ++i) A.grad[(size_t)b * nw + nu * lane + i] = out[i];
  }
  const double* lm = A.lam ? A.lam + (size_t)b * ng + lane * R : nullptr;
  auto gt_lam = [&](double* acc) {   // acc += G_k^T lam_k
    if (act && lm) {
      for (int r = 0; r < nb; ++r) acc[box_state(r)] += lm[r];
      for (int jn = 0; jn < n_obs; ++jn) {
        const double dx_ = st.X[0] - obs[3 * jn], dy_ = st.X[1] - obs[3 * jn + 1];
        const double iD = 1.0 / sqrt(dx_ * dx_ + dy_ * dy_);
        acc[0] += -lm[nb + jn] * dx_ * iD; acc[1] += -lm[nb + jn] * dy_ * iD;
      }
    }
  };
  if (A.jtv) {
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = 0.0;
    gt_lam(a);
    adjoint(a, lamn); Bt(lamn, out);
    if (hasu) for (int i = 0; i < nu; ++i) A.jtv[(size_t)b * nw + nu * lane + i] = out[i];
  }
  if (A.lamp) {
    // lam_p of CasADi's result dict (NMPC_TT.py:358-365 returns it, nobody reads it): minus the gradient of the Lagrangian with
    // respect to p = [X_0; x_t; y_t; theta_t].  d/dX_0 is the adjoint at stage 0 (the stage-0 cost and rows count here, unlike in
    // the gradient with respect to w); the stage costs depend on the target only through (x - x_t, y - y_t), so d/d(x_t, y_t) =
    // -sum_k dl_k/d(x, y); theta_t does not enter.  With a per-stage target prediction the target entries of p are unused: 0.
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = 0.0;
#pragma unroll
    for (int v = 0; v < 6; ++v) a[cost_state(v)] = A.sigma * gl[v];
    gt_lam(a);
    adjoint(a, lamn);
    const double sx = warp_sum(hasu ? A.sigma * gl[0] : 0.0), sy = warp_sum(hasu ? A.sigma * gl[1] : 0.0);
    if (lane == 0) {
      double l0[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) l0[i] = a[i] + lamn[i];
      l0[3] += e03 * lamn[0] + e13 * lamn[1] + e23 * lamn[2];
      l0[4] += e04 * lamn[0] + e14 * lamn[1];
      double* lp = A.lamp + (size_t)b * npar;
      const int ns = pr.model ? 5 : 8;
      for (int i = 0; i < ns; ++i) lp[i] = -l0[i];
      lp[ns] = A.tgt ? 0.0 : sx; lp[ns + 1] = A.tgt ? 0.0 : sy; lp[ns + 2] = 0.0;
    }
  }
  if (A.hv) {
    // adjoint of the Lagrangian sigma f + lam^T g
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = 0.0;
#pragma unroll
    for (int v = 0; v < 6; ++v) a[cost_state(v)] = A.sigma * gl[v];
    gt_lam(a);
    adjoint(a, lamn);
    // linearised rollout of the direction v
    double dx[8];
    {
      double a5[5];
#pragma unroll
      for (int c = 0; c < 5; ++c) a5[c] = hasu ? T * vv[c + 1] : 0.0;
      scan_excl<5>(a5, lane);
#pragma unroll
      for (int c = 0; c < 5; ++c) dx[3 + c] = a5[c];
      const double tvv = hasu ? T * vv[0] : 0.0;
      double a3[3] = {e03 * dx[3] + e04 * dx[4] + tvv * st.cps * st.cth, e13 * dx[3] + e14 * dx[4] + tvv * st.sps * st.cth,
                      e23 * dx[3] + tvv * st.sth};
      scan_excl<3>(a3, lane);
      dx[0] = a3[0]; dx[1] = a3[1]; dx[2] = a3[2];
    }
    // w_x = Q dx + S^T v_u,  w_u = S dx
    double wx[8], wu0 = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) wx[i] = 0.0;
    if (act) {
      if (hasu && lane >= 1) {
#pragma unroll
        for (int uu = 0; uu < 6; ++uu)
#pragma unroll
          for (int v = 0; v < 6; ++v) wx[cost_state(uu)] += A.sigma * Hl[tri(uu, v)] * dx[cost_state(v)];
      }
      if (lm) for (int jn = 0; jn < n_obs; ++jn) {
        const double dx_ = st.X[0] - obs[3 * jn], dy_ = st.X[1] - obs[3 * jn + 1];
        const double D = sqrt(dx_ * dx_ + dy_ * dy_), iD = 1.0 / D, nx = dx_ * iD, ny = dy_ * iD;
        const double cur = -lm[nb + jn] * iD;
        wx[0] += cur * ((1.0 - nx * nx) * dx[0] - nx * ny * dx[1]);
        wx[1] += cur * (-nx * ny * dx[0] + (1.0 - ny * ny) * dx[1]);
      }
      if (hasu) {
        const double L0 = T * lamn[0], L1 = T * lamn[1], L2 = T * lamn[2], v = u[0];
        const double cc = st.cps * st.cth, sc = st.sps * st.cth, cs = st.cps * st.sth, ss = st.sps * st.sth;
        const double q33 = -v * (L0 * cc + L1 * sc + L2 * st.sth), q44 = -v * (L0 * cc + L1 * sc), q34 = v * (L0 * ss - L1 * cs);
        const double svt = -L0 * cs - L1 * ss + L2 * st.cth, svp = -L0 * sc + L1 * cc;
        wx[3] += q33 * dx[3] + q34 * dx[4] + svt * vv[0];
        wx[4] += q34 * dx[3] + q44 * dx[4] + svp * vv[0];
        wu0 = svt * dx[3] + svp * dx[4];
      }
    }
    adjoint(wx, lamn); Bt(lamn, out);
    out[0] += wu0;
    if (hasu) for (int i = 0; i < nu; ++i) A.hv[(size_t)b * nw + nu * lane + i] = out[i];
  }
}

struct StepArgs {
  double T, hv, hh; int N, B, model;
  const double* x_sol; double *p, *u_warm; const double* vw; double *fov, *err;
};

__global__ void nmpc_step_kernel(const StepArgs A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  const int nu = model_nu(A.model), nw = nu * A.N;
  const double* xs = A.x_sol + (size_t)b * nw;
  double u0[NU] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int i = 0; i < nu; ++i) u0[i] = xs[i];
  // warm start: drop the first stage, repeat the last (NMPC_TT.py:20-23).  x_sol may alias u_warm.
  double* uw = A.u_warm + (size_t)b * nw;
  for (int k = 0; k < A.N - 1; ++k)
    for (int i = 0; i < nu; ++i) uw[nu * k + i] = xs[nu * (k + 1) + i];
  if (A.u_warm != A.x_sol)
    for (int i = 0; i < nu; ++i) uw[nu * (A.N - 1) + i] = xs[nu * (A.N - 1) + i];
  closed_loop_shift_model(A.model, A.T, A.hv, A.hh, A.p + (size_t)b * model_np(A.model), u0, A.vw[2 * b], A.vw[2 * b + 1],
                    A.fov ? A.fov + 2 * (size_t)b : nullptr, A.err ? A.err + b : nullptr);
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(const std::string& m) { g_err = m; return 1; }
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(e_));        \
  } while (0)

// like CK, but releases the half-built handle first (nmpc_create)
#define CKH(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) { nmpc_destroy(h); return fail(std::string(#call) + ": " + cudaGetErrorString(e_)); } \
  } while (0)

struct nmpc_handle {
  nmpc_spec spec; int device; int sm_count;
  Prob pr; Opt opt;
  const IpmInst* inst; size_t smem_bytes; int blocks_per_sm, max_blocks, warps_per_block;
  double* d_ric; int ric_stride; unsigned* d_ricmap; double* d_cold; int cold_stride;
  // per-call bookkeeping, double-buffered by call parity: the launch of call n resets / produces the buffers of call n+1
  int32_t *d_order[2], *d_keep_iters; int order_cap, prev_B, auto_order, parity, have_order; const int32_t* order_next;
  const double *weights, *tgt;
  double *ws_lamx, *ws_lamg;       // nmpc_set_warm_start
  const double* sched_table; const int32_t *sched_id, *sched_phase; int sched_rows, sched_len, sched_iter;   // nmpc_set_schedule
  double* d_tgt_pred; int tgt_pred_cap;        // NMPC_PREDICT_TARGET: the trajectory the kernel predicts, [tgt_pred_cap][N][2]
  double* move_obs; const double* move_vel;    // nmpc_set_obstacle_motion
  double *d_sigx, *d_sigg; int sig_cap;        // NMPC_KEEP_BARRIER: Sigma_x [sig_cap][n_w], Sigma_g [sig_cap][n_g] of the last solve
  int kept_B;                                  // B of the last solve when it kept them, else 0 (what nmpc_sensitivity needs)
  // nmpc_sensitivity reads the kept Sigmas and uses the Riccati scratch, possibly on another stream than the solves (the host
  // calls run on own_stream): ev_keep marks the end of the keeping solve, ev_sens the end of the last sensitivity launch
  cudaEvent_t ev_keep, ev_sens; cudaStream_t keep_stream, sens_stream; int sens_pending;
  int* d_counter;                  // [4]: queue counter x2, done counter x2
  unsigned long long* d_stats;     // [2][NSTAT]
  unsigned long long* stats_last;  // the half written by the last call
  // staging for nmpc_solve_host
  double *d_p, *d_x0, *d_lbx, *d_ubx, *d_lbg, *d_ubg, *d_obs, *d_x, *d_f, *d_g, *d_lamx, *d_lamg;
  int32_t *d_status, *d_iters; size_t obs_cap;
  cudaStream_t own_stream, last_stream;
  int64_t launches;
  double* dbg; int dbg_rows;
  int fill, pair_trials;
};

// The refusals several entry points share, each naming `fn`, the public function the caller called.  Those in `which` are
// checked in this order; an entry point that makes them at different places of its own order calls this once per place.
enum : unsigned { NULL_HANDLE = 1u, NO_OBSTACLES = 2u, PREDICT_WITHOUT_VW = 4u, PREDICT_WITH_TRAJECTORY = 8u, KEEP_WITHOUT_OUTPUTS = 16u,
                  NOT_KEPT = 32u, KEPT_OTHER_B = 64u, WEIGHTS_OF_MODEL_1 = 128u, NO_OBSTACLE_ROWS = 256u };
static int refused(const nmpc_handle* h, const char* fn, unsigned which, const double* obst = nullptr, uint32_t flags = 0, int32_t B = 0,
                   const double* dx_dw = nullptr) {
  if ((which & NULL_HANDLE) && !h) return fail(std::string(fn) + ": null handle");
  if ((which & NO_OBSTACLE_ROWS) && h->pr.n_obs == 0) return fail(std::string(fn) + ": this problem has no obstacle rows (n_obs = 0)");
  if ((which & NO_OBSTACLES) && h->pr.n_obs > 0 && !obst) return fail(std::string(fn) + ": obstacle table required");
  if ((which & PREDICT_WITHOUT_VW) && (flags & NMPC_PREDICT_TARGET))
    return fail(std::string(fn) + ": NMPC_PREDICT_TARGET needs the target's (v, omega) of the step: use nmpc_solve_and_step or nmpc_run_closed_loop");
  if ((which & PREDICT_WITH_TRAJECTORY) && (flags & NMPC_PREDICT_TARGET) && h->tgt)
    return fail(std::string(fn) + ": NMPC_PREDICT_TARGET and a target trajectory (nmpc_set_target_trajectory) exclude each other");
  if ((which & KEEP_WITHOUT_OUTPUTS) && (flags & NMPC_KEEP_BARRIER))
    return fail(std::string(fn) + ": NMPC_KEEP_BARRIER is for nmpc_solve, nmpc_solve_host and nmpc_solve_host_async (the fused and "
                                  "free-running calls return no multipliers to differentiate with)");
  if ((which & NOT_KEPT) && !h->kept_B)
    return fail(std::string(fn) + ": the last solve on this handle did not keep its barrier data (pass NMPC_KEEP_BARRIER to it)");
  if ((which & KEPT_OTHER_B) && B != h->kept_B)
    return fail(std::string(fn) + ": B = " + std::to_string(B) + " differs from the B = " + std::to_string(h->kept_B) + " of the last solve");
  if ((which & WEIGHTS_OF_MODEL_1) && dx_dw && h->pr.model)
    return fail(std::string(fn) + ": dx_dw is for model 0 only (the gimbal-less model has no cost weights)");
  return 0;
}

// What every solve entry point passes on from its caller, in the order of SolveArgs; the rest starts null / zero.
static SolveArgs solve_args(int32_t B, const double* p, const double* x0, const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                            const double* obst, uint32_t flags, double* x, double* f, double* g, double* lam_x, double* lam_g, int32_t* status, int32_t* iters) {
  return SolveArgs{{}, {}, B, p, x0, lbx, ubx, lbg, ubg, obst, (flags & NMPC_OBS_PER_INSTANCE) ? 1 : 0, x, f, g, lam_x, lam_g, status, iters};
}

// One launch of the IPM kernel for the entry point `fn`, after nmpc_solve's checks and, when `fused`, those of the fused calls
// before them.  A holds what the caller passed (step_* for the fused calls, run_* for the free-running one); the rest is handle state.
static int launch_solve(nmpc_handle* h, SolveArgs& A, uint32_t flags, cudaStream_t s, const char* fn, bool fused = false) {
  const std::string f(fn);
  if (refused(h, fn, NULL_HANDLE)) return 1;
  h->kept_B = 0;                        // whatever this call does, the barrier data of an earlier solve no longer belongs to the last solve
  if (fused) {
    if (refused(h, fn, KEEP_WITHOUT_OUTPUTS, nullptr, flags)) return 1;
    if (!A.step_p || !A.step_u) return fail(f + ": null required pointer");
    if (!A.step_vw && !h->sched_table) return fail(f + ": target_vw is NULL and no schedule is set (nmpc_set_schedule)");
    if (A.step_err && !A.step_fov) return fail(f + ": err_accum needs fov_centre");
    if (A.x == A.step_u) return fail(f + ": x must not alias u_warm (pass NULL if the solution itself is not needed)");
    if (h->move_obs && A.obs != h->move_obs) return fail(f + ": obstacle motion is set (nmpc_set_obstacle_motion): obst must be the registered field");
    if (h->move_obs && A.B > 1 && !(flags & NMPC_OBS_PER_INSTANCE)) return fail(f + ": obstacle motion needs a per-instance obstacle field (NMPC_OBS_PER_INSTANCE)");
  }
  A.run_steps = A.run_steps > 1 ? A.run_steps : 1;
  const int sched_steps = fused && !A.step_vw ? A.run_steps : 0;      // the schedule's step counter (mpc_iter) advances, B <= 0 included
  const int B = A.B;
  if (B <= 0) { h->sched_iter += sched_steps; return 0; }
  if (!A.p || !A.x0 || !A.lbx || !A.ubx || !A.lbg || !A.ubg || (!A.x && !fused)) return fail(f + ": null required pointer");
  if (refused(h, fn, NO_OBSTACLES | (fused ? PREDICT_WITH_TRAJECTORY : PREDICT_WITHOUT_VW), A.obs, flags)) return 1;
  CK(cudaSetDevice(h->device));
  const bool predict = (flags & NMPC_PREDICT_TARGET) != 0;
  A.pr = h->pr; A.o = h->opt;
  const int par = h->parity;            // flipped only after a successful launch (see below)
  A.counter = h->d_counter + par; A.counter_next = h->d_counter + (par ^ 1);
  A.done = h->d_counter + 2 + par; A.done_next = h->d_counter + 2 + (par ^ 1);
  A.stats = h->d_stats + NSTAT * par; A.stats_next = h->d_stats + NSTAT * (par ^ 1);
  A.ric = h->d_ric; A.ric_stride = h->ric_stride; A.ricmap = h->d_ricmap;
  A.cold = h->d_cold; A.cold_stride = h->cold_stride;
  A.dbg = h->dbg; A.dbg_rows = h->dbg_rows;
  if (h->sens_pending && h->sens_stream != s) CK(cudaStreamWaitEvent(s, h->ev_sens, 0));     // the Riccati scratch is shared
  h->sens_pending = 0;
  if (B > h->order_cap) {     // (re)allocate the scheduling buffers; the previous counts are dropped
    CK(cudaStreamSynchronize(s));
    for (int i = 0; i < 2; ++i) { if (h->d_order[i]) cudaFree(h->d_order[i]); h->d_order[i] = nullptr; }
    if (h->d_keep_iters) cudaFree(h->d_keep_iters);
    h->d_keep_iters = nullptr; h->order_cap = 0; h->prev_B = 0; h->have_order = 0;
    // (a failure here returns before anything of this call was enqueued: parity and counters are untouched, the
    //  partially allocated buffers are freed by the next attempt or by nmpc_destroy)
    CK(cudaMalloc(&h->d_order[0], sizeof(int32_t) * B)); CK(cudaMalloc(&h->d_order[1], sizeof(int32_t) * B));
    CK(cudaMalloc(&h->d_keep_iters, sizeof(int32_t) * B));
    h->order_cap = B;
  }
  const bool keep = (flags & NMPC_KEEP_BARRIER) != 0;
  if (keep && B > h->sig_cap) {     // the kept barrier data, grown like the scheduling buffers
    CK(cudaStreamSynchronize(s));
    if (h->d_sigx) cudaFree(h->d_sigx);
    if (h->d_sigg) cudaFree(h->d_sigg);
    h->d_sigx = h->d_sigg = nullptr; h->sig_cap = 0;
    CK(cudaMalloc(&h->d_sigx, sizeof(double) * (size_t)model_nu(h->pr.model) * h->pr.N * B));
    CK(cudaMalloc(&h->d_sigg, sizeof(double) * (size_t)h->pr.R * h->pr.S * B));
    h->sig_cap = B;
  }
  if (predict && B > h->tgt_pred_cap) {     // the predicted trajectories, grown like the scheduling buffers
    CK(cudaStreamSynchronize(s));
    if (h->d_tgt_pred) cudaFree(h->d_tgt_pred);
    h->d_tgt_pred = nullptr; h->tgt_pred_cap = 0;
    CK(cudaMalloc(&h->d_tgt_pred, sizeof(double) * 2 * (size_t)h->pr.N * B));
    h->tgt_pred_cap = B;
  }
  A.iters_keep = h->d_keep_iters;
  A.sched_table = h->sched_table; A.sched_id = h->sched_id; A.sched_phase = h->sched_phase; A.sched_len = h->sched_len; A.sched_iter = h->sched_iter;
  A.tgt_pred = predict ? h->d_tgt_pred : nullptr;
  A.tgt = predict ? h->d_tgt_pred : h->tgt;
  A.obs_move = A.step_p ? h->move_obs : nullptr; A.obs_vel = h->move_vel;
  A.lam_x0 = h->ws_lamx; A.lam_g0 = h->ws_lamg; A.ws_shift = (h->ws_lamx && A.step_p) ? 1 : 0;
  A.weights = h->weights;
  A.pair_trials = h->pair_trials;
  A.sig_x = keep ? h->d_sigx : nullptr; A.sig_g = keep ? h->d_sigg : nullptr;
  // fetch order: explicit (nmpc_set_order) > the order the previous call on this handle prepared for the same B > natural
  A.order = h->order_next; h->order_next = nullptr;
  if (!A.order && h->auto_order && h->have_order && h->prev_B == B) A.order = h->d_order[par];
  A.order_out = h->auto_order ? h->d_order[par ^ 1] : nullptr;       // ... and this call prepares the next one's
  // Grid: one block per SM at most; with `fill` > 1 a small batch is packed onto fewer SMs (fill instances per warp,
  // refilled from the queue) so that concurrent solves of other handles find free SMs instead of SMs held by blocks
  // whose eight warps wait for one straggler.
  int blocks = B < h->max_blocks ? B : h->max_blocks;
  if (h->fill > 1) {
    const int packed = (B + h->warps_per_block * h->fill - 1) / (h->warps_per_block * h->fill);
    if (packed < blocks) blocks = packed < 1 ? 1 : packed;
  }
  if (const int rc = h->inst->launch(A, blocks, h->smem_bytes, s)) {
    // The kernel that would have reset the NEXT call's queue / done / work counters did not run: keep the parity (the
    // next call reuses THIS call's buffers) and put them back to their clean state, so that a later call can never
    // start from a stale queue counter and return without having written its outputs.
    cudaMemsetAsync(h->d_counter, 0, 4 * sizeof(int), s);
    cudaMemsetAsync(h->d_stats, 0, 2 * NSTAT * sizeof(unsigned long long), s);
    h->have_order = 0; h->prev_B = 0;
    return fail(f + ": launch failed: " + cudaGetErrorString((cudaError_t)rc));
  }
  // the launch is enqueued: it owns buffer set `par` and prepares set `par ^ 1` for the next call
  h->parity = par ^ 1;
  h->stats_last = h->d_stats + NSTAT * par;
  h->have_order = h->auto_order;
  h->launches = 1;
  h->prev_B = B;
  h->last_stream = s;
  h->sched_iter += sched_steps;
  h->kept_B = keep ? B : 0;
  if (keep) { CK(cudaEventRecord(h->ev_keep, s)); h->keep_stream = s; }
  return 0;
}

// nmpc_eval and nmpc_lam_p: A holds the call's arrays; `missing` says that one the entry point requires is NULL.
static int launch_eval(nmpc_handle* h, const char* fn, EvalArgs A, uint32_t flags, bool missing, void* cuda_stream) {
  if (refused(h, fn, NULL_HANDLE)) return 1;
  if (A.B <= 0) return 0;
  if (refused(h, fn, PREDICT_WITHOUT_VW, nullptr, flags)) return 1;
  if (missing) return fail(std::string(fn) + ": null required pointer");
  if (refused(h, fn, NO_OBSTACLES, A.obs)) return 1;
  if (A.jtv && !A.lam) return fail(std::string(fn) + ": jtv needs lam");
  if (A.hv && !A.v) return fail(std::string(fn) + ": hv needs v");
  CK(cudaSetDevice(h->device));
  A.pr = h->pr; A.obs_per_instance = (flags & NMPC_OBS_PER_INSTANCE) ? 1 : 0;
  A.weights = h->weights; A.tgt = h->tgt;
  const int warps = 4;
  nmpc_eval_kernel<<<(A.B + warps - 1) / warps, warps * 32, 0, (cudaStream_t)cuda_stream>>>(A);
  CK(cudaGetLastError());
  h->last_stream = (cudaStream_t)cuda_stream; h->launches = 1;
  return 0;
}

extern "C" {

const char* nmpc_last_error(void) { return g_err.c_str(); }
const char* nmpc_version(void) { return "nmpc_b200 0.1 (sm_100a)"; }
int32_t nmpc_n_w(const nmpc_spec* s) { return model_nu(s->model) * s->N; }
int32_t nmpc_n_g(const nmpc_spec* s) { return (model_nb(s->model) + s->n_obs) * (s->N + 1); }
int32_t nmpc_n_p(const nmpc_spec* s) { return model_np(s->model); }

extern "C" int nmpc_destroy(nmpc_handle* h);
int nmpc_create(const nmpc_spec* spec, int device, nmpc_handle** out) {
  if (!spec || !out) return fail("nmpc_create: null argument");
  if (spec->N < 1 || spec->N + 1 > NMPC_MAX_STAGES) return fail("nmpc_create: need 1 <= N <= 31");
  if (spec->n_obs < 0 || spec->n_obs > NMPC_MAX_OBS) return fail("nmpc_create: need 0 <= n_obs <= 16");
  if (!(spec->T > 0)) return fail("nmpc_create: T must be positive");
  if (spec->model != NMPC_MODEL_GIMBAL && spec->model != NMPC_MODEL_GIMBAL_LESS) return fail("nmpc_create: model must be NMPC_MODEL_GIMBAL (0) or NMPC_MODEL_GIMBAL_LESS (1)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("nmpc_create: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail("nmpc_create: bad device index");
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail("nmpc_create: kernels are built for sm_100a only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
  CK(cudaSetDevice(device));
  nmpc_handle* h = new (std::nothrow) nmpc_handle();
  if (!h) return fail("nmpc_create: out of memory");
  memset(h, 0, sizeof *h);
  h->spec = *spec; h->device = device; h->sm_count = prop.multiProcessorCount;
  h->pr.T = spec->T; h->pr.w1 = spec->w1; h->pr.w2 = spec->w2; h->pr.hv = 0.5 * spec->vfov; h->pr.hh = 0.5 * spec->hfov;
  h->pr.N = spec->N; h->pr.n_obs = spec->n_obs; h->pr.R = model_nb(spec->model) + spec->n_obs; h->pr.S = spec->N + 1;
  h->pr.model = spec->model;
  if (spec->model == NMPC_MODEL_GIMBAL_LESS) { h->pr.w1 = 1.0; h->pr.w2 = 0.0; }     // distance-only cost (NMPC_TT.m:100-104)
  h->opt = Opt();
  h->opt.max_iter = spec->max_iter > 0 ? spec->max_iter : 100;
  h->opt.scaling = spec->scaling; h->opt.tol = spec->tol > 0 ? spec->tol : 1e-8;
  h->inst = nullptr;
  for (const IpmInst& in : IPM_INSTS) if (in.N == spec->N && in.n_obs == spec->n_obs && in.model == spec->model) h->inst = &in;
  if (!h->inst) {
    std::string have;
    for (const IpmInst& in : IPM_INSTS) have += " (" + std::to_string(in.N) + "," + std::to_string(in.n_obs) + (in.model ? ",model 1)" : ")");
    delete h;
    return fail("nmpc_create: no kernel instantiation for this (N, n_obs, model); built:" + have + " -- add it to csrc/Makefile INSTS and the table in nmpc_b200.cu");
  }
  {
    const int rc = h->inst->prepare(&h->blocks_per_sm, &h->smem_bytes, &h->warps_per_block, &h->cold_stride);
    if (rc != 0) { delete h; return fail(std::string("nmpc_create: kernel setup failed: ") + cudaGetErrorString((cudaError_t)rc)); }
  }
  if (h->blocks_per_sm < 1) { delete h; return fail("nmpc_create: kernel does not fit on an SM"); }
  h->max_blocks = h->sm_count * h->blocks_per_sm;
  h->pair_trials = 1;         // N <= 15: a trial pass of the line search also evaluates the next trial point (bit-identical)
  if (const char* e = getenv("NMPC_B200_PAIR_TRIALS")) h->pair_trials = atoi(e) != 0;      // tuning knob: 0 = one trial point per pass
  h->fill = spec->fill > 1 ? spec->fill : 1;
  h->auto_order = 1;
  if (const char* e = getenv("NMPC_B200_AUTO_ORDER")) h->auto_order = atoi(e) != 0;
  h->ric_stride = RIC_N * h->pr.N;
  CKH(cudaMalloc(&h->d_ric, sizeof(double) * (size_t)h->ric_stride * h->max_blocks * h->warps_per_block));   // L2-resident Riccati scratch
  CKH(cudaMalloc(&h->d_cold, sizeof(double) * (size_t)h->cold_stride * h->max_blocks * h->warps_per_block));   // rare paths: restoration, watchdog
  CKH(cudaMalloc(&h->d_ricmap, sizeof(unsigned) * 32 * RIC_MAP_WORDS));
  {
    const int rc = h->inst->ricmap(h->d_ricmap, 0);
    if (rc != 0) { nmpc_destroy(h); return fail(std::string("nmpc_create: map kernel failed: ") + cudaGetErrorString((cudaError_t)rc)); }
    CKH(cudaDeviceSynchronize());
  }
  CKH(cudaMalloc(&h->d_counter, 4 * sizeof(int)));
  CKH(cudaMemset(h->d_counter, 0, 4 * sizeof(int)));
  CKH(cudaMalloc(&h->d_stats, 2 * NSTAT * sizeof(unsigned long long)));
  CKH(cudaMemset(h->d_stats, 0, 2 * NSTAT * sizeof(unsigned long long)));
  CKH(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  CKH(cudaEventCreateWithFlags(&h->ev_keep, cudaEventDisableTiming));
  CKH(cudaEventCreateWithFlags(&h->ev_sens, cudaEventDisableTiming));
  const int mb = spec->max_batch > 0 ? spec->max_batch : 0;
  if (mb > 0) {
    const size_t nw = (size_t)model_nu(spec->model) * spec->N, ng = (size_t)h->pr.R * h->pr.S;
    CKH(cudaMalloc(&h->d_p, sizeof(double) * mb * model_np(spec->model))); CKH(cudaMalloc(&h->d_x0, sizeof(double) * mb * nw));
    CKH(cudaMalloc(&h->d_lbx, sizeof(double) * nw)); CKH(cudaMalloc(&h->d_ubx, sizeof(double) * nw));
    CKH(cudaMalloc(&h->d_lbg, sizeof(double) * ng)); CKH(cudaMalloc(&h->d_ubg, sizeof(double) * ng));
    h->obs_cap = (size_t)mb * 3 * (spec->n_obs > 0 ? spec->n_obs : 1);
    CKH(cudaMalloc(&h->d_obs, sizeof(double) * h->obs_cap));
    CKH(cudaMalloc(&h->d_x, sizeof(double) * mb * nw)); CKH(cudaMalloc(&h->d_f, sizeof(double) * mb));
    CKH(cudaMalloc(&h->d_g, sizeof(double) * mb * ng)); CKH(cudaMalloc(&h->d_lamx, sizeof(double) * mb * nw));
    CKH(cudaMalloc(&h->d_lamg, sizeof(double) * mb * ng));
    CKH(cudaMalloc(&h->d_status, sizeof(int32_t) * mb)); CKH(cudaMalloc(&h->d_iters, sizeof(int32_t) * mb));
  }
  *out = h;
  return 0;
}

int nmpc_destroy(nmpc_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  void* ptrs[] = {h->d_ric, h->d_cold, h->d_counter, h->d_stats, h->d_p, h->d_x0, h->d_lbx, h->d_ubx, h->d_lbg, h->d_ubg, h->d_obs,
                  h->d_x, h->d_f, h->d_g, h->d_lamx, h->d_lamg, h->d_status, h->d_iters, h->d_order[0], h->d_order[1], h->d_keep_iters, h->d_ricmap, h->d_tgt_pred,
                  h->d_sigx, h->d_sigg};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->ev_keep) cudaEventDestroy(h->ev_keep);
  if (h->ev_sens) cudaEventDestroy(h->ev_sens);
  delete h;
  return 0;
}

int nmpc_solve(nmpc_handle* h, int32_t B, const double* p, const double* x0,
               const double* lbx, const double* ubx, const double* lbg, const double* ubg,
               const double* obst, uint32_t flags,
               double* x, double* f, double* g, double* lam_x, double* lam_g,
               int32_t* status, int32_t* iters, void* cuda_stream) {
  SolveArgs A = solve_args(B, p, x0, lbx, ubx, lbg, ubg, obst, flags, x, f, g, lam_x, lam_g, status, iters);
  return launch_solve(h, A, flags, (cudaStream_t)cuda_stream, "nmpc_solve");
}

int nmpc_solve_and_step(nmpc_handle* h, int32_t B, double* p, double* u_warm,
                        const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                        const double* obst, uint32_t flags, const double* target_vw,
                        double* x, double* f, double* fov_centre, double* err_accum,
                        int32_t* status, int32_t* iters, void* cuda_stream) {
  SolveArgs A = solve_args(B, p, u_warm, lbx, ubx, lbg, ubg, obst, flags, x, f, nullptr, nullptr, nullptr, status, iters);
  A.step_p = p; A.step_u = u_warm; A.step_vw = target_vw; A.step_fov = fov_centre; A.step_err = err_accum;
  return launch_solve(h, A, flags, (cudaStream_t)cuda_stream, "nmpc_solve_and_step", true);
}

int nmpc_run_closed_loop(nmpc_handle* h, int32_t B, int32_t steps, double* p, double* u_warm,
                         const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                         const double* obst, uint32_t flags, const double* target_vw,
                         double* x, double* f, double* fov_centre, double* err_accum,
                         int32_t* status_log, int32_t* iters_log, int32_t* converged, void* cuda_stream) {
  if (refused(h, "nmpc_run_closed_loop", NULL_HANDLE)) return 1;
  if (steps < 1) return fail("nmpc_run_closed_loop: steps must be >= 1");
  if (h->tgt) return fail("nmpc_run_closed_loop: a caller-given target trajectory (nmpc_set_target_trajectory) needs the step-by-step calls; "
                          "NMPC_PREDICT_TARGET predicts it on the device");
  SolveArgs A = solve_args(B, p, u_warm, lbx, ubx, lbg, ubg, obst, flags, x, f, nullptr, nullptr, nullptr, nullptr, nullptr);
  A.step_p = p; A.step_u = u_warm; A.step_vw = target_vw; A.step_fov = fov_centre; A.step_err = err_accum;
  A.run_steps = steps; A.status_log = status_log; A.iters_log = iters_log; A.conv_count = converged;
  return launch_solve(h, A, flags, (cudaStream_t)cuda_stream, "nmpc_run_closed_loop", true);
}

int nmpc_solve_host(nmpc_handle* h, int32_t B, const double* p, const double* x0,
                    const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                    const double* obst, uint32_t flags,
                    double* x, double* f, double* g, double* lam_x, double* lam_g,
                    int32_t* status, int32_t* iters) {
  const int rc = nmpc_solve_host_async(h, B, p, x0, lbx, ubx, lbg, ubg, obst, flags, x, f, g, lam_x, lam_g, status, iters);
  return rc ? rc : nmpc_synchronize(h);
}

int nmpc_synchronize(nmpc_handle* h) {
  if (!h) return fail("nmpc_synchronize: null handle");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->own_stream));
  return 0;
}

int nmpc_query(nmpc_handle* h, int32_t* busy) {
  if (!h || !busy) return fail("nmpc_query: null argument");
  CK(cudaSetDevice(h->device));
  const cudaError_t e = cudaStreamQuery(h->own_stream);
  if (e != cudaSuccess && e != cudaErrorNotReady) return fail(std::string("nmpc_query: ") + cudaGetErrorString(e));
  *busy = e == cudaErrorNotReady ? 1 : 0;
  return 0;
}

int nmpc_solve_host_async(nmpc_handle* h, int32_t B, const double* p, const double* x0,
                          const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                          const double* obst, uint32_t flags,
                          double* x, double* f, double* g, double* lam_x, double* lam_g,
                          int32_t* status, int32_t* iters) {
  if (refused(h, "nmpc_solve_host", NULL_HANDLE)) return 1;
  if (B <= 0) return 0;
  if (refused(h, "nmpc_solve_host", PREDICT_WITHOUT_VW, nullptr, flags)) return 1;
  if (B > h->spec.max_batch) return fail("nmpc_solve_host: B exceeds spec.max_batch");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = h->own_stream;
  const size_t nw = (size_t)model_nu(h->pr.model) * h->pr.N, ng = (size_t)h->pr.R * h->pr.S;
  const size_t nobs = (size_t)3 * h->pr.n_obs * ((flags & NMPC_OBS_PER_INSTANCE) ? B : 1);
  CK(cudaMemcpyAsync(h->d_p, p, sizeof(double) * B * model_np(h->pr.model), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_x0, x0, sizeof(double) * B * nw, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_lbx, lbx, sizeof(double) * nw, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_ubx, ubx, sizeof(double) * nw, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_lbg, lbg, sizeof(double) * ng, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->d_ubg, ubg, sizeof(double) * ng, cudaMemcpyHostToDevice, s));
  if (nobs) CK(cudaMemcpyAsync(h->d_obs, obst, sizeof(double) * nobs, cudaMemcpyHostToDevice, s));
  SolveArgs A = solve_args(B, h->d_p, h->d_x0, h->d_lbx, h->d_ubx, h->d_lbg, h->d_ubg, h->d_obs, flags, h->d_x, h->d_f,
                           g ? h->d_g : nullptr, lam_x ? h->d_lamx : nullptr, lam_g ? h->d_lamg : nullptr, h->d_status, h->d_iters);
  if (const int rc = launch_solve(h, A, flags, s, "nmpc_solve_host")) return rc;
  CK(cudaMemcpyAsync(x, h->d_x, sizeof(double) * B * nw, cudaMemcpyDeviceToHost, s));
  if (f) CK(cudaMemcpyAsync(f, h->d_f, sizeof(double) * B, cudaMemcpyDeviceToHost, s));
  if (g) CK(cudaMemcpyAsync(g, h->d_g, sizeof(double) * B * ng, cudaMemcpyDeviceToHost, s));
  if (lam_x) CK(cudaMemcpyAsync(lam_x, h->d_lamx, sizeof(double) * B * nw, cudaMemcpyDeviceToHost, s));
  if (lam_g) CK(cudaMemcpyAsync(lam_g, h->d_lamg, sizeof(double) * B * ng, cudaMemcpyDeviceToHost, s));
  if (status) CK(cudaMemcpyAsync(status, h->d_status, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, s));
  if (iters) CK(cudaMemcpyAsync(iters, h->d_iters, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, s));
  return 0;
}

int nmpc_eval(nmpc_handle* h, int32_t B, const double* w, const double* p, const double* obst, uint32_t flags,
              double sigma, const double* lam, const double* v,
              double* f, double* g, double* grad_f, double* jtv, double* hv, void* cuda_stream) {
  return launch_eval(h, "nmpc_eval", EvalArgs{{}, B, w, p, obst, 0, nullptr, nullptr, sigma, lam, v, f, g, grad_f, jtv, hv}, flags, !w || !p, cuda_stream);
}

int nmpc_lam_p(nmpc_handle* h, int32_t B, const double* x_sol, const double* p, const double* obst, uint32_t flags,
               const double* lam_g, double* lam_p, void* cuda_stream) {
  const EvalArgs A{{}, B, x_sol, p, obst, 0, nullptr, nullptr, 1.0, lam_g, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, lam_p};
  return launch_eval(h, "nmpc_lam_p", A, flags, !x_sol || !p || !lam_g || !lam_p, cuda_stream);
}

// One launch of the sensitivity kernel for the entry point `fn`: the p and weight columns (dx_dp, required, and dx_dw) or,
// with `obstacles`, the obstacle columns (dx_do, required).
static int launch_sens(nmpc_handle* h, const char* fn, bool obstacles, int32_t B, const double* x_sol, const double* p, const double* lam_g,
                       const double* obst, uint32_t flags, double* dx_dp, double* dx_dw, double* dx_do, int32_t* sens_status, void* cuda_stream) {
  const std::string f(fn);
  if (refused(h, fn, NULL_HANDLE | (obstacles ? NO_OBSTACLE_ROWS : 0u))) return 1;
  if (B <= 0) return 0;
  if (refused(h, fn, NOT_KEPT | KEPT_OTHER_B | WEIGHTS_OF_MODEL_1 | PREDICT_WITHOUT_VW, nullptr, flags, B, dx_dw)) return 1;
  if (!x_sol || !p || !lam_g || !(obstacles ? dx_do : dx_dp)) return fail(f + ": null required pointer");
  if (refused(h, fn, NO_OBSTACLES, obst)) return 1;
  CK(cudaSetDevice(h->device));
  // x_sol enters as the start point x0 (ph_load puts it where the solve keeps its iterate) and as x
  SolveArgs A = solve_args(B, p, x_sol, nullptr, nullptr, nullptr, nullptr, obst, flags, const_cast<double*>(x_sol), nullptr, nullptr,
                           nullptr, const_cast<double*>(lam_g), nullptr, nullptr);
  A.pr = h->pr; A.o = h->opt;
  A.weights = h->weights; A.tgt = h->tgt;
  A.sig_x = h->d_sigx; A.sig_g = h->d_sigg;
  A.ric = h->d_ric; A.ric_stride = h->ric_stride; A.ricmap = h->d_ricmap;
  A.dx_dp = dx_dp; A.dx_dw = dx_dw; A.sens_status = sens_status; A.dx_do = dx_do;
  const cudaStream_t s = (cudaStream_t)cuda_stream;
  if (h->keep_stream != s) CK(cudaStreamWaitEvent(s, h->ev_keep, 0));      // the kept Sigmas are complete
  const int slots = h->max_blocks * h->warps_per_block;      // the Riccati scratch holds one slot per resident warp of the solve
  if (const int rc = h->inst->sens(A, B < slots ? B : slots, s)) return fail(f + ": launch failed: " + cudaGetErrorString((cudaError_t)rc));
  CK(cudaEventRecord(h->ev_sens, s));
  h->sens_pending = 1; h->sens_stream = s;
  h->last_stream = s; h->launches = 1;
  return 0;
}

int nmpc_sensitivity(nmpc_handle* h, int32_t B, const double* x_sol, const double* p, const double* lam_g, const double* obst,
                     uint32_t flags, double* dx_dp, double* dx_dw, int32_t* sens_status, void* cuda_stream) {
  return launch_sens(h, "nmpc_sensitivity", false, B, x_sol, p, lam_g, obst, flags, dx_dp, dx_dw, nullptr, sens_status, cuda_stream);
}

int nmpc_sensitivity_obstacles(nmpc_handle* h, int32_t B, const double* x_sol, const double* p, const double* lam_g,
                               const double* obst, uint32_t flags, double* dx_dobst, int32_t* sens_status, void* cuda_stream) {
  return launch_sens(h, "nmpc_sensitivity_obstacles", true, B, x_sol, p, lam_g, obst, flags, nullptr, nullptr, dx_dobst, sens_status, cuda_stream);
}

int nmpc_barrier_data(nmpc_handle* h, double* sig_x, double* sig_g, void* cuda_stream) {
  if (refused(h, "nmpc_barrier_data", NULL_HANDLE)) return 1;
  if (refused(h, "nmpc_barrier_data", NOT_KEPT)) return 1;
  CK(cudaSetDevice(h->device));
  if (h->keep_stream != (cudaStream_t)cuda_stream) CK(cudaStreamWaitEvent((cudaStream_t)cuda_stream, h->ev_keep, 0));
  const size_t B = h->kept_B, nw = (size_t)model_nu(h->pr.model) * h->pr.N, ng = (size_t)h->pr.R * h->pr.S;
  if (sig_x) CK(cudaMemcpyAsync(sig_x, h->d_sigx, sizeof(double) * B * nw, cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream));
  if (sig_g) CK(cudaMemcpyAsync(sig_g, h->d_sigg, sizeof(double) * B * ng, cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream));
  return 0;
}

int nmpc_step(nmpc_handle* h, int32_t B, const double* x_sol, double* p,
              double* u_warm, const double* target_vw, double* fov_centre, double* err_accum, void* cuda_stream) {
  if (!h) return fail("nmpc_step: null handle");
  if (B <= 0) return 0;
  if (!x_sol || !p || !u_warm || !target_vw) return fail("nmpc_step: null required pointer");
  CK(cudaSetDevice(h->device));
  if (err_accum && !fov_centre) return fail("nmpc_step: err_accum needs fov_centre");
  StepArgs A{h->pr.T, h->pr.hv, h->pr.hh, h->pr.N, B, h->pr.model, x_sol, p, u_warm, target_vw, fov_centre, err_accum};
  nmpc_step_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)cuda_stream>>>(A);
  CK(cudaGetLastError());
  h->last_stream = (cudaStream_t)cuda_stream; h->launches = 1;
  return 0;
}

int nmpc_set_order(nmpc_handle* h, const int32_t* dev_order) {
  if (!h) return fail("nmpc_set_order: null handle");
  h->order_next = dev_order;
  return 0;
}

int nmpc_set_weights(nmpc_handle* h, const double* dev_weights) {
  if (!h) return fail("nmpc_set_weights: null handle");
  h->weights = dev_weights;
  return 0;
}

int nmpc_set_target_trajectory(nmpc_handle* h, const double* dev_targets) {
  if (!h) return fail("nmpc_set_target_trajectory: null handle");
  h->tgt = dev_targets;
  return 0;
}

int nmpc_set_obstacle_motion(nmpc_handle* h, double* dev_obst, const double* dev_vel) {
  if (!h) return fail("nmpc_set_obstacle_motion: null handle");
  if ((dev_obst == nullptr) != (dev_vel == nullptr)) return fail("nmpc_set_obstacle_motion: give both the obstacle field and the velocities, or neither");
  if (dev_obst && h->pr.n_obs == 0) return fail("nmpc_set_obstacle_motion: this handle has no obstacle rows (spec.n_obs = 0)");
  h->move_obs = dev_obst; h->move_vel = dev_vel;
  return 0;
}

int nmpc_set_warm_start(nmpc_handle* h, double* dev_lam_x0, double* dev_lam_g0, const nmpc_warm_opts* opts) {
  if (!h) return fail("nmpc_set_warm_start: null handle");
  if ((dev_lam_x0 == nullptr) != (dev_lam_g0 == nullptr)) return fail("nmpc_set_warm_start: give both multiplier guesses or neither");
  h->ws_lamx = dev_lam_x0; h->ws_lamg = dev_lam_g0;
  if (opts) {
    const Opt d = Opt();
    auto pick = [](double v, double dflt) { return v > 0.0 ? v : dflt; };
    h->opt.ws_mu_init = pick(opts->mu_init, d.ws_mu_init);
    h->opt.ws_bound_push = pick(opts->bound_push, d.ws_bound_push); h->opt.ws_bound_frac = pick(opts->bound_frac, d.ws_bound_frac);
    h->opt.ws_slack_push = pick(opts->slack_bound_push, d.ws_slack_push); h->opt.ws_slack_frac = pick(opts->slack_bound_frac, d.ws_slack_frac);
    h->opt.ws_mult_push = pick(opts->mult_bound_push, d.ws_mult_push);
  }
  return 0;
}

int nmpc_set_schedule(nmpc_handle* h, const double* dev_table, int32_t n_rows, int32_t len,
                      const int32_t* dev_row_of_instance, const int32_t* dev_phase, int32_t mpc_iter) {
  if (!h) return fail("nmpc_set_schedule: null handle");
  if (dev_table && (n_rows < 1 || len < 1)) return fail("nmpc_set_schedule: need n_rows >= 1 and len >= 1");
  h->sched_table = dev_table; h->sched_rows = n_rows; h->sched_len = len;
  h->sched_id = dev_row_of_instance; h->sched_phase = dev_phase; h->sched_iter = mpc_iter;
  return 0;
}

int nmpc_set_debug_log(nmpc_handle* h, double* dev_buf, int32_t rows) {
  if (!h) return fail("nmpc_set_debug_log: null handle");
  h->dbg = dev_buf; h->dbg_rows = dev_buf ? rows : 0;
  return 0;
}

int nmpc_get_stats(nmpc_handle* h, nmpc_stats* out) {
  if (!h || !out) return fail("nmpc_get_stats: null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->last_stream));
  unsigned long long st[NSTAT];
  CK(cudaMemcpy(st, h->stats_last ? h->stats_last : h->d_stats, sizeof st, cudaMemcpyDeviceToHost));
  out->kernel_launches = h->launches; out->factorizations = (int64_t)st[0]; out->ls_trials = (int64_t)st[1]; out->soc_accepted = (int64_t)st[2];
  out->resto_calls = (int64_t)st[3]; out->resto_iters = (int64_t)st[4]; out->watchdog_starts = (int64_t)st[5];
  out->soft_resto_steps = (int64_t)st[6]; out->filter_resets = (int64_t)st[7]; out->trial_passes = (int64_t)st[8];
  return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// FP64 roofline denominator: register-resident DFMA loop on every SM (MEASURED_PEAKS.json has no FP64 entry)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nmpc_dfma_peak_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x * 1e-3, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  const double s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (s == 123.456) out[0] = s;   // never true; keeps the loop alive
}

extern "C" int nmpc_measure_fp64_peak(int device, double* tflops) {
  if (!tflops) return fail("nmpc_measure_fp64_peak: null argument");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
  double* d = nullptr; CK(cudaMalloc(&d, sizeof(double)));
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
  double best = 0.0;
  for (int rep = 0; rep < 6; ++rep) {
    CK(cudaEventRecord(e0, 0));
    nmpc_dfma_peak_kernel<<<blocks, threads>>>(d, iters, 0.999999, 1e-9);
    CK(cudaEventRecord(e1, 0));
    CK(cudaEventSynchronize(e1));
    float ms = 0; CK(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
    if (rep > 0) best = fmax(best, fl / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  *tflops = best;
  return 0;
}
