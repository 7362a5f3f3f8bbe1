// nmpc_device.cuh -- device-side building blocks of the batched NMPC solver (sm_100a, FP64).
//
// One warp owns one NLP instance; lane k owns horizon stage k (N + 1 <= 32).
//   * rollout (NMPC_TT.py:160-167) = warp prefix sums: the five angle states are pure integrators
//     of their rate controls, the positions are prefix sums of T*v*[cos(psi)cos(th), sin(psi)cos(th), sin(th)].
//   * stage cost (NMPC_TT.py:193-221) in its compact form  w1*dist + w2*((P/a)^2 + (Q/b)^2 - 1)
//     with hand-derived gradient and Hessian (chain rule through the intermediates (Dx, Dy, a, b, X7)).
//   * Newton step of the reduced (single-shooting) primal-dual system = stage-structured LQ problem,
//     solved by a Riccati recursion (nmpc_riccati.cuh): per stage a 15 x 15 matrix built by all 32 lanes, a 6 x 6
//     Cholesky in registers, 9 forward/back substitutions and a 44-entry trailing update.
// Code-size discipline: transcendental functions and the big phases are __noinline__ so that every
// heavy instruction sequence exists once (v1 was 785 KB of SASS and stalled on instruction fetch).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

namespace nmpc {

constexpr unsigned FULL = 0xffffffffu;
constexpr int NX = 8, NU = 6, NPAR = 11;
// Model 1 = the gimbal-less tracker of MATLAB/Dynamic Obstacles/NMPC_TT.m:25-35 (states x, y, z, theta, psi; controls v,
// omega_2, omega_3; p = [state(5); target(3)]; cost = horizontal distance, :100-104; rows [z, theta], :107-111).  Its dynamics
// are the first five rows of model 0's, so it runs on the same 8-state / 6-control machinery with the camera states held
// at zero: the three camera controls are ABSENT variables (no bounds, no multipliers, zero gradient; a unit entry on the
// diagonal of the control block keeps the stage systems decoupled and positive, their step is exactly zero), and only the
// first NB = 2 box rows exist.  The C ABI sees the model's own sizes (3N controls, 2 (N + 1) rows, p[8]).
__host__ __device__ constexpr int model_nu(int model) { return model ? 3 : 6; }
__host__ __device__ constexpr int model_nb(int model) { return model ? 2 : 5; }
__host__ __device__ constexpr int model_np(int model) { return model ? 8 : 11; }

// ---- per-lane vectors in shared memory: index e * S + stage ------------------------------------
enum LvEnt { LV_U = 0, LV_ZL = 6, LV_ZU = 12, LV_X = 18, LV_GL = 26, LV_DX = 32, LV_DU = 40, LV_N = 46 };
// ---- per-row (constraint) arrays in shared memory: index (arr * R + r) * S + stage --------------
// The obstacle rows have no lower bound in this NLP family (lbg = -inf, NMPC_TT.py:280-282), so the two arrays that belong
// to lower bounds (multiplier v_L and reciprocal slack 1/(s - l)) exist for the five box rows only: they come last and
// hold NBOX rows instead of R.  A finite lower bound on an obstacle row is refused (NMPC_INVALID_NUMBER).
// (the scaled row values g themselves are not kept: every reader visits the rows with the cached states X at hand and
// recomputes g = dc * row(X), bit for bit what ph_derivs had)
enum RowArr { A_S = 0, A_Y, A_VU, A_DS, A_DC, A_IU, A_NFULL, A_VL = A_NFULL, A_IL, A_NROW };
// ---- per-stage LQ data (entry-major: e * S + stage).  Entries [0, LQ_DEAD) are dead once the
//      factorisation has succeeded and are reused by the second-order-correction arrays. ----------
enum LqEnt {
  LQ_Q = 0,        // 24: 21 = packed lower triangle over (x,y,z,X5,X6,X7), +3 = (theta,theta),(psi,theta),(psi,psi)
  LQ_DEAD = 24,
  LQ_QA = 24,      // 8 : grad l + G^T (Sigma_s c)                     -- q = QA + mu*QB + dw*QD
  LQ_SV = 32,      // 2 : d2/dv dtheta, d2/dv dpsi (only non-zeros of the control-state block)
  LQ_RD = 34,      // 6 : diagonal control block Sigma_x (without delta_w)
  LQ_RB = 40,      // 6 : control gradient per unit mu                 -- r = mu * RB
  LQ_DD = 46,      // 3 : direction d = (cps*cth, sps*cth, sth)
  LQ_EE = 49,      // 5 : T*E03, T*E13, T*E23, T*E04, T*E14
  LQ_ZERO = 54,    // 1 : 0.0 (lets the Riccati add its stage terms without branches)
  LQ_NFOLD = 55,   // ---- the entries below hold the mu / delta_w parts separately, so that an inertia-correction retry
                   //      re-factors without re-evaluating anything.  Layouts that gain a resident warp by dropping them
                   //      (Lay::FOLD) fold mu and delta_w into Q / QA in ph_derivs and re-run it on a retry instead.
  LQ_DG = 55,      // 5 : dc_r^2 of the five box rows                  -- delta_w part of G^T D_s G
  LQ_NN = 60,      // 3 : sum_j dc_j^2 n_j n_j^T (xx, xy, yy)          -- delta_w part of G^T D_s G
  LQ_QD = 63,      // 8 : G^T c                                        -- delta_w part of q
  LQ_QB = 71,      // 8 : G^T beta                                     -- mu part of q
  LQ_N = 79
};
// second-order-correction scratch in shared memory (offsets in units of S doubles inside the `soc` region):
//   CT [R] (residual of the last trial point), DUS [6], Q2 [8];  the two arrays only the SOC itself touches (DS2, CSOC)
//   live in the cold global scratch
// Riccati factors in the per-warp global (L2-resident) scratch, per stage:
constexpr int RIC_K = 0;      // 54: rows r=0..5 of [K | kappa], 9 doubles each
constexpr int RIC_L = 54;     // 21: Cholesky factor of Lambda (packed lower) + 6 inverse diagonal
constexpr int RIC_K2 = 81;    // 6 : kappa of the SOC right-hand side
constexpr int RIC_N = 88;
constexpr int FILT_CAP = 24;
constexpr int ALG_N = 50;     // per-warp algorithm state kept in shared memory
constexpr int STG_N = 282;    // Riccati staging area (nmpc_riccati.cuh)

// scalar results returned by the phases through shared memory
enum Res { R_F = 0, R_DU, R_PR, R_SUMY, R_SUMZ, R_VIOL, R_PMAX, R_PMIN, R_APR, R_ADU, R_GBD, R_THETA, R_TINY,
           R_FT, R_THT, R_LBT, R_DTT, R_YMAX,
           R_DU1, R_CO1,          // 1-norms of the dual infeasibility and of (slack * multiplier - mu): soft restoration test
           R_OTH, R_OINF,         // restoration mode: 1-norm / max-norm of the ORIGINAL problem's residual g - s
           R_DYMAX,               // max |dy| of the step (tiny-step logic)
           R_NFILT,               // filter length after an augmentation (written by lane 0)
           R_FT2, R_THT2, R_LBT2, R_DTT2,     // R_FT .. R_DTT of the next backtracking trial point (paired ph_trial, lane SW)
           R_N };
constexpr int RES_N = 28;
static_assert(R_N <= RES_N, "RES region is 28 doubles");

__host__ __device__ inline int tri(int r, int c) { return r >= c ? r * (r + 1) / 2 + c : c * (c + 1) / 2 + r; }
// state index of the five linear ("box") rows [z, theta, X5, X6, X7]   NMPC_TT.py:236-240
__device__ __forceinline__ int box_state(int r) { return r == 0 ? 2 : (r == 1 ? 3 : r + 3); }
// compact cost variable (x,y,z,X5,X6,X7) -> state index
__device__ __forceinline__ int cost_state(int v) { return v < 3 ? v : v + 2; }
// index into LQ_Q of the state-Hessian entry (i, j); -1 for structural zeros
__device__ __forceinline__ int q_index(int i, int j) {
  const bool ai = (i == 3 || i == 4), aj = (j == 3 || j == 4);
  if (ai != aj) return -1;
  if (ai) return 21 + (i - 3) + (j - 3);            // (3,3)->21, (3,4)/(4,3)->22, (4,4)->23
  const int ci = i < 3 ? i : i - 2, cj = j < 3 ? j : j - 2;
  return tri(ci, cj);
}

// ---- no-inline math: one copy of each slow sequence ---------------------------------------------
static __device__ __noinline__ double n_tan(double x) { return tan(x); }
static __device__ __noinline__ double n_log(double x) { return log(x); }
static __device__ __noinline__ double n_pow(double x, double y) { return pow(x, y); }
static __device__ __noinline__ double2 n_sincos(double x) { double2 r; sincos(x, &r.x, &r.y); return r; }
__device__ __forceinline__ double rcp(double x) { return __drcp_rn(x); }
// IPOPT's CalculateSafeSlack: a slack that rounding has pushed to (or below) eps * min(1, mu) is replaced by a tiny
// positive value and the bound moved.  Here the accepted VARIABLE is moved instead (ph_accept / ph_repair), to
// slack = max(slack, 0) + slack_move * max(1, |bound|), slack_move = eps^(3/4).
__device__ __forceinline__ double safe_value(double sl, double bnd) { return fmax(sl, 0.0) + 1.8189894035458565e-12 * fmax(1.0, fabs(bnd)); }

// ---- warp collectives ---------------------------------------------------------------------------
static __device__ __noinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
// warp_sum within each aligned group of W lanes.  When the lanes >= W hold +0.0, lane 0 gets bit for bit what warp_sum
// gives it: the butterfly steps with offsets >= W then only add +0.0 to lane 0's partial sum, which changes nothing but
// -0.0 -> +0.0, and the first add does exactly that.
template <int W>
static __device__ __noinline__ double seg_sum(double v) {
  v = __dadd_rn(v, 0.0);
#pragma unroll
  for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
static __device__ __noinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
  return v;
}
static __device__ __noinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
  return v;
}
// exclusive prefix sums of NV independent values (interleaved for ILP).  W (a power of two >= the number of stages): lanes >= W
// hold zeros and are not needed, so the steps with offsets >= W are dropped (they would add exact zeros: same results).
template <int NV, int W = 32>
__device__ __forceinline__ void scan_excl(double* v, int lane) {
#pragma unroll
  for (int o = 1; o < W; o <<= 1) {
    double t[NV];
#pragma unroll
    for (int c = 0; c < NV; ++c) t[c] = __shfl_up_sync(FULL, v[c], o);
    if (lane >= o) {
#pragma unroll
      for (int c = 0; c < NV; ++c) v[c] += t[c];
    }
  }
#pragma unroll
  for (int c = 0; c < NV; ++c) { const double e = __shfl_up_sync(FULL, v[c], 1); v[c] = lane == 0 ? 0.0 : e; }
}
// inclusive suffix sums of NV independent values (W as above)
template <int NV, int W = 32>
__device__ __forceinline__ void rscan_incl(double* v, int lane) {
#pragma unroll
  for (int o = 1; o < W; o <<= 1) {
    double t[NV];
#pragma unroll
    for (int c = 0; c < NV; ++c) t[c] = __shfl_down_sync(FULL, v[c], o);
    if (lane + o < 32) {
#pragma unroll
      for (int c = 0; c < NV; ++c) v[c] += t[c];
    }
  }
}
__device__ __forceinline__ double shfl_next(double v, int lane) {   // value of lane+1 (0 for the last lane)
  const double t = __shfl_down_sync(FULL, v, 1);
  return lane == 31 ? 0.0 : t;
}

// ---- problem constants passed by value to the kernels ---------------------------------------------
struct Prob {
  double T, w1, w2, hv, hh;   // hv = VFOV/2, hh = HFOV/2
  int N, n_obs, R, S;         // R = (5 | 2) + n_obs rows per stage, S = N + 1 stages
  int model;                  // 0: UAV + gimballed camera (the Python scripts), 1: gimbal-less tracker
};

// ---- compile-time shared-memory layout of one warp's workspace (offsets from the warp's slice base).
//      With N and n_obs as template parameters every workspace access is an LDS/STS with an immediate offset.
#ifndef NMPC_WPB_MAX
#define NMPC_WPB_MAX 8     // 8 warps x 255 registers is the whole register file of an SM
#endif
__host__ __device__ constexpr int even_up(int n) { return (n + 1) & ~1; }
template <int N_, int NOBS_, bool FOLD_, int MODEL_ = 0>
struct LayT {
  static constexpr int MODEL = MODEL_, NB = model_nb(MODEL_), NUA = model_nu(MODEL_), NPA = model_np(MODEL_);
  static constexpr int N = N_, S = N_ + 1, R = NB + NOBS_, NOBS = NOBS_;
  static constexpr int SW = S <= 8 ? 8 : (S <= 16 ? 16 : 32);      // width of the warp scans over the stages
  static constexpr bool PAIR = 2 * SW <= 32;                        // a second trial point fits lanes SW .. 2 SW - 1 (ph_trial)
  static constexpr bool FOLD = FOLD_;
  static constexpr int LQ_NE = FOLD_ ? LQ_NFOLD : LQ_N;
  static constexpr int LV0 = 0;
  static constexpr int RW0 = even_up(LV0 + LV_N * S);
  static constexpr int RW_N = (A_NFULL * R + (A_NROW - A_NFULL) * NB) * S;
  __host__ __device__ static constexpr int rw(int arr, int r) { return RW0 + (arr < A_NFULL ? arr * R + r : A_NFULL * R + (arr - A_NFULL) * NB + r) * S; }
  static constexpr int LQ0 = even_up(RW0 + RW_N);
  // Second-order-correction scratch in shared memory: du_soc [6] and q' [8], in the LQ entries that are dead after
  // the factorisation (the residual of the last trial point, c_t [R], goes to the cold scratch with the other SOC arrays).
  static constexpr int SOC_N = 14;
  static constexpr bool SOC_ALIAS = SOC_N <= LQ_DEAD;
  static constexpr int SOC_LO = SOC_N;
  static_assert(SOC_ALIAS, "SOC scratch must fit the dead LQ entries");
  static constexpr int SOCX0 = even_up(LQ0 + LQ_NE * S);
  static constexpr int STG0 = even_up(SOCX0 + (SOC_N - SOC_LO) * S);
  __host__ __device__ static constexpr int soc(int e) { return e < SOC_LO ? LQ0 + e * S : SOCX0 + (e - SOC_LO) * S; }
  static constexpr int OBS0 = STG0 + STG_N;
  static constexpr int ALG0 = even_up(OBS0 + 3 * NOBS_ + 1);     // algorithm state (nmpc_solve.cuh: AlgF), ALG_N doubles
  static constexpr int RES0 = ALG0 + ALG_N;
  static constexpr int PAR0 = RES0 + RES_N;
  static constexpr int TOTAL = even_up(PAR0 + 14);   // p (11), w1, w2 of this instance
  // warps (= concurrent instances) per block: as many slices as fit in the 227 KB a block may use, at most NMPC_WPB_MAX
  // ---- cold per-warp scratch in global memory (touched only by the watchdog, the soft restoration phase and the
  //      restoration phase): restoration row arrays, reference controls, the restoration problem's own filter, and three
  //      slots that hold a saved iterate + step
  static constexpr int RSZ = R * S;
  static constexpr int CG_ROWS = 0;                     // 13 arrays [R][S]: n, p, z_n, z_p, dn, dp, dy, dn_soc, dp_soc, dy_soc, ds_soc, c_soc, c_t
  static constexpr int CG_UR = 13 * RSZ;                // [6][S] reference controls x_R of the restoration problem
  static constexpr int CG_FILT = CG_UR + 6 * S;         // [2][FILT_CAP][2]: filter of the original problem, of the restoration problem
  static constexpr int CG_PARK = CG_FILT + 4 * FILT_CAP;   // [ALG_N] algorithm state of the original problem while the restoration phase runs
  static constexpr int CG_SLOT = CG_PARK + ALG_N;
  static constexpr int SLOT_N = 32 * S + 8 * RSZ + 2 * NB * S;   // U ZL ZU (18 S) | DX DU (14 S) | S Y VU IU (4 RS) | VL IL (2 NB S) | n p z_n z_p (4 RS)
  static constexpr int COLD_TOTAL = even_up(CG_SLOT + 3 * SLOT_N);
  static constexpr int WPB_FIT = (227 * 1024) / (TOTAL * 8);
  static constexpr int WPB = WPB_FIT < 1 ? 1 : (WPB_FIT > NMPC_WPB_MAX ? NMPC_WPB_MAX : WPB_FIT);
};

// FOLD where it buys another resident warp per SM (big layouts), the separate mu / delta_w entries otherwise
#ifndef NMPC_FOLD_MIN_S
#define NMPC_FOLD_MIN_S 20     // measured: (30,10) 3 -> 4 warps per SM is +16 % (config 5); (15,10) 6 -> 7 warps is -3 % (config 4), so short horizons keep the separate entries
#endif
template <int N_, int NOBS_, int MODEL_ = 0>
using Lay = LayT<N_, NOBS_, (N_ + 1 >= NMPC_FOLD_MIN_S) && (LayT<N_, NOBS_, true, MODEL_>::WPB > LayT<N_, NOBS_, false, MODEL_>::WPB), MODEL_>;

// ---- stage state of one lane -----------------------------------------------------------------------
struct Stage {
  double X[NX];
  double sth, cth, sps, cps;
};

// Rollout by prefix sums.  u is this lane's control (ignored for lanes >= N).  NMPC_TT.py:139-148,160-167
template <int W = 32>
__device__ __forceinline__ void rollout(const Prob& pr, const double* __restrict__ X0, const double* u, int lane, Stage& st) {
  const bool has_u = lane < pr.N;
  const double T = pr.T;
  double a[5];
#pragma unroll
  for (int c = 0; c < 5; ++c) a[c] = has_u ? T * u[c + 1] : 0.0;
  scan_excl<5, W>(a, lane);
#pragma unroll
  for (int c = 0; c < 5; ++c) st.X[3 + c] = X0[3 + c] + a[c];
  const double2 sct = n_sincos(st.X[3]), scp = n_sincos(st.X[4]);
  st.sth = sct.x; st.cth = sct.y; st.sps = scp.x; st.cps = scp.y;
  const double tv = has_u ? T * u[0] : 0.0;
  double inc[3] = {tv * st.cps * st.cth, tv * st.sps * st.cth, tv * st.sth};
  scan_excl<3, W>(inc, lane);
  st.X[0] = X0[0] + inc[0]; st.X[1] = X0[1] + inc[1]; st.X[2] = X0[2] + inc[2];
}

// FOV geometry shared by value / derivative evaluation
struct Fov {
  double t6p, t6m, t5p, t5m, s7, c7;
};
__device__ __forceinline__ void fov_trig(const Prob& pr, const double* X, Fov& f) {
  f.t6p = n_tan(X[6] + pr.hv); f.t6m = n_tan(X[6] - pr.hv);
  f.t5p = n_tan(X[5] + pr.hh); f.t5m = n_tan(X[5] - pr.hh);
  const double2 sc = n_sincos(X[7]); f.s7 = sc.x; f.c7 = sc.y;
}

// problem constants with this instance's cost weights (NMPC_TT.py:204-205; per instance for weight sweeps)
__device__ __forceinline__ Prob with_weights(const Prob& pr, double w1, double w2) { Prob q = pr; q.w1 = w1; q.w2 = w2; return q; }

// stage cost value (compact form of NMPC_TT.py:209-220)
__device__ __forceinline__ double stage_cost(const Prob& pr, const double* X, double xt, double yt) {
  Fov f; fov_trig(pr, X, f);
  const double z = X[2];
  const double ia = rcp(z * 0.5 * (f.t6p - f.t6m)), ib = rcp(z * 0.5 * (f.t5p - f.t5m));
  const double Dx = xt - X[0] - z * 0.5 * (f.t6p + f.t6m);
  const double Dy = yt - X[1] - z * 0.5 * (f.t5p + f.t5m);
  const double U = (f.c7 * Dx + f.s7 * Dy) * ia, V = (f.s7 * Dx - f.c7 * Dy) * ib;
  const double ex = X[0] - xt, ey = X[1] - yt;
  return pr.w1 * sqrt(ex * ex + ey * ey) + pr.w2 * (U * U + V * V - 1.0);
}

// stage cost with gradient gl[6] and packed Hessian Hl[21] over (x, y, z, X5, X6, X7)
__device__ __forceinline__ double stage_cost_d2(const Prob& pr, const double* X, double xt, double yt, double* gl, double* Hl) {
  Fov f; fov_trig(pr, X, f);
  const double z = X[2];
  const double d6p = 1.0 + f.t6p * f.t6p, d6m = 1.0 + f.t6m * f.t6m, d5p = 1.0 + f.t5p * f.t5p, d5m = 1.0 + f.t5m * f.t5m;
  const double e6p = 2.0 * f.t6p * d6p, e6m = 2.0 * f.t6m * d6m, e5p = 2.0 * f.t5p * d5p, e5m = 2.0 * f.t5m * d5m;
  const double al = 0.5 * (f.t6p - f.t6m), al1 = 0.5 * (d6p - d6m), al2 = 0.5 * (e6p - e6m);
  const double ga = 0.5 * (f.t6p + f.t6m), ga1 = 0.5 * (d6p + d6m), ga2 = 0.5 * (e6p + e6m);
  const double be = 0.5 * (f.t5p - f.t5m), be1 = 0.5 * (d5p - d5m), be2 = 0.5 * (e5p - e5m);
  const double ep = 0.5 * (f.t5p + f.t5m), ep1 = 0.5 * (d5p + d5m), ep2 = 0.5 * (e5p + e5m);
  const double a = z * al, b = z * be;
  const double Dx = xt - X[0] - z * ga, Dy = yt - X[1] - z * ep;
  const double s7 = f.s7, c7 = f.c7;
  const double Ph = c7 * Dx + s7 * Dy, Qh = s7 * Dx - c7 * Dy;
  const double ia = rcp(a), ib = rcp(b);
  const double U = Ph * ia, V = Qh * ib;
  // intermediates m = (Dx, Dy, a, b, X7)
  const double Um[5] = {c7 * ia, s7 * ia, -U * ia, 0.0, -Qh * ia};
  const double Vm[5] = {s7 * ib, -c7 * ib, 0.0, -V * ib, Ph * ib};
  double gm[5], Hm[5][5];
#pragma unroll
  for (int i = 0; i < 5; ++i) gm[i] = 2.0 * (U * Um[i] + V * Vm[i]);
#pragma unroll
  for (int i = 0; i < 5; ++i)
#pragma unroll
    for (int j = 0; j < 5; ++j) Hm[i][j] = 2.0 * (Um[i] * Um[j] + Vm[i] * Vm[j]);
  const double U2 = 2.0 * U, V2 = 2.0 * V, ia2 = ia * ia, ib2 = ib * ib;
  auto addsym = [&](int i, int j, double v) { Hm[i][j] += v; if (i != j) Hm[j][i] += v; };
  addsym(0, 2, U2 * (-c7 * ia2)); addsym(1, 2, U2 * (-s7 * ia2)); addsym(2, 2, U2 * (2.0 * U * ia2));
  addsym(0, 4, U2 * (-s7 * ia)); addsym(1, 4, U2 * (c7 * ia)); addsym(2, 4, U2 * (Qh * ia2)); addsym(4, 4, U2 * (-U));
  addsym(0, 3, V2 * (-s7 * ib2)); addsym(1, 3, V2 * (c7 * ib2)); addsym(3, 3, V2 * (2.0 * V * ib2));
  addsym(0, 4, V2 * (c7 * ib)); addsym(1, 4, V2 * (s7 * ib)); addsym(3, 4, V2 * (-Ph * ib2)); addsym(4, 4, V2 * (-V));
  // Jacobian of m w.r.t. v = (x, y, z, X5, X6, X7)
  const double Jm[5][6] = {{-1.0, 0.0, -ga, 0.0, -z * ga1, 0.0},
                           {0.0, -1.0, -ep, -z * ep1, 0.0, 0.0},
                           {0.0, 0.0, al, 0.0, z * al1, 0.0},
                           {0.0, 0.0, be, z * be1, 0.0, 0.0},
                           {0.0, 0.0, 0.0, 0.0, 0.0, 1.0}};
  double HJ[5][6];
#pragma unroll
  for (int i = 0; i < 5; ++i)
#pragma unroll
    for (int v = 0; v < 6; ++v) {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j < 5; ++j) acc += Hm[i][j] * Jm[j][v];
      HJ[i][v] = acc;
    }
  const double w2 = pr.w2;
#pragma unroll
  for (int v = 0; v < 6; ++v) {
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < 5; ++i) acc += gm[i] * Jm[i][v];
    gl[v] = w2 * acc;
  }
#pragma unroll
  for (int u = 0; u < 6; ++u)
#pragma unroll
    for (int v = 0; v <= u; ++v) {
      double acc = 0.0;
#pragma unroll
      for (int i = 0; i < 5; ++i) acc += Jm[i][u] * HJ[i][v];
      Hl[tri(u, v)] = w2 * acc;
    }
  // curvature of the intermediates themselves
  Hl[tri(4, 2)] += w2 * (gm[0] * (-ga1) + gm[2] * al1);          // (z, X6)
  Hl[tri(4, 4)] += w2 * (gm[0] * (-z * ga2) + gm[2] * (z * al2)); // (X6, X6)
  Hl[tri(3, 2)] += w2 * (gm[1] * (-ep1) + gm[3] * be1);          // (z, X5)
  Hl[tri(3, 3)] += w2 * (gm[1] * (-z * ep2) + gm[3] * (z * be2)); // (X5, X5)
  // distance term
  const double ex = X[0] - xt, ey = X[1] - yt;
  const double D = sqrt(ex * ex + ey * ey), iD = rcp(D);
  const double nx = ex * iD, ny = ey * iD, w1 = pr.w1;
  gl[0] += w1 * nx; gl[1] += w1 * ny;
  Hl[tri(0, 0)] += w1 * iD * (1.0 - nx * nx);
  Hl[tri(1, 0)] += w1 * iD * (-nx * ny);
  Hl[tri(1, 1)] += w1 * iD * (1.0 - ny * ny);
  return w1 * D + w2 * (U * U + V * V - 1.0);
}

// model 1: distance-only stage cost (MATLAB/Dynamic Obstacles/NMPC_TT.m:100-104), same output layout
__device__ __forceinline__ double stage_cost_dist(const double* X, double xt, double yt) {
  const double ex = X[0] - xt, ey = X[1] - yt;
  return sqrt(ex * ex + ey * ey);
}
__device__ __forceinline__ double stage_cost_dist_d2(const double* X, double xt, double yt, double* gl, double* Hl) {
#pragma unroll
  for (int v = 0; v < 6; ++v) gl[v] = 0.0;
#pragma unroll
  for (int e = 0; e < 21; ++e) Hl[e] = 0.0;
  const double ex = X[0] - xt, ey = X[1] - yt;
  const double D = sqrt(ex * ex + ey * ey), iD = rcp(D);
  const double nx = ex * iD, ny = ey * iD;
  gl[0] = nx; gl[1] = ny;
  Hl[tri(0, 0)] = iD * (1.0 - nx * nx); Hl[tri(1, 0)] = iD * (-nx * ny); Hl[tri(1, 1)] = iD * (1.0 - ny * ny);
  return D;
}

// Closed-loop shift of ONE instance (NMPC_TT.py:13-30, :399-402, :435): plant Euler step with the first input u0, target
// Euler step with (tv, tw), FOV centre of the new state and the tracking-error term.  st = [x(8); x_t, y_t, theta_t] in
// place.  Used by nmpc_step_kernel (one thread per instance) and by the fused epilogue of the IPM kernel (lane 0).
__device__ __forceinline__ void closed_loop_shift(double T, double hv, double hh, double* st, const double* u0, double tv, double tw,
                                                  double* fov, double* err) {
  double x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = st[i];
  double sth, cth, sps, cps;
  sincos(x[3], &sth, &cth); sincos(x[4], &sps, &cps);
  const double v = u0[0];
  x[0] += T * (v * cps * cth); x[1] += T * (v * sps * cth); x[2] += T * (v * sth);
#pragma unroll
  for (int i = 1; i < 6; ++i) x[i + 2] += T * u0[i];
#pragma unroll
  for (int i = 0; i < 8; ++i) st[i] = x[i];
  double* tg = st + NX;
  const double tx0 = tg[0], ty0 = tg[1];          // target of THIS step: the error pairs it with the NEXT FOV centre
  const double th = tg[2];
  tg[0] += T * tv * cos(th); tg[1] += T * tv * sin(th); tg[2] += T * tw;
  if (fov) {
    const double t6p = tan(x[6] + hv), t6m = tan(x[6] - hv), t5p = tan(x[5] + hh), t5m = tan(x[5] - hh);
    const double a_p = (x[2] * t6p - x[2] * t6m) / 2, b_p = (x[2] * t5p - x[2] * t5m) / 2;
    const double xe = x[0] + a_p + x[2] * t6m, ye = x[1] + b_p + x[2] * t5m;
    fov[0] = xe; fov[1] = ye;
    if (err) *err += sqrt((xe - tx0) * (xe - tx0) + (ye - ty0) * (ye - ty0));     // NMPC_TT.py:435
  }
}

// the same on the caller's p record of either model: model 1 holds [state(5); target(3)] (MATLAB/Dynamic Obstacles/shift1.m)
__device__ __forceinline__ void closed_loop_shift_model(int model, double T, double hv, double hh, double* p, const double* u0, double tv, double tw,
                                                        double* fov, double* err) {
  if (!model) { closed_loop_shift(T, hv, hh, p, u0, tv, tw, fov, err); return; }
  double st[NPAR], u6[NU] = {u0[0], u0[1], u0[2], 0.0, 0.0, 0.0};
#pragma unroll
  for (int i = 0; i < 5; ++i) st[i] = p[i];
  st[5] = 0.0; st[6] = 0.0; st[7] = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i) st[8 + i] = p[5 + i];
  closed_loop_shift(T, hv, hh, st, u6, tv, tw, fov, err);
#pragma unroll
  for (int i = 0; i < 5; ++i) p[i] = st[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) p[5 + i] = st[8 + i];
}

// 6x6 Cholesky on a packed lower triangle (in place).  Returns false when a pivot is not positive.
__device__ __forceinline__ bool chol6(double* L, double* inv_diag) {
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double d = L[tri(j, j)];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= L[tri(j, k)] * L[tri(j, k)];
    ok = ok && (d > 0.0);
    const double id = rsqrt(d);
    L[tri(j, j)] = d * id; inv_diag[j] = id;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      double s = L[tri(i, j)];
#pragma unroll
      for (int k = 0; k < j; ++k) s -= L[tri(i, k)] * L[tri(j, k)];
      L[tri(i, j)] = s * id;
    }
  }
  return ok;
}
__device__ __forceinline__ void chol6_solve(const double* L, const double* inv_diag, double* b) {
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double s = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) s -= L[tri(i, k)] * b[k];
    b[i] = s * inv_diag[i];
  }
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double s = b[i];
#pragma unroll
    for (int k = i + 1; k < 6; ++k) s -= L[tri(k, i)] * b[k];
    b[i] = s * inv_diag[i];
  }
}

}  // namespace nmpc
