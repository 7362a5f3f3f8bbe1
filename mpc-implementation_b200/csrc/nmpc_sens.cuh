// nmpc_sens.cuh -- solution sensitivities of converged solves (nmpc_sensitivity, nmpc_sensitivity_obstacles): dw*/dp,
// dw*/d(w1, w2) and dw*/d(cx, cy, r) of every obstacle.
//
// At the final iterate of a solve that kept its barrier data (NMPC_KEEP_BARRIER: Sigma_x, Sigma_g from ph_output) the
// sensitivity is the implicit-function derivative of the barrier KKT system at delta_w = 0 (DESIGN.md section 1):
//     K dw/dth = -(grad2_{w th} L + J^T Sigma_g J_th),      K = grad2_{ww} L + Sigma_x + J^T Sigma_g J,
// the IPM's Newton matrix with other right-hand sides.  One warp per instance builds it as the stage LQ problem ph_derivs
// builds, in the unscaled units of lam_x / lam_g (df = dc = 1, no mu or delta_w parts), factors it once with riccati_factor
// and runs one forward sweep per column:
//   state columns    dx_0 = e_i and no linear terms (stage 0's rows and cost do not depend on w)
//   target columns   linear terms -d2 l_k / dX d(x, y) of stages 1..N-1 (the cost depends on (x - x_t, y - y_t) only), dx_0 = 0;
//                    exactly 0 with a per-stage target trajectory, as lam_p; theta_t never enters the NLP: exactly 0
//   weight columns   linear terms grad_X dist_k and grad_X fov_k of each stage cost (model 0)
//   obstacle columns linear terms y d(grad_X g)/dth + J^T Sigma_g dg/dth of the obstacle's row g = r - ||(x, y) - c|| on stages
//                    1..N (the terminal stage included: its rows depend on w), dx_0 = 0
// Each family runs only when its output is given; all share the one factorisation.
// A non-positive pivot means the reduced Hessian is not positive definite at delta_w = 0 and the sensitivity is undefined:
// NaN columns and sens_status 1.
#pragma once
#include "nmpc_solve.cuh"

namespace nmpc {

#define smem (smem_all + (threadIdx.x >> 5) * L::TOTAL)
#define LV(e) smem[L::LV0 + (e) * L::S + lane]
#define LQ(e) smem[L::LQ0 + (e) * L::S + lane]
#define PAR(i) smem[L::PAR0 + (i)]

template <class L>
__device__ __noinline__ void sens_instance(const SolveArgs& A, double* ric, int b, int lane) {
  const Prob& pr = A.pr; constexpr int N = L::N, S = L::S, R = L::R, NUA = L::NUA, NPA = L::NPA, NXP = NPA - 3;
  constexpr int nw = NUA * N;
  const double T = pr.T;
  const bool act = lane <= N, hasu = lane < N;
  ph_load<L>(A, b, lane, 0);            // p, weights, obstacles; x0 is the solution here: LV_U = w*
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
  if (hasu && lane >= 1) cost_d2<L>(A, st.X, lane, gl, Hl);      // stage 0 is constant in w
  // Lagrangian gradient seed of the adjoint (gl + G^T y) and state Hessian (cost + G^T Sigma_g G + y-curvature of the rows)
  double a[8], q66[21], qtt = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 0.0;
#pragma unroll
  for (int v = 0; v < 6; ++v) a[cost_state(v)] = gl[v];
#pragma unroll
  for (int e = 0; e < 21; ++e) q66[e] = Hl[e];
  if (act) {
    const double* sg = A.sig_g + (size_t)b * R * S + lane * R;
    const double* yg = A.lam_g + (size_t)b * R * S + lane * R;
#pragma unroll
    for (int r = 0; r < L::NB; ++r) {
      const int si = box_state(r);
      a[si] += yg[r];
      if (si == 3) qtt += sg[r];
      else { const int c = si < 3 ? si : si - 2; q66[tri(c, c)] += sg[r]; }
    }
#pragma unroll 1
    for (int jn = 0; jn < L::NOBS; ++jn) {
      double nx, ny, iD;
      obs_value<L>(st.X, jn, nx, ny, iD);
      const double w = sg[L::NB + jn], y = yg[L::NB + jn], cur = -y * iD;      // y * d2h,  d2h = -(I - n n^T)/D
      q66[0] += w * nx * nx + cur * (1.0 - nx * nx);
      q66[1] += w * nx * ny - cur * nx * ny;
      q66[2] += w * ny * ny + cur * (1.0 - ny * ny);
      a[0] -= y * nx; a[1] -= y * ny;
    }
  }
  double lamn[8];
  adjoint<L::SW>(a, dy, act, lane, lamn);
  if (act) {
    // ph_derivs' curvature of T*v*d(theta, psi) weighted by the next-stage adjoint
    double svt = 0.0, svp = 0.0, q33 = 0.0, q34 = 0.0, q44 = 0.0;
    if (hasu) {
      const double L0 = T * lamn[0], L1 = T * lamn[1], L2 = T * lamn[2], v = u[0];
      const double cc = st.cps * st.cth, sc = st.sps * st.cth, cs = st.cps * st.sth, ss = st.sps * st.sth;
      q33 = -v * (L0 * cc + L1 * sc + L2 * st.sth);
      q44 = -v * (L0 * cc + L1 * sc);
      q34 = v * (L0 * ss - L1 * cs);
      svt = -L0 * cs - L1 * ss + L2 * st.cth;
      svp = -L0 * sc + L1 * cc;
    }
#pragma unroll
    for (int e = 0; e < 21; ++e) LQ(LQ_Q + e) = q66[e];
    LQ(LQ_Q + 21) = qtt + q33; LQ(LQ_Q + 22) = q34; LQ(LQ_Q + 23) = q44;
    LQ(LQ_SV + 0) = svt; LQ(LQ_SV + 1) = svp;
#pragma unroll
    for (int i = 0; i < 6; ++i) {      // absent controls (model 1) keep the unit diagonal
      LQ(LQ_RD + i) = (hasu && i < NUA) ? A.sig_x[(size_t)b * nw + NUA * lane + i] : 1.0;
      LQ(LQ_RB + i) = 0.0;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) LQ(LQ_QA + i) = 0.0;
    LQ(LQ_DD + 0) = st.cps * st.cth; LQ(LQ_DD + 1) = st.sps * st.cth; LQ(LQ_DD + 2) = st.sth;
    LQ(LQ_EE + 0) = dy.e03; LQ(LQ_EE + 1) = dy.e13; LQ(LQ_EE + 2) = dy.e23; LQ(LQ_EE + 3) = dy.e04; LQ(LQ_EE + 4) = dy.e14;
    LQ(LQ_ZERO) = 0.0;
    if (!L::FOLD) {
#pragma unroll
      for (int e = LQ_NFOLD; e < LQ_N; ++e) LQ(e) = 0.0;
    }
  }
  __syncwarp();
  // mu = delta_w = 0: the factor's own right-hand side is zero, so its kappa is exactly 0
  const bool ok = riccati_factor<L>(T, ric, A.ricmap, 0.0, 0.0, lane);
  __syncwarp();
  if (lane == 0 && A.sens_status) A.sens_status[b] = ok ? 0 : 1;
  // column j: p for j < NPA, (w1, w2) for j < NPA + 2, then (cx, cy, r) of each obstacle; a family runs when its output is given
  constexpr int NO = 3 * L::NOBS, JO = NPA + 2;
  const double2 tg = stage_target<L>(A, lane);
#pragma unroll 1
  for (int j = 0; j < JO + NO; ++j) {
    if (!(j < NPA ? A.dx_dp : (j < JO ? (L::MODEL ? nullptr : A.dx_dw) : A.dx_do))) continue;
    const bool zero = j == NPA - 1 || (j >= NXP && j < NPA && A.tgt != nullptr);
    if (ok && !zero) {
      if (j < NXP) {
        if (lane < 8) smem[L::LV0 + (LV_DX + lane) * S] = lane == j ? 1.0 : 0.0;
        __syncwarp();
        riccati_forward<L, true>(T, ric, false, lane, L::LV0 + LV_DX * S, L::LV0 + LV_DU * S);
      } else {
        double q[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) q[i] = 0.0;
        if (hasu && lane >= 1 && j < JO) {
          if (j < NPA) {
            const int c = j - NXP;      // d/dx_t = -d/dx, d/dy_t = -d/dy
#pragma unroll
            for (int v = 0; v < 6; ++v) q[cost_state(v)] = -Hl[tri(v, c)];
          } else {
            double g1[6], H1[21];
            stage_cost_d2(with_weights(pr, j == NPA ? 1.0 : 0.0, j == NPA ? 0.0 : 1.0), st.X, tg.x, tg.y, g1, H1);
#pragma unroll
            for (int v = 0; v < 6; ++v) q[cost_state(v)] = g1[v];
          }
        }
        if (act && lane >= 1 && j >= JO) {      // row g = r - D of obstacle jn on stages 1..N (the terminal one included)
          const int jn = (j - JO) / 3, t = j - JO - 3 * jn;
          double nx, ny, iD;
          obs_value<L>(st.X, jn, nx, ny, iD);
          const size_t ro = (size_t)b * R * S + lane * R + L::NB + jn;
          const double w = A.sig_g[ro], y = A.lam_g[ro];
          if (t == 2) { q[0] = -w * nx; q[1] = -w * ny; }     // J^T Sigma_g dg/dr = -Sigma_g n
          else {      // y d(-n)/dc_t = y (e_t - n_t n) / D,  J^T Sigma_g dg/dc_t = -Sigma_g n_t n
            const double m = t ? ny : nx, c = y * iD;
            q[0] = c * ((t ? 0.0 : 1.0) - m * nx) - w * m * nx;
            q[1] = c * ((t ? 1.0 : 0.0) - m * ny) - w * m * ny;
          }
        }
        if (act) {
#pragma unroll
          for (int i = 0; i < 8; ++i) smem[L::soc(SOC_Q2) + i * S + lane] = q[i];
        }
        __syncwarp();
        riccati_resolve<L>(T, L::soc(SOC_Q2), ric, 0.0, lane);
        riccati_forward<L>(T, ric, true, lane, L::LV0 + LV_DX * S, L::LV0 + LV_DU * S);
      }
    }
    if (hasu) {
      double* col = j < NPA ? A.dx_dp + (size_t)b * nw * NPA + j
                            : (j < JO ? A.dx_dw + (size_t)b * nw * 2 + (j - NPA) : A.dx_do + (size_t)b * nw * NO + (j - JO));
      const int ld = j < NPA ? NPA : (j < JO ? 2 : NO);
#pragma unroll
      for (int i = 0; i < NUA; ++i) col[(size_t)(NUA * lane + i) * ld] = !ok ? CUDART_NAN : (zero ? 0.0 : LV(LV_DU + i));
    }
    __syncwarp();
  }
}

// one warp per block, each on its own Lay::TOTAL slice of dynamic shared memory and Riccati scratch slot
template <int N_, int NOBS_, int MODEL_>
__global__ void __launch_bounds__(32) nmpc_sens_kernel(const __grid_constant__ SolveArgs A) {
  using L = Lay<N_, NOBS_, MODEL_>;
  const int lane = threadIdx.x & 31;
  double* ric = A.ric + (size_t)blockIdx.x * A.ric_stride;
  for (int b = blockIdx.x; b < A.B; b += gridDim.x) { sens_instance<L>(A, ric, b, lane); __syncwarp(); }
}

#undef smem
#undef LV
#undef LQ
#undef PAR

}  // namespace nmpc
