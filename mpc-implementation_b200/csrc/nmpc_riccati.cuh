// nmpc_riccati.cuh -- warp-parallel Riccati factorisation / solves of the stage-structured Newton system.
//
// Per stage k (backward) the 15 x 15 symmetric "stage KKT matrix" in the ordering (u (6), x (8), rhs (1)) is
//     H = Z^T P+ Z + [R S; S^T Q],   h = Z^T p+ + [r; q],          Z = [B_k | A_k]  (8 x 14),
// and eliminating the six control pivots by a right-looking Cholesky leaves P_k (8 x 8) and p_k in the trailing
// block, L (6 x 6), L^-1 Psi (6 x 8) and L^-1 psi in the pivot columns.  All 32 lanes work: every lane OWNS up
// to four entries of the packed lower triangle (registers), operands are exchanged through a shared-memory
// staging area, loops are rolled so the stage body is small (the first version was 1900 unrolled instructions with
// 9 of 32 lanes active and stalled on instruction fetch).
// "Inertia correct" (IPOPT)  <=>  all six pivots of every stage positive.
//
// All workspace accesses go through the `extern __shared__` array with compile-time offsets (Lay<N, NOBS>), so
// they compile to LDS/STS with immediates (passing shared pointers across __noinline__ calls made them generic
// LD/ST + R2UR: 41 % of this function's instructions in v2).
#pragma once
#include "nmpc_device.cuh"

namespace nmpc {

// The block holds Lay::WPB warps, each solving its own instance in its own Lay::TOTAL slice of dynamic shared
// memory; `smem` is the executing warp's slice (every function that uses it has the layout type L in scope).
extern __shared__ double smem_all[];
#define smem (smem_all + (threadIdx.x >> 5) * L::TOTAL)

// staging area layout (doubles, relative to Lay::STG0); every base is even (16-byte aligned)
constexpr int SG_PP = 0;      // [9][9]  rows 0..7 = P+ (symmetric), row 8 = p+
constexpr int SG_Y = 82;      // [3][8]  Y_c = P+ z_c of the three special columns c = 0, 9, 10
constexpr int SG_H = 106;     // [120]   packed lower triangle of the 15 x 15 stage matrix [H | h]
constexpr int SG_W = 226;     // [9][6]  W = [Psi | psi]^T L^-T  (rows: 8 states + rhs)
constexpr int SG_X = 280;     // [1]     where the lanes without a second trailing entry store theirs
static_assert(SG_X + 1 <= STG_N, "staging area too small");
// lane 0 owns two corrected entries of the stage matrix (e = 0 and e = 64); this lane computes the second one for it
constexpr int RIC_CB_LANE = 24;
static_assert(RIC_L % 2 == 0 && RIC_N % 2 == 0, "riccati_factor stores L with 16-byte stores");

// state-Hessian entry Q_k[i][j] (+ delta_w part), used for the terminal stage only
template <class L>
__device__ __forceinline__ double q_entry(int k, int i, int j, double dw) {
  const int qi = q_index(i, j);
  double v = qi >= 0 ? smem[L::LQ0 + (LQ_Q + qi) * L::S + k] : 0.0;
  if (!L::FOLD) {
    if (i < 2 && j < 2) v += dw * smem[L::LQ0 + (LQ_NN + i + j) * L::S + k];
    else if (i == j && i != 4) v += dw * smem[L::LQ0 + (LQ_DG + ((i == 2) ? 0 : (i == 3 ? 1 : i - 3))) * L::S + k];
  }
  return v;
}

// ---- per-lane ownership maps of the factorisation -------------------------------------------------------------
// They depend on the lane and the layout only, so they are computed once per (N, n_obs) instantiation by
// ric_map_kernel (at nmpc_create) into a global table of RIC_MAP_WORDS x 32 words, [word][lane], and loaded by
// riccati_factor (18 coalesced L1-resident loads instead of ~800 instructions of index arithmetic per call).
// All entries are shared-memory indices relative to the warp's slice, packed two per word:
//   w0..1 o0[4]   w2..3 o1[4]   w4..5 o2[4]   w6..7 ymain[4]   w8 zy0|zy1   w9 zy2|zc0   w10 zc1|zc2   w11 cy|th0
//   w12 th1|twa0   w13 twb0|twa1   w14 twb1|tp0[0]   w15 tp1[0]|tp0[1]   w16 tp1[1]|(unused)
//   w17 codes = cmain code (2 bits: 0, 1, T, T^2) x 4 | c3 flag x 4 << 8 | correction A x 4 << 12 | correction B << 16
constexpr int RIC_MAP_WORDS = 18;

template <class L>
__device__ void ric_map_build(int lane, unsigned* __restrict__ out /* [RIC_MAP_WORDS][32] */) {
  constexpr int S = L::S;
  constexpr int PP = L::STG0 + SG_PP, YS = L::STG0 + SG_Y, HS = L::STG0 + SG_H, WS = L::STG0 + SG_W;
  constexpr int LQ0 = L::LQ0;
  // Column c of Z = [B | A] is T e_{c+2} (c = 1..5) or e_{c-6} (c >= 6), plus stage-dependent entries in rows 0..2
  // for the "special" columns c = 0 (v: no unit part), 9 (theta), 10 (psi).
  auto spec = [](int c) { return c == 0 || c == 9 || c == 10; };
  auto sid = [](int c) { return c >= 6 ? c - 6 : c + 2; };                 // row of the unit entry (c >= 1)
  auto spj = [](int c) { return c == 0 ? 0 : c - 8; };                     // special column -> 0, 1, 2
  // rows 0..2 of special column j, read at stage k from LQ0 + zoff + k: T * d (j = 0; riccati_factor applies the T),
  // the first / last two entries of T E (j = 1 / 2), and 0 for Z[2][10]
  auto zoff = [](int j, int s) { return LQ0 + S * (j == 0 ? LQ_DD + s : (j == 1 ? LQ_EE + s : (s < 2 ? LQ_EE + 3 + s : LQ_ZERO))); };
  auto row_of = [](int e) { int a = 0; while ((a + 1) * (a + 2) / 2 <= e) ++a; return a; };
  // ---- BUILDING the stage matrix: entry e = lane + 32 m of the packed lower triangle,
  //      ent = cmain * smem[ymain] + lq[o0] + mu * lq[o1] + dw * (lq[o2] + c3)
  int o0[4], o1[4], o2[4], ymain[4]; unsigned codes = 0;
  for (int m = 0; m < 4; ++m) {
    const int e = lane + 32 * m;
    const int a = row_of(e), b = e - a * (a + 1) / 2;
    const bool valid = e < 119;                       // e == 119 is (14,14): not needed
    int p0 = LQ_ZERO, p1 = LQ_ZERO, p2 = LQ_ZERO, cc = 0;
    int ym = PP, cm = 0;                              // cm: 0 -> 0.0, 1 -> 1.0, 2 -> T, 3 -> T*T
    if (valid) {
      if (a < 6) { if (a == b) { p0 = LQ_RD + a; cc = 1; } }
      else if (a < 14) {
        if (b < 6) { if (b == 0 && a == 9) p0 = LQ_SV + 0; else if (b == 0 && a == 10) p0 = LQ_SV + 1; }
        else {
          const int i = a - 6, j = b - 6, qi = q_index(i, j);
          if (qi >= 0) p0 = LQ_Q + qi;
          if (!L::FOLD) {
            if (i < 2 && j < 2) p2 = LQ_NN + i + j;
            else if (i == j && i != 4) p2 = LQ_DG + ((i == 2) ? 0 : (i == 3 ? 1 : i - 3));
          }
        }
      } else {
        if (b < 6) p1 = LQ_RB + b;
        else { p0 = LQ_QA + (b - 6); if (!L::FOLD) { p1 = LQ_QB + (b - 6); p2 = LQ_QD + (b - 6); } }
      }
      // H[a][b] = z_a^T P+ z_b,  h[b] = z_b^T p+ : the part that is ONE scaled entry of P+ / p+ / Y_special
      const int ca = (a >= 1 && a < 6) ? 1 : 0, cb = (b >= 1 && b < 6) ? 1 : 0;    // powers of T
      if (a == 14) {
        if (b != 0) { ym = PP + 72 + sid(b); cm = 1 + cb; }                  // b == 0: correction only
      } else if (!spec(a) && !spec(b)) { ym = PP + sid(a) * 9 + sid(b); cm = 1 + ca + cb; }
      else if (spec(b) && !spec(a)) { ym = YS + spj(b) * 8 + sid(a); cm = 1 + ca; }
      else if (spec(a) && !spec(b)) { ym = YS + spj(a) * 8 + sid(b); cm = 1 + cb; }
      else if (a != 0) { ym = YS + spj(b) * 8 + sid(a); cm = 1; }            // both special: unit part of z_a (none for a == 0)
    }
    o0[m] = LQ0 + p0 * S; o1[m] = LQ0 + p1 * S; o2[m] = LQ0 + p2 * S;
    ymain[m] = ym; codes |= (unsigned)cm << (2 * m); codes |= (unsigned)cc << (8 + m);
  }
  // ---- Y_j = P+ z_j, j = lane / 8 (stored by lanes 0..23)
  const int yj = lane < 24 ? lane >> 3 : 0;
  // ---- the nine entries whose z_a AND z_b (or p+) are special get  sum_s Z[s][za] * Yv[s]  on top, added by the lane
  //      that builds the entry (bit m of correction A); lane 0 builds two of them and takes the second (e = 64, m = 2:
  //      correction B) from lane RIC_CB_LANE, which builds none
  int zc = 0, cy = PP;
  for (int q = 0; q < 9; ++q) {
    const int ca_[9] = {0, 9, 10, 9, 10, 10, 14, 14, 14}, cb_[9] = {0, 0, 0, 9, 9, 10, 0, 9, 10};
    const int a = ca_[q], b = cb_[q], e = a * (a + 1) / 2 + b;
    const bool second = e == 64;
    if ((e & 31) == lane && !second) codes |= 1u << (12 + e / 32);
    if (lane == 0 && second) codes |= 1u << 16;
    if (second ? lane == RIC_CB_LANE : (e & 31) == lane) {
      zc = spj(a == 14 ? b : a);
      cy = a == 14 ? PP + 72 : YS + spj(b) * 8;
    }
  }
  // ---- TRAILING update: t = lane + 32 r over the packed lower triangle of the 9 x 9 block (t >= 44: no entry, the
  //      lane computes H[6][6] - W_0 . W_0 again and stores it to SG_X)
  int th[2], twa[2], twb[2], tp0[2], tp1[2];
  for (int r = 0; r < 2; ++r) {
    const int t = lane + 32 * r;
    const int a = row_of(t), b = t - a * (a + 1) / 2;
    const bool valid = t < 44;                        // t == 44 is (rhs, rhs)
    th[r] = HS + (valid ? (a + 6) * (a + 7) / 2 + (b + 6) : 27);
    twa[r] = WS + (valid ? a : 0) * 6; twb[r] = WS + (valid ? b : 0) * 6;
    tp0[r] = !valid ? L::STG0 + SG_X : (a == 8 ? PP + 72 + b : PP + a * 9 + b);
    tp1[r] = !valid ? L::STG0 + SG_X : (a == 8 ? PP + 72 + b : PP + b * 9 + a);
  }
  auto pk = [](int lo, int hi) { return (unsigned)lo | ((unsigned)hi << 16); };
  unsigned w[RIC_MAP_WORDS] = {pk(o0[0], o0[1]), pk(o0[2], o0[3]), pk(o1[0], o1[1]), pk(o1[2], o1[3]), pk(o2[0], o2[1]), pk(o2[2], o2[3]),
                               pk(ymain[0], ymain[1]), pk(ymain[2], ymain[3]), pk(zoff(yj, 0), zoff(yj, 1)), pk(zoff(yj, 2), zoff(zc, 0)),
                               pk(zoff(zc, 1), zoff(zc, 2)), pk(cy, th[0]), pk(th[1], twa[0]), pk(twb[0], twa[1]), pk(twb[1], tp0[0]),
                               pk(tp1[0], tp0[1]), pk(tp1[1], 0), codes};
  for (int i = 0; i < RIC_MAP_WORDS; ++i) out[i * 32 + lane] = w[i];
}
template <class L>
__global__ void ric_map_kernel(unsigned* out) { ric_map_build<L>(threadIdx.x & 31, out); }

template <class L>
__device__ __noinline__ bool riccati_factor(double T, double* __restrict__ ric, const unsigned* __restrict__ map, double mu, double dw, int lane) {
  constexpr int S = L::S, N = L::N;
  constexpr int PP = L::STG0 + SG_PP, YS = L::STG0 + SG_Y, HS = L::STG0 + SG_H, WS = L::STG0 + SG_W;
  constexpr int LQ0 = L::LQ0;
  unsigned w[RIC_MAP_WORDS];
#pragma unroll
  for (int i = 0; i < RIC_MAP_WORDS; ++i) w[i] = __ldg(map + i * 32 + lane);
  auto lo16 = [](unsigned v) { return (int)(v & 0xffffu); };
  auto hi16 = [](unsigned v) { return (int)(v >> 16); };
  const int o0[4] = {lo16(w[0]), hi16(w[0]), lo16(w[1]), hi16(w[1])}, o1[4] = {lo16(w[2]), hi16(w[2]), lo16(w[3]), hi16(w[3])};
  const int o2[4] = {lo16(w[4]), hi16(w[4]), lo16(w[5]), hi16(w[5])}, ymain[4] = {lo16(w[6]), hi16(w[6]), lo16(w[7]), hi16(w[7])};
  const int zy[3] = {lo16(w[8]), hi16(w[8]), lo16(w[9])}, zc[3] = {hi16(w[9]), lo16(w[10]), hi16(w[10])};
  const int cy = lo16(w[11]);
  const int th[2] = {hi16(w[11]), lo16(w[12])};
  const int twa[2] = {hi16(w[12]), hi16(w[13])}, twb[2] = {lo16(w[13]), lo16(w[14])};
  const int tp0[2] = {hi16(w[14]), hi16(w[15])}, tp1[2] = {lo16(w[15]), lo16(w[16])};
  const unsigned codes = w[17];
  double c3[4], cmain[4];
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const unsigned cm = (codes >> (2 * m)) & 3u;
    cmain[m] = cm == 0 ? 0.0 : (cm == 1 ? 1.0 : (cm == 2 ? T : T * T));
    c3[m] = ((codes >> (8 + m)) & 1u) ? 1.0 : 0.0;
  }
  // Z entries of column 0 are T * d; the others are read as they are (x 1.0 is exact)
  const double fy = zy[0] == LQ0 + LQ_DD * S ? T : 1.0, fc = zc[0] == LQ0 + LQ_DD * S ? T : 1.0;
  const int yi = lane & 7, yj = lane < 24 ? lane >> 3 : 0;
  // lane c < 9 owns row c of W and column c of K; lanes 9..31 compute row 8 again and store the same values to the same
  // addresses as lane 8, so that no store needs a branch
  const int wc = lane < 9 ? lane : 8, wr = HS + (wc + 6) * (wc + 7) / 2;
  // ---- terminal stage: P_N = Q_N, p_N = q_N
#pragma unroll 1
  for (int o = lane; o < 72; o += 32) {
    const int i = o >> 3, j = o & 7;
    smem[PP + i * 9 + j] = i < 8 ? q_entry<L>(N, i, j, dw)
                                 : (L::FOLD ? smem[LQ0 + (LQ_QA + j) * S + N]
                                            : smem[LQ0 + (LQ_QA + j) * S + N] + mu * smem[LQ0 + (LQ_QB + j) * S + N] + dw * smem[LQ0 + (LQ_QD + j) * S + N]);
  }
  __syncwarp();
  // Per stage: Y -> sync -> [H | h] -> sync -> Cholesky, W -> sync -> trailing update, K, L -> sync.  Every value is
  // computed by the same operations in the same order as when Z, the nine corrections and L were staged through
  // shared memory with a sync each; the intrinsics pin the contractions that staging used to force.
#pragma unroll 1
  for (int k = N - 1; k >= 0; --k) {
    double zyv[3], zcv[3];
#pragma unroll
    for (int s = 0; s < 3; ++s) { zyv[s] = __dmul_rn(fy, smem[zy[s] + k]); zcv[s] = __dmul_rn(fc, smem[zc[s] + k]); }
    // Y_c = P+ z_c for the special columns c = 0, 9, 10 (lanes 0..23)
    {
      double acc = __fma_rn(zyv[2], smem[PP + yi * 9 + 2], __fma_rn(zyv[0], smem[PP + yi * 9], __dmul_rn(zyv[1], smem[PP + yi * 9 + 1])));
      if (yj > 0) acc = __dadd_rn(acc, smem[PP + yi * 9 + 2 + yj]);
      if (lane < 24) smem[YS + lane] = acc;
    }
    __syncwarp();
    // [H | h] -> staging, with the corrections of the nine entries whose z_a and z_b (or p+) are both special
    const double ca = __fma_rn(zcv[2], smem[cy + 2], __fma_rn(zcv[0], smem[cy], __dmul_rn(zcv[1], smem[cy + 1])));
    const double cb = __shfl_sync(FULL, ca, RIC_CB_LANE);
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      double v = cmain[m] * smem[ymain[m]] + smem[o0[m] + k] + mu * smem[o1[m] + k] + dw * (smem[o2[m] + k] + c3[m]);
      if ((codes >> (12 + m)) & 1u) v = __dadd_rn(v, ca);
      if (m == 2 && ((codes >> 16) & 1u)) v = __dadd_rn(v, cb);
      if (m < 3 || lane < 24) smem[HS + lane + 32 * m] = v;
    }
    __syncwarp();
    // Cholesky of the 6 x 6 control block, redundantly in every lane's registers (uniform inertia verdict)
    double Lf[21], idg[6];
#pragma unroll
    for (int e = 0; e < 21; ++e) Lf[e] = smem[HS + e];
    if (!chol6(Lf, idg)) return false;
    // row wc of W = [Psi | psi]^T L^-T
    double wv[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      double s_ = smem[wr + j];
#pragma unroll
      for (int m = 0; m < j; ++m) s_ -= wv[m] * Lf[tri(j, m)];
      wv[j] = s_ * idg[j];
      smem[WS + wc * 6 + j] = wv[j];
    }
    __syncwarp();
    // trailing block -> P_k, p_k for the next stage
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      double acc = smem[th[r]];
#pragma unroll
      for (int j = 0; j < 6; ++j) acc -= smem[twa[r] + j] * smem[twb[r] + j];
      smem[tp0[r]] = acc; smem[tp1[r]] = acc;
    }
    // column wc of K = L^-T W^T, and L with 1/diag for the SOC re-solves (every lane holds the same L and stores it):
    // read only after the recursion, so they are computed here, next to the trailing update, and not at all for the
    // stages of a failed factorisation
    double* rk = ric + k * RIC_N;
#pragma unroll
    for (int i = 5; i >= 0; --i) {
      double s_ = wv[i];
#pragma unroll
      for (int m = i + 1; m < 6; ++m) s_ -= Lf[tri(m, i)] * wv[m];
      wv[i] = s_ * idg[i];
    }
#pragma unroll
    for (int r = 0; r < 6; ++r) rk[RIC_K + r * 9 + wc] = wv[r];
    double2* dl = reinterpret_cast<double2*>(rk + RIC_L);
#pragma unroll
    for (int e = 0; e < 10; ++e) dl[e] = make_double2(Lf[2 * e], Lf[2 * e + 1]);
    dl[10] = make_double2(Lf[20], idg[0]); dl[11] = make_double2(idg[1], idg[2]); dl[12] = make_double2(idg[3], idg[4]);
    rk[RIC_L + 26] = idg[5];
    __syncwarp();
  }
  return true;
}

// Forward sweep: du_k = -K_k dx_k - kappa_k, dx_{k+1} = A_k dx_k + B_k du_k.  Lane r < 6 computes row r of du
// from its row of [K | kappa] (prefetched one stage ahead from the L2-resident scratch); dx is replicated.
// Lane k keeps its own stage's dx, du and writes them to the shared-memory entries dx0 / du0 (offsets, [.][S]).
// X0 (the sensitivity kernel, nmpc_sens.cuh): the sweep starts from the dx_0 the caller has put in the stage-0 entries of dx0
// instead of from 0.
template <class L, bool X0 = false>
__device__ __noinline__ void riccati_forward(double T, const double* ric, bool soc, int lane, int dx0, int du0) {
  constexpr int S = L::S, N = L::N, LQ0 = L::LQ0;
  const int r = lane < 6 ? lane : 5;
  double dx[8], mydx[8], mydu[6];
#pragma unroll
  for (int i = 0; i < 8; ++i) { dx[i] = X0 ? smem[dx0 + i * S] : 0.0; mydx[i] = 0.0; }
#pragma unroll
  for (int i = 0; i < 6; ++i) mydu[i] = 0.0;
  double row[9];
  auto load_row = [&](int k) {
    const double* rk = ric + k * RIC_N;
#pragma unroll
    for (int i = 0; i < 8; ++i) row[i] = __ldcg(rk + RIC_K + r * 9 + i);   // written by this kernel: never the .nc path
    row[8] = soc ? __ldcg(rk + RIC_K2 + r) : __ldcg(rk + RIC_K + r * 9 + 8);
  };
  load_row(0);
#pragma unroll 1
  for (int k = 0; k < N; ++k) {
    double acc = row[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += row[i] * dx[i];
    if (k + 1 < N) load_row(k + 1);
    double du[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) du[i] = -__shfl_sync(FULL, acc, i);
    if (lane == k) {
#pragma unroll
      for (int i = 0; i < 8; ++i) mydx[i] = dx[i];
#pragma unroll
      for (int i = 0; i < 6; ++i) mydu[i] = du[i];
    }
    const double d0 = smem[LQ0 + (LQ_DD + 0) * S + k], d1 = smem[LQ0 + (LQ_DD + 1) * S + k], d2 = smem[LQ0 + (LQ_DD + 2) * S + k];
    const double e03 = smem[LQ0 + (LQ_EE + 0) * S + k], e13 = smem[LQ0 + (LQ_EE + 1) * S + k], e23 = smem[LQ0 + (LQ_EE + 2) * S + k];
    const double e04 = smem[LQ0 + (LQ_EE + 3) * S + k], e14 = smem[LQ0 + (LQ_EE + 4) * S + k];
    const double tv = T * du[0];
    dx[0] += e03 * dx[3] + e04 * dx[4] + tv * d0;
    dx[1] += e13 * dx[3] + e14 * dx[4] + tv * d1;
    dx[2] += e23 * dx[3] + tv * d2;
#pragma unroll
    for (int i = 1; i < 6; ++i) dx[i + 2] += T * du[i];
  }
  if (lane == N) {
#pragma unroll
    for (int i = 0; i < 8; ++i) mydx[i] = dx[i];
  }
  if (lane <= N) {
#pragma unroll
    for (int i = 0; i < 8; ++i) smem[dx0 + i * S + lane] = mydx[i];
#pragma unroll
    for (int i = 0; i < 6; ++i) smem[du0 + i * S + lane] = mydu[i];
  }
  __syncwarp();
}

// Backward sweep for a new state gradient q' (shared-memory entries q20, [8][S]) with the stored factors
// (second-order-correction right-hand sides).
template <class L>
__device__ __noinline__ void riccati_resolve(double T, int q20, double* ric, double mu, int lane) {
  constexpr int S = L::S, N = L::N, LQ0 = L::LQ0;
  double p[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) p[i] = smem[q20 + i * S + N];
#pragma unroll 1
  for (int k = N - 1; k >= 0; --k) {
    double* rk = ric + k * RIC_N;
    const double d0 = smem[LQ0 + (LQ_DD + 0) * S + k], d1 = smem[LQ0 + (LQ_DD + 1) * S + k], d2 = smem[LQ0 + (LQ_DD + 2) * S + k];
    const double e03 = smem[LQ0 + (LQ_EE + 0) * S + k], e13 = smem[LQ0 + (LQ_EE + 1) * S + k], e23 = smem[LQ0 + (LQ_EE + 2) * S + k];
    const double e04 = smem[LQ0 + (LQ_EE + 3) * S + k], e14 = smem[LQ0 + (LQ_EE + 4) * S + k];
    double psi[6], kap[6];
    psi[0] = mu * smem[LQ0 + (LQ_RB + 0) * S + k] + T * (d0 * p[0] + d1 * p[1] + d2 * p[2]);
#pragma unroll
    for (int r = 1; r < 6; ++r) psi[r] = mu * smem[LQ0 + (LQ_RB + r) * S + k] + T * p[r + 2];
    double Lf[21], idg[6];
#pragma unroll
    for (int e = 0; e < 21; ++e) Lf[e] = __ldcg(rk + RIC_L + e);
#pragma unroll
    for (int r = 0; r < 6; ++r) { idg[r] = __ldcg(rk + RIC_L + 21 + r); kap[r] = psi[r]; }
    chol6_solve(Lf, idg, kap);
    double pn[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) pn[i] = smem[q20 + i * S + k] + p[i];
    pn[3] += e03 * p[0] + e13 * p[1] + e23 * p[2];
    pn[4] += e04 * p[0] + e14 * p[1];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      double acc = 0.0;
#pragma unroll
      for (int r = 0; r < 6; ++r) acc += __ldcg(rk + RIC_K + r * 9 + i) * psi[r];
      pn[i] -= acc;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) p[i] = pn[i];
#pragma unroll
    for (int r = 0; r < 6; ++r) if (lane == r) rk[RIC_K2 + r] = kap[r];
  }
  __syncwarp();
}

}  // namespace nmpc
