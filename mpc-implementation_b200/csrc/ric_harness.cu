// ric_harness.cu -- test harness of the Riccati factorisation and sweeps (nmpc_riccati.cuh) on caller-supplied LQ data.
// Built into its own libnmpc_ric_harness.so for tests/test_riccati_kernel.py; libnmpc_b200.so does not contain it.
//
// One warp (a block of 32 threads) per instance, with one Lay::TOTAL slice of dynamic shared memory, runs the device
// functions of nmpc_ipm_kernel in the order solve_instance runs them:
//   1. shared slice <- poison [TOTAL] (the caller's pattern), ric rows 0..N (one row past the last stage) <- ric_poison
//   2. LQ entries [LQ_NE][S] at Lay::LQ0 <- lq[b]
//   3. riccati_factor for each (mu, dw) of seq[b] in turn, ok[b][i] <- its verdict; a failed pair followed by another
//      replays an inertia-correction retry on the same shared memory
//   4. if the last pair succeeded: riccati_forward (dx -> LV_DX, du -> LV_DU); slice -> slices[b][0]
//   5. if q2 is given: q' -> soc(SOC_Q2), riccati_resolve, riccati_forward(soc) (dx -> LV_DX, du -> soc(SOC_DUS))
//   6. slice -> slices[b][1]  (the ric rows are the caller's buffer)
// The ownership map is built by ric_map_kernel in a launch of its own before the harness kernel, as nmpc_create does:
// riccati_factor reads it through the read-only data path, which must not see a table written by the same kernel.
// All buffers are device pointers; the harness copies nothing between host and device.
#include <cuda_runtime.h>
#include "../../include/nmpc_b200.h"
#include "nmpc_solve.cuh"

using namespace nmpc;

namespace {

template <class L>
__global__ void __launch_bounds__(32) ric_harness_kernel(const double* __restrict__ Ts, const double* __restrict__ lq,
                                                         const double* __restrict__ seq, int nseq, const double* __restrict__ q2,
                                                         const double* __restrict__ poison, const double* __restrict__ ric_poison,
                                                         const unsigned* __restrict__ map, int* __restrict__ ok_out,
                                                         double* __restrict__ slices, double* __restrict__ ric_all) {
  constexpr int S = L::S;
  const int b = blockIdx.x, lane = threadIdx.x & 31;
  double* sm = smem_all;                  // the block is one warp: its slice starts at the base
  double* ric = ric_all + (size_t)b * S * RIC_N;
  for (int i = lane; i < L::TOTAL; i += 32) sm[i] = poison[i];
  for (int i = lane; i < S * RIC_N; i += 32) ric[i] = ric_poison[i % RIC_N];
  __syncwarp();
  for (int i = lane; i < L::LQ_NE * S; i += 32) sm[L::LQ0 + i] = lq[(size_t)b * L::LQ_NE * S + i];
  __syncwarp();
  const double T = Ts[b];
  bool ok = false;
  double mu = 0.0;
  for (int i = 0; i < nseq; ++i) {
    mu = seq[((size_t)b * nseq + i) * 2];
    ok = riccati_factor<L>(T, ric, map, mu, seq[((size_t)b * nseq + i) * 2 + 1], lane);
    __syncwarp();
    if (lane == 0) ok_out[b * nseq + i] = ok ? 1 : 0;
  }
  if (ok) riccati_forward<L>(T, ric, false, lane, L::LV0 + LV_DX * S, L::LV0 + LV_DU * S);
  double* out = slices + (size_t)b * 2 * L::TOTAL;
  for (int i = lane; i < L::TOTAL; i += 32) out[i] = sm[i];
  __syncwarp();
  if (ok && q2 != nullptr) {
    for (int i = lane; i < 8 * S; i += 32) sm[L::soc(SOC_Q2) + i] = q2[(size_t)b * 8 * S + i];
    __syncwarp();
    riccati_resolve<L>(T, L::soc(SOC_Q2), ric, mu, lane);
    riccati_forward<L>(T, ric, true, lane, L::LV0 + LV_DX * S, L::soc(SOC_DUS));
  }
  for (int i = lane; i < L::TOTAL; i += 32) out[L::TOTAL + i] = sm[i];
}

template <class L>
int ric_run(int B, const double* T, const double* lq, const double* seq, int nseq, const double* q2, const double* poison,
            const double* ric_poison, unsigned* map, int* ok, double* slices, double* ric, cudaStream_t s) {
  const size_t bytes = sizeof(double) * L::TOTAL;
  if (bytes > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(ric_harness_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
  }
  ric_map_kernel<L><<<1, 32, 0, s>>>(map);
  ric_harness_kernel<L><<<B, 32, bytes, s>>>(T, lq, seq, nseq, q2, poison, ric_poison, map, ok, slices, ric);
  return (int)cudaGetLastError();
}

// the layout constants the tests read (their order is RIC_CONSTS in tests/test_riccati_kernel.py)
template <class L>
int ric_consts(long long* out) {
  const long long v[] = {L::N, L::S, L::MODEL, L::FOLD, L::TOTAL, L::LV0, L::RW0, L::LQ0, L::LQ_NE, L::SOCX0, L::STG0,
                         L::OBS0, L::ALG0, L::RES0, L::PAR0, L::soc(SOC_DUS), L::soc(SOC_Q2), STG_N, RIC_N, RIC_K, RIC_L,
                         RIC_K2, RIC_MAP_WORDS, LV_DX, LV_DU, LV_N, LQ_Q, LQ_DEAD, LQ_QA, LQ_SV, LQ_RD, LQ_RB, LQ_DD,
                         LQ_EE, LQ_ZERO, LQ_DG, LQ_NN, LQ_QD, LQ_QB};
  const int n = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < n; ++i) out[i] = v[i];
  return n;
}

}  // namespace

#define RIC_LAYOUT(tag, ...)                                                                                               \
  extern "C" int ric_run_##tag(int B, const double* T, const double* lq, const double* seq, int nseq, const double* q2,    \
                               const double* poison, const double* ric_poison, unsigned* map, int* ok, double* slices,    \
                               double* ric, void* stream) {                                                               \
    return ric_run<__VA_ARGS__>(B, T, lq, seq, nseq, q2, poison, ric_poison, map, ok, slices, ric, (cudaStream_t)stream); \
  }                                                                                                                        \
  extern "C" int ric_consts_##tag(long long* out) { return ric_consts<__VA_ARGS__>(out); }

// the seven production instantiations, with the FOLD choice of production
RIC_LAYOUT(p15_3, Lay<15, 3>)
RIC_LAYOUT(p15_10, Lay<15, 10>)
RIC_LAYOUT(p30_10, Lay<30, 10>)
RIC_LAYOUT(p30_3, Lay<30, 3>)
RIC_LAYOUT(p5_3, Lay<5, 3>)
RIC_LAYOUT(p15_7, Lay<15, 7>)
RIC_LAYOUT(p15_0_1, Lay<15, 0, 1>)
// edges: both LQ layouts whatever NMPC_FOLD_MIN_S picks, a single backward stage, two stages, and S = 32 (every lane owns a
// stage, lane 31 is lane N of the forward sweep)
RIC_LAYOUT(f15_3, LayT<15, 3, true>)
RIC_LAYOUT(n30_10, LayT<30, 10, false>)
RIC_LAYOUT(n1_3, LayT<1, 3, false>)
RIC_LAYOUT(n2_3, LayT<2, 3, false>)
RIC_LAYOUT(n31_16, LayT<31, 16, false>)
