// nmpc_inst.cu -- one translation unit per (N, n_obs, model) instantiation of the IPM kernel (compiled in parallel):
//   nvcc -DINST_N=15 -DINST_NOBS=3 [-DINST_MODEL=0] -c nmpc_inst.cu -o inst_15_3.o
#include <cuda_runtime.h>
#include "../../include/nmpc_b200.h"
#include "nmpc_sens.cuh"

#if !defined(INST_N) || !defined(INST_NOBS)
#error "compile with -DINST_N=<horizon> -DINST_NOBS=<obstacle rows>"
#endif
#ifndef INST_MODEL
#define INST_MODEL 0
#endif
#define NMPC_CAT_(a, b, c, d) a##_##b##_##c##_##d
#define NMPC_CAT3(a, b, c, d) NMPC_CAT_(a, b, c, d)
#define NMPC_CAT(a, b, c) NMPC_CAT3(a, b, c, INST_MODEL)

namespace nmpc {

int NMPC_CAT(ipm_prepare, INST_N, INST_NOBS)(int* blocks_per_sm, size_t* smem_bytes, int* warps_per_block, int* cold_doubles) {
  using L = Lay<INST_N, INST_NOBS, INST_MODEL>;
  const size_t bytes = (size_t)L::TOTAL * sizeof(double) * L::WPB;
  *warps_per_block = L::WPB;
  *cold_doubles = L::COLD_TOTAL;
  cudaError_t e = cudaFuncSetAttribute(nmpc_ipm_kernel<INST_N, INST_NOBS, INST_MODEL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(nmpc_ipm_kernel<INST_N, INST_NOBS, INST_MODEL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return (int)e;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, nmpc_ipm_kernel<INST_N, INST_NOBS, INST_MODEL>, 32 * L::WPB, bytes);
  *smem_bytes = bytes;
  return (int)e;
}

// fills the [RIC_MAP_WORDS][32] table the factorisation loads its ownership maps from (once, at nmpc_create)
int NMPC_CAT(ipm_ricmap, INST_N, INST_NOBS)(unsigned* dev_table, cudaStream_t s) {
  ric_map_kernel<Lay<INST_N, INST_NOBS, INST_MODEL>><<<1, 32, 0, s>>>(dev_table);
  return (int)cudaGetLastError();
}

int NMPC_CAT(ipm_launch, INST_N, INST_NOBS)(const SolveArgs& A, int blocks, size_t bytes, cudaStream_t s) {
  using L = Lay<INST_N, INST_NOBS, INST_MODEL>;
  if (A.sig_x) nmpc_ipm_kernel<INST_N, INST_NOBS, INST_MODEL, true><<<blocks, 32 * L::WPB, bytes, s>>>(A);      // NMPC_KEEP_BARRIER
  else nmpc_ipm_kernel<INST_N, INST_NOBS, INST_MODEL><<<blocks, 32 * L::WPB, bytes, s>>>(A);
  return (int)cudaGetLastError();
}

// nmpc_sensitivity: `blocks` warps (one per block) over the B instances, each on Riccati scratch slot blockIdx.x
int NMPC_CAT(ipm_sens, INST_N, INST_NOBS)(const SolveArgs& A, int blocks, cudaStream_t s) {
  using L = Lay<INST_N, INST_NOBS, INST_MODEL>;
  const size_t bytes = sizeof(double) * L::TOTAL;
  cudaError_t e = cudaFuncSetAttribute(nmpc_sens_kernel<INST_N, INST_NOBS, INST_MODEL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return (int)e;
  nmpc_sens_kernel<INST_N, INST_NOBS, INST_MODEL><<<blocks, 32, bytes, s>>>(A);
  return (int)cudaGetLastError();
}

}  // namespace nmpc
