// The sampler kernels with bfloat16 logits (sdrm_sample_bf16): K1 in every data flow and K6, launched with the parameters
// engine_host.cu prepares.  A translation unit of their own (see engine_launch.cuh).
#include <cuda_runtime.h>
#include <stdlib.h>

#include "../../include/sdrm_b200.h"
#include "engine_launch.cuh"
#include "host_util.h"

namespace sdrm {

// run-time watchdog limit of this translation unit's kernels (ptx_sm100.cuh): SDRM_WATCHDOG_MS in the environment, 0 = none
static int apply_watchdog_env_bf16() {
  static bool done = false;
  if (done) return SDRM_OK;
  done = true;
  const char* e = getenv("SDRM_WATCHDOG_MS");
  if (!e || !*e) return SDRM_OK;
  const unsigned long long ns = strtoull(e, nullptr, 10) * 1000000ull;
  SDRM_CUDA(cudaMemcpyToSymbol(g_sdrm_watchdog_ns, &ns, sizeof ns));
  return SDRM_OK;
}

int launch_engine_bf16(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split) {
  { int wrc = apply_watchdog_env_bf16(); if (wrc) return wrc; }
  static bool done[64] = {false};
  int dev = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (!(dev < 64 && done[dev])) {
    SDRM_CUDA(cudaFuncSetAttribute((sdrm_layer_engine_kernel<1, false, false, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
    SDRM_CUDA(cudaFuncSetAttribute((sdrm_layer_engine_kernel<2, false, false, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
    SDRM_CUDA(cudaFuncSetAttribute((sdrm_layer_engine_kernel<2, true, false, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
    SDRM_CUDA(cudaFuncSetAttribute((sdrm_layer_engine_kernel<1, false, true, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
    if (dev < 64) done[dev] = true;
  }
  return launch_engine_t<true>(P, grid, cluster, st, split);
}

int launch_small_chain_bf16(const SmallParams& S, int nt, unsigned ctas, cudaStream_t st) {
  { int wrc = apply_watchdog_env_bf16(); if (wrc) return wrc; }
  auto launch = [&](auto kernel, int smem) -> int {
    SDRM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kernel<<<ctas, SMALL_THREADS, smem, st>>>(S);
    SDRM_CUDA(cudaGetLastError());
    return SDRM_OK;
  };
  if (nt <= 3) return launch(sdrm_small_chain_kernel<3, true>, SmallGeom<3>::SMEM_BYTES);
  if (nt <= 5) return launch(sdrm_small_chain_kernel<5, true>, SmallGeom<5>::SMEM_BYTES);
  return launch(sdrm_small_chain_kernel<8, true>, SmallGeom<8>::SMEM_BYTES);
}

}  // namespace sdrm
