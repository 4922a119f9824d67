// Launch of the K1 layer engine in each of its data flows and of K6, shared by engine_host.cu (fp32 logits) and engine_bf16.cu
// (bfloat16 logits, sdrm_sample_bf16).  The two sets of instantiations live in separate translation units so that the
// fp32 kernels compile exactly as they do without the bfloat16 ones.
#pragma once
#include <cuda_runtime.h>

#include "host_util.h"
#include "layer_engine.cuh"
#include "layer_engine_kernel.cuh"
#include "small_chain_kernel.cuh"

namespace sdrm {

typedef void (*EngineKernel)(ChainParams);

// The K1 instantiation of a data flow (BF16: the ones that store the logits as bfloat16): single CTAs, CTA pairs, resident
// pairs, column split.  The only place that names them, so a translation unit's module lists them in this order.
template <bool BF16>
static EngineKernel engine_kernel(int cluster, bool resident, bool split) {
  if (!split && cluster == 1) return sdrm_layer_engine_kernel<1, false, false, BF16>;
  if (!split && !resident) return sdrm_layer_engine_kernel<2, false, false, BF16>;
  if (!split) return sdrm_layer_engine_kernel<2, true, false, BF16>;
  return sdrm_layer_engine_kernel<1, false, true, BF16>;
}

// Per-device set-up of this translation unit's K1 kernels: the watchdog limit and the dynamic shared-memory size of the four
// instantiations.
template <bool BF16>
static int engine_setup() {
  static bool done[64] = {false};
  int dev = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && done[dev]) return SDRM_OK;
  { int rc = apply_watchdog_env(); if (rc) return rc; }
  const EngineKernel kernels[4] = {engine_kernel<BF16>(1, false, false), engine_kernel<BF16>(2, false, false),
                                   engine_kernel<BF16>(2, true, false), engine_kernel<BF16>(1, false, true)};
  for (EngineKernel k : kernels) SDRM_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
  if (dev < 64) done[dev] = true;
  return SDRM_OK;
}

// launch configuration of `grid` engine CTAs in clusters of `cluster` CTAs (not copyable: cfg.attrs points into it)
struct EngineClusterConfig {
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr;
  EngineClusterConfig(int grid, int cluster, cudaStream_t st) {
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(ENGINE_THREADS);
    cfg.dynamicSmemBytes = ENGINE_SMEM_BYTES;
    cfg.stream = st;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr; cfg.numAttrs = 1;
  }
  EngineClusterConfig(const EngineClusterConfig&) = delete;
  EngineClusterConfig& operator=(const EngineClusterConfig&) = delete;
};

// split > 1: column-split mode, single-CTA tiles in clusters of `split` CTAs per row tile
template <bool BF16>
static int launch_engine_t(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split) {
  { int rc = engine_setup<BF16>(); if (rc) return rc; }
  const EngineKernel kernel = engine_kernel<BF16>(cluster, P.resident != 0, split > 1);
  if (split > 1 || cluster == 2) {
    EngineClusterConfig c(grid, split > 1 ? split : cluster, st);
    SDRM_CUDA(cudaLaunchKernelEx(&c.cfg, kernel, P));
    return SDRM_OK;
  }
  if (cluster != 1) return sdrm_fail(SDRM_ERR_BAD_ARG, "launch_engine: cluster size");
  kernel<<<grid, ENGINE_THREADS, ENGINE_SMEM_BYTES, st>>>(P);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

// K6 with nt = ceil(widest width / 8) n-tiles of 8 columns
template <bool BF16>
static int launch_small_chain_t(const SmallParams& S, int nt, unsigned ctas, cudaStream_t st) {
  auto launch = [&](auto kernel, int smem) -> int {
    SDRM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kernel<<<ctas, SMALL_THREADS, smem, st>>>(S);
    SDRM_CUDA(cudaGetLastError());
    return SDRM_OK;
  };
  if (nt <= 3) return launch(sdrm_small_chain_kernel<3, BF16>, SmallGeom<3>::SMEM_BYTES);
  if (nt <= 5) return launch(sdrm_small_chain_kernel<5, BF16>, SmallGeom<5>::SMEM_BYTES);
  return launch(sdrm_small_chain_kernel<8, BF16>, SmallGeom<8>::SMEM_BYTES);
}

// engine_bf16.cu: the same launches with bfloat16 logits
int launch_engine_bf16(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split);
int launch_small_chain_bf16(const SmallParams& S, int nt, unsigned ctas, cudaStream_t st);

}  // namespace sdrm
