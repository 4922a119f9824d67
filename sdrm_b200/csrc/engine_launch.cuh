// Launch of the K1 layer engine in each of its data flows, shared by engine_host.cu (fp32 logits) and engine_bf16.cu
// (bfloat16 logits, sdrm_sample_bf16).  The two sets of instantiations live in separate translation units so that the
// fp32 kernels compile exactly as they do without the bfloat16 ones.
#pragma once
#include <cuda_runtime.h>

#include "host_util.h"
#include "layer_engine.cuh"
#include "layer_engine_kernel.cuh"
#include "small_chain_kernel.cuh"

namespace sdrm {

// BF16: the instantiations that store the logits as bfloat16
template <bool BF16>
static int launch_engine_t(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split) {
  if (split > 1) {   // column-split mode: single-CTA tiles, a cluster of `split` CTAs per row tile
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(ENGINE_THREADS);
    cfg.dynamicSmemBytes = ENGINE_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = split; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr; cfg.numAttrs = 1;
    SDRM_CUDA(cudaLaunchKernelEx(&cfg, (sdrm_layer_engine_kernel<1, false, true, BF16>), P));
    return SDRM_OK;
  }
  if (cluster == 1) {
    sdrm_layer_engine_kernel<1, false, false, BF16><<<grid, ENGINE_THREADS, ENGINE_SMEM_BYTES, st>>>(P);
    SDRM_CUDA(cudaGetLastError());
    return SDRM_OK;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(ENGINE_THREADS);
  cfg.dynamicSmemBytes = ENGINE_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  if (cluster == 2 && P.resident) SDRM_CUDA(cudaLaunchKernelEx(&cfg, (sdrm_layer_engine_kernel<2, true, false, BF16>), P));
  else if (cluster == 2) SDRM_CUDA(cudaLaunchKernelEx(&cfg, (sdrm_layer_engine_kernel<2, false, false, BF16>), P));
  else return sdrm_fail(SDRM_ERR_BAD_ARG, "launch_engine: cluster size");
  return SDRM_OK;
}

// engine_bf16.cu: the same launches with bfloat16 logits (K1 in any data flow; K6 with nt = ceil(widest width / 8) n-tiles)
int launch_engine_bf16(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split);
int launch_small_chain_bf16(const SmallParams& S, int nt, unsigned ctas, cudaStream_t st);

}  // namespace sdrm
