// The sampler kernels with bfloat16 logits (sdrm_sample_bf16): K1 in every data flow and K6, launched with the parameters
// engine_host.cu prepares.  A translation unit of their own (see engine_launch.cuh).
#include <cuda_runtime.h>

#include "../../include/sdrm_b200.h"
#include "engine_launch.cuh"
#include "host_util.h"

namespace sdrm {

int launch_engine_bf16(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split) {
  return launch_engine_t<true>(P, grid, cluster, st, split);
}

int launch_small_chain_bf16(const SmallParams& S, int nt, unsigned ctas, cudaStream_t st) {
  return launch_small_chain_t<true>(S, nt, ctas, st);
}

}  // namespace sdrm
