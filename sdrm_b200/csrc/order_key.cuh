// The order-preserving unsigned key of a score shared by the per-row selections (K7 recommend.cu, K12 row_select.cu): one
// unsigned comparison of two keys is the comparison of the scores, with NaN ranked as -inf and -0.0 equal to +0.0.  32 bits for
// fp32, 16 for bf16 (kept as its raw bits).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

namespace sdrm_order {

__device__ __forceinline__ uint32_t canonical_bits(float v) {
  v = v + 0.0f;                          // -0.0 -> +0.0: equal scores must have equal keys
  return __float_as_uint((v != v) ? -CUDART_INF_F : v);   // NaN ranks as -inf
}
__device__ __forceinline__ uint32_t score_ord(float x) {
  const uint32_t u = canonical_bits(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ uint32_t score_ord(uint16_t x) {
  const uint32_t u = canonical_bits(__uint_as_float(static_cast<uint32_t>(x) << 16)) >> 16;   // (exact: bf16 is fp32's top half)
  return (u & 0x8000u) ? (~u & 0xFFFFu) : (u | 0x8000u);
}

}  // namespace sdrm_order
