// Error plumbing and driver entry points shared by the C-ABI translation units.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdio.h>

int sdrm_fail(int code, const char* msg);  // records the thread-local message, returns code

#define SDRM_CUDA(expr)                                                                         \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      char _m[256];                                                                             \
      snprintf(_m, sizeof _m, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
               __LINE__);                                                                       \
      return sdrm_fail(-3, _m);                                                                 \
    }                                                                                           \
  } while (0)

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda); null when the driver lacks it
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// uint8 0/1 operand image [rows, pitch] (K8 / K9): box = 128 columns x box_rows rows, SWIZZLE_128B
static inline int make_u8_map(CUtensorMap* map, const void* base, long long rows, long long pitch, unsigned box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return sdrm_fail(-3, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(pitch), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(pitch)};
  const cuuint32_t box[2] = {128u, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char msg[160];
    snprintf(msg, sizeof msg, "cuTensorMapEncodeTiled (u8) failed (%d) rows=%lld pitch=%lld box_rows=%u", static_cast<int>(r), rows, pitch, box_rows);
    return sdrm_fail(-3, msg);
  }
  return 0;
}
