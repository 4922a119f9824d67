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
