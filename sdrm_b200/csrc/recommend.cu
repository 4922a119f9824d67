// K7 — top-k recommendation of every user row with the user's seen items excluded (the reference's
// mask_training_examples + argpartition, utilities.py:116-171, as one kernel).
//
// One CTA of 256 threads owns one user row.  The row's history (CSR: indptr int64, indices int32) is first set into a bitmap in
// shared memory, one bit per item, so no dense mask exists anywhere.  The top k of the remaining items is then found by an MSB-first
// radix select over unique 64-bit keys
//     key = ord(score) << IB | (n_items - 1 - item)        (IB = index bits, a multiple of 8)
// where ord() is the order-preserving unsigned image of the score (32 bits for fp32, 16 for bf16; NaN folded into -inf, -0.0 into
// +0.0).  One unsigned comparison of two keys IS the output order: descending score, ties to the lower item index.  Each pass reads
// the row (from L2 after the first), counts the keys that share the digits fixed so far in a 256-bin shared histogram and fixes the
// next 8-bit digit; it stops as soon as the bin holding the k-th key is taken whole.  A last pass collects the k keys at or above
// that threshold, and a rank count over the k keys in shared memory sorts them.  Continuous scores should resolve in 2-3 counting
// passes (an estimate from the digit widths); tied scores continue into the index digits.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/sdrm_b200.h"
#include "host_util.h"
#include "order_key.cuh"

namespace sdrm_rec {

constexpr int THREADS = 256;
constexpr int MAX_K = 256;          // = THREADS: one output entry per thread in the final rank count
constexpr int MAX_ITEMS = 1 << 20;  // bitmap of 128 KB of shared memory
constexpr int UNROLL = 4;           // loads in flight per thread and pass
static_assert(THREADS == 256, "one histogram bin per thread");

using sdrm_order::score_ord;   // order-preserving unsigned image of a score: 32 bits for fp32, 16 for bf16

__device__ __forceinline__ void store_value(float* p, uint32_t o) {
  *p = __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o);
}
__device__ __forceinline__ void store_value(uint16_t* p, uint32_t o) {
  *p = static_cast<uint16_t>((o & 0x8000u) ? (o & 0x7FFFu) : (~o & 0xFFFFu));
}
__device__ __forceinline__ float neg_inf(float) { return -CUDART_INF_F; }
__device__ __forceinline__ uint16_t neg_inf(uint16_t) { return 0xFF80u; }

// Every thread of the CTA calls this with the same `base`, so each warp runs it converged (the histogram aggregates with
// __match_any_sync).  f(key, valid) is called for each of the UNROLL items base + u * THREADS + tid.
template <typename T, typename F>
__device__ __forceinline__ void scan_chunk(const T* __restrict__ x, const uint32_t* seen, int n_items, int ib, int base, F&& f) {
  T c[UNROLL];
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const int j = base + u * THREADS + static_cast<int>(threadIdx.x);
    c[u] = (j < n_items) ? x[j] : T(0);
  }
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const int j = base + u * THREADS + static_cast<int>(threadIdx.x);
    const bool valid = j < n_items && !((seen[j >> 5] >> (j & 31)) & 1u);
    const unsigned long long key = (static_cast<unsigned long long>(score_ord(c[u])) << ib) |
                                   static_cast<unsigned long long>(n_items - 1 - j);
    f(key, valid);
  }
}

template <typename T>
__global__ void __launch_bounds__(THREADS) recommend_topk_kernel(const T* __restrict__ logits, int n_items, long long ld,
                                                                 const int64_t* __restrict__ indptr,
                                                                 const int32_t* __restrict__ hist, long long nnz, int k,
                                                                 T* __restrict__ val_out, int64_t* __restrict__ idx_out,
                                                                 int* __restrict__ status) {
  extern __shared__ uint32_t seen[];   // exclusion bitmap: bit j of the row's seen items
  __shared__ unsigned int bins[256];
  __shared__ unsigned long long top[MAX_K];
  __shared__ unsigned int warp_sum[THREADS / 32];
  __shared__ int s_digit, s_above, s_cnt, s_count;

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const long long row = blockIdx.x;
  const T* x = logits + row * ld;
  const int words = (n_items + 31) >> 5;

  for (int w = tid; w < words; w += THREADS) seen[w] = 0u;
  __syncthreads();
  long long hs = indptr[row], he = indptr[row + 1];
  if (hs < 0 || he < hs || he > nnz) {
    if (tid == 0) atomicOr(status, SDRM_RECOMMEND_BAD_INDPTR);
    hs = he = 0;
  }
  for (long long e = hs + tid; e < he; e += THREADS) {
    const int it = hist[e];
    if (it < 0 || it >= n_items) atomicOr(status, SDRM_RECOMMEND_BAD_INDEX);
    else atomicOr(&seen[it >> 5], 1u << (it & 31));
  }
  __syncthreads();

  // index bits: a whole number of digits that holds n_items - 1
  const int ib = n_items <= (1 << 8) ? 8 : n_items <= (1 << 16) ? 16 : 24;
  const int key_bits = ib + 8 * static_cast<int>(sizeof(T));
  unsigned long long pfx = 0ull;   // digits fixed so far (bits at and above shift + 8)
  int need = k;                    // keys still to take below the fixed digits
  unsigned long long thr = 0ull;   // the k-th key: the answer is {key >= thr}
  for (int shift = key_bits - 8; shift >= 0; shift -= 8) {
    bins[tid] = 0u;
    __syncthreads();
    const unsigned long long hi_mask = ~0ull << (shift + 8);   // (shift + 8 <= 56)
    for (int base = 0; base < n_items; base += UNROLL * THREADS) {
      scan_chunk(x, seen, n_items, ib, base, [&](unsigned long long key, bool valid) {
        const bool in = valid && (key & hi_mask) == pfx;
        if (!__any_sync(0xffffffffu, in)) return;
        const unsigned d = in ? static_cast<unsigned>(key >> shift) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        if (in && __ffs(peers) - 1 == lane) atomicAdd(&bins[d], static_cast<unsigned>(__popc(peers)));
      });
    }
    __syncthreads();
    // inclusive scan over the bins from the top digit down: thread t holds digit 255 - t
    const unsigned cnt = bins[255 - tid];
    unsigned incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sum[tid >> 5] = incl;
    if (tid == 0) s_digit = -1;
    __syncthreads();
    for (int w = 0; w < (tid >> 5); ++w) incl += warp_sum[w];
    const unsigned excl = incl - cnt;
    if (excl < static_cast<unsigned>(need) && static_cast<unsigned>(need) <= incl) {
      s_digit = 255 - tid;
      s_above = static_cast<int>(excl);
      s_cnt = static_cast<int>(cnt);
    }
    __syncthreads();
    const int digit = s_digit;
    if (digit < 0) {
      // (only on the first pass: fewer than k items are left after the exclusion) -- flag it, fill the row with (-1, -inf)
      if (tid == 0) atomicOr(status, SDRM_RECOMMEND_TOO_FEW_ITEMS);
      if (tid < k) {
        idx_out[row * k + tid] = -1;
        val_out[row * k + tid] = neg_inf(T());
      }
      return;
    }
    pfx |= static_cast<unsigned long long>(digit) << shift;
    if (s_cnt == need - s_above || shift == 0) {   // the bin is taken whole: done (at shift 0 a bin holds one key)
      thr = pfx;
      break;
    }
    need -= s_above;
  }

  if (tid == 0) s_count = 0;
  __syncthreads();
  for (int base = 0; base < n_items; base += UNROLL * THREADS) {
    scan_chunk(x, seen, n_items, ib, base, [&](unsigned long long key, bool valid) {
      if (valid && key >= thr) {
        const int pos = atomicAdd(&s_count, 1);
        if (pos < MAX_K) top[pos] = key;
      }
    });
  }
  __syncthreads();
  if (tid < k) {
    const unsigned long long key = top[tid];
    int rank = 0;
    for (int i = 0; i < k; ++i) rank += top[i] > key ? 1 : 0;
    idx_out[row * k + rank] = static_cast<int64_t>(n_items - 1) - static_cast<int64_t>(key & ((1ull << ib) - 1ull));
    store_value(val_out + row * k + rank, static_cast<uint32_t>(key >> ib));
  }
}

template <typename T>
static int recommend_impl(const T* d_logits, int64_t rows, int n_items, int64_t ld, const int64_t* d_indptr,
                          const int32_t* d_indices, int64_t nnz, int k, T* d_val_out, int64_t* d_idx_out, int32_t* d_status,
                          void* stream) {
  if (!d_logits || !d_indptr || !d_val_out || !d_idx_out || !d_status || (nnz > 0 && !d_indices))
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_recommend_topk: null pointer");
  if (rows < 0 || n_items < 1 || ld < n_items || nnz < 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_recommend_topk: bad shape");
  if (rows > 0x7FFFFFFFLL) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_recommend_topk: more than 2^31 - 1 rows");
  if (n_items > MAX_ITEMS) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_recommend_topk: n_items above 2^20");
  if (k < 1 || k > MAX_K || k > n_items) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_recommend_topk: k must be in [1, min(256, n_items)]");
  if (rows == 0) return SDRM_OK;
  // Once per device, allow the largest bitmap (2^20 bits).  The 48 KB default covers static + dynamic shared memory, and
  // the static part (histogram, top list) would leave a gap below 48 KB of bitmap.  Every caller sets the same value.
  static bool attr_done[64] = {false};
  int dev = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (!(dev < 64 && attr_done[dev])) {
    SDRM_CUDA(cudaFuncSetAttribute(recommend_topk_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(MAX_ITEMS / 32 * sizeof(uint32_t))));
    if (dev < 64) attr_done[dev] = true;
  }
  const size_t smem = static_cast<size_t>((n_items + 31) >> 5) * sizeof(uint32_t);
  recommend_topk_kernel<T><<<static_cast<unsigned>(rows), THREADS, smem, static_cast<cudaStream_t>(stream)>>>(
      d_logits, n_items, ld, d_indptr, d_indices, nnz, k, d_val_out, d_idx_out, d_status);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

}  // namespace sdrm_rec

extern "C" {

int sdrm_recommend_topk(const float* d_logits, int64_t rows, int n_items, int64_t ld, const int64_t* d_indptr,
                        const int32_t* d_indices, int64_t nnz, int k, float* d_val_out, int64_t* d_idx_out,
                        int32_t* d_status, void* stream) {
  return sdrm_rec::recommend_impl<float>(d_logits, rows, n_items, ld, d_indptr, d_indices, nnz, k, d_val_out, d_idx_out,
                                         d_status, stream);
}

int sdrm_recommend_topk_bf16(const uint16_t* d_logits, int64_t rows, int n_items, int64_t ld, const int64_t* d_indptr,
                             const int32_t* d_indices, int64_t nnz, int k, uint16_t* d_val_out, int64_t* d_idx_out,
                             int32_t* d_status, void* stream) {
  return sdrm_rec::recommend_impl<uint16_t>(d_logits, rows, n_items, ld, d_indptr, d_indices, nnz, k, d_val_out, d_idx_out,
                                            d_status, stream);
}

}  // extern "C"
