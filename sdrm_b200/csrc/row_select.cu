// K12 — per-row selection: row j of the score matrix keeps exactly k_j ones, its k_j highest scores with ties to the lower item
// index (the activity-matched binarisation of sdrm_b200/sparsify.py), packed in sdrm_threshold_pack's layout.
//
// One CTA of 512 threads owns one row at a time.  The order is K7's (order_key.cuh): NaN ranks as -inf, -0.0 equals +0.0.
//  1. Staging pass: the row is read from global memory once and, when it fits (STAGE_BYTES), copied into dynamic shared memory;
//     the same pass counts the top 8-bit digit of every key in warp-private shared histograms.  A wider row is reread from
//     global memory by every later pass (a wave of CTAs then holds more rows than L2 does: those reads go to HBM).
//  2. MSB-first radix select over the key (32 bits for fp32, 16 for bf16), 8 bits per pass: each pass fixes the digit of the
//     k-th largest key and stops as soon as that digit's bin is taken whole.  It ends with a prefix P of the key's top bits,
//     `need`, the number of keys still to take among those whose prefix equals P, and `cnt`, how many such keys there are.
//  3. Pack pass: warp w owns a contiguous range of 32-column words and forms each word with one ballot.  A key whose prefix is
//     above P is kept; of the keys whose prefix equals P the first `need` in column order are kept (all of them when need == cnt,
//     else a per-warp count of those keys orders the warps first).  No index bits are needed in the key.
// k = 0 and k = n_cols write the row without reading it.
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/sdrm_b200.h"
#include "host_util.h"
#include "order_key.cuh"

// Timing builds of tools/ablate_topk_pack.py only (the bits are then wrong): 1 = the staging pass alone, 2 = staging and the
// radix select without the pack pass.
#ifndef SDRM_TOPK_ABLATE
#define SDRM_TOPK_ABLATE 0
#endif

namespace sdrm_sel {

constexpr int THREADS = 512;
constexpr int WARPS = THREADS / 32;
constexpr int BINS = 256;
constexpr int MAX_COLS = 1 << 20;       // the width bound of K7, K8 and K9
constexpr int STAGE_BYTES = 80 * 1024;  // a 20 480-item fp32 row (40 960 bf16): two CTAs per SM with the histograms
constexpr int UNROLL = 4;               // 16-byte loads in flight per thread in the staging pass

using sdrm_order::score_ord;

template <typename T> struct KeyBits;
template <> struct KeyBits<float> { static constexpr int value = 32; };
template <> struct KeyBits<uint16_t> { static constexpr int value = 16; };

template <typename T>
__global__ void __launch_bounds__(THREADS, 2) topk_pack_kernel(const T* __restrict__ scores, long long rows, int n_cols, long long ld,
                                                               const int32_t* __restrict__ kk, uint32_t* __restrict__ bits,
                                                               long long words_per_row, unsigned long long* __restrict__ count,
                                                               int32_t* __restrict__ status, int staged) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* stage = reinterpret_cast<T*>(smem_raw);
  __shared__ uint32_t hist[WARPS][BINS];
  __shared__ unsigned warp_sum[BINS / 32];
  __shared__ unsigned warp_ties[WARPS];
  __shared__ int s_digit;
  __shared__ unsigned s_above, s_cnt;

  constexpr int KB = KeyBits<T>::value;
  constexpr int VEC = 16 / static_cast<int>(sizeof(T));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int words = (n_cols + 31) >> 5;
  const int tail = n_cols & 31;
  unsigned long long ones = 0;

  for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
    const T* g = scores + row * ld;
    uint32_t* out = bits + row * words_per_row;
    const int k = kk[row];
    if (k <= 0 || k >= n_cols) {   // nothing to select: all zeros, all ones, or a bad k (flagged, row left all zeros)
      const bool bad = k < 0 || k > n_cols;
      if (bad && tid == 0) atomicOr(status, SDRM_TOPK_PACK_BAD_K);
      const bool fill = !bad && k == n_cols;
      for (int w = tid; w < words; w += THREADS) {
        const uint32_t word = !fill ? 0u : (w == words - 1 && tail) ? (1u << tail) - 1u : 0xFFFFFFFFu;
        out[w] = word;
        ones += __popc(word);
      }
      continue;   // (k is the same for the whole CTA: no barrier is skipped by part of it)
    }

    // ---- 1. staging pass with the histogram of the top digit ------------------------------------------------------------
    for (int i = tid; i < WARPS * BINS; i += THREADS) (&hist[0][0])[i] = 0u;
    __syncthreads();
    uint32_t* mine = hist[warp];
    auto count_top = [&](T v) {
      if (SDRM_TOPK_ABLATE != 1) atomicAdd(mine + (score_ord(v) >> (KB - 8)), 1u);
    };
    const bool vec = staged && (reinterpret_cast<uintptr_t>(g) & 15) == 0;
    int c_done = 0;
    if (vec) {
      const int n_vec = n_cols / VEC;
      const uint4* gv = reinterpret_cast<const uint4*>(g);
      uint4* sv = reinterpret_cast<uint4*>(stage);
      int i = tid;
      for (; i + (UNROLL - 1) * THREADS < n_vec; i += UNROLL * THREADS) {
        uint4 v[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) v[u] = __ldcs(gv + i + u * THREADS);
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          sv[i + u * THREADS] = v[u];
          const T* e = reinterpret_cast<const T*>(&v[u]);
#pragma unroll
          for (int j = 0; j < VEC; ++j) count_top(e[j]);
        }
      }
      for (; i < n_vec; i += THREADS) {
        const uint4 v = __ldcs(gv + i);
        sv[i] = v;
        const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int j = 0; j < VEC; ++j) count_top(e[j]);
      }
      c_done = n_vec * VEC;
    }
    for (int c = c_done + tid; c < n_cols; c += THREADS) {
      const T v = staged ? __ldcs(g + c) : __ldg(g + c);
      if (staged) stage[c] = v;
      count_top(v);
    }
    __syncthreads();
    const T* x = staged ? stage : g;   // a generic pointer: shared memory for a staged row, else global memory
    if (SDRM_TOPK_ABLATE == 1) {
      if (tid == 0) out[0] = static_cast<uint32_t>(x[k]);   // (keeps the stage live)
      __syncthreads();
      continue;
    }

    // ---- 2. radix select ---------------------------------------------------------------------------------------------------
    int shift = KB - 8;
    uint32_t pfx = 0;   // the digits fixed so far: key >> (shift + 8) once the digit at `shift` is being counted
    int need = k;       // keys still to take among those whose fixed digits equal pfx
    unsigned cnt = 0;
    for (;;) {
      // bins summed over the warps, inclusive scan from the top digit down: thread t < 256 holds digit 255 - t
      unsigned c = 0, incl = 0;
      if (tid < BINS) {
#pragma unroll
        for (int w = 0; w < WARPS; ++w) c += hist[w][BINS - 1 - tid];
        incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += v;
        }
        if (lane == 31) warp_sum[warp] = incl;
      }
      __syncthreads();
      if (tid < BINS) {
        for (int w = 0; w < warp; ++w) incl += warp_sum[w];
        const unsigned excl = incl - c;
        if (excl < static_cast<unsigned>(need) && static_cast<unsigned>(need) <= incl) {
          s_digit = BINS - 1 - tid;
          s_above = excl;
          s_cnt = c;
        }
      }
      __syncthreads();
      pfx = (pfx << 8) | static_cast<uint32_t>(s_digit);
      need -= static_cast<int>(s_above);
      cnt = s_cnt;
      if (cnt == static_cast<unsigned>(need) || shift == 0) break;   // the bin is taken whole, or the whole key is fixed
      shift -= 8;
      for (int i = tid; i < WARPS * BINS; i += THREADS) (&hist[0][0])[i] = 0u;
      __syncthreads();
      auto count_digit = [&](uint32_t key) {
        if ((key >> (shift + 8)) == pfx) atomicAdd(mine + ((key >> shift) & 255u), 1u);
      };
      if (staged) {   // 16-byte shared-memory loads (the stage is padded to 16 bytes; columns past n_cols are skipped)
        const uint4* sv = reinterpret_cast<const uint4*>(stage);
        const int n_vec = (n_cols + VEC - 1) / VEC;
        for (int i = tid; i < n_vec; i += THREADS) {
          const uint4 v = sv[i];
          const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
          for (int j = 0; j < VEC; ++j)
            if (i * VEC + j < n_cols) count_digit(score_ord(e[j]));
        }
      } else {
        for (int c2 = tid; c2 < n_cols; c2 += THREADS) count_digit(score_ord(__ldg(g + c2)));
      }
      __syncthreads();
    }

    if (SDRM_TOPK_ABLATE == 2) {
      if (tid == 0) out[0] = pfx ^ static_cast<uint32_t>(need);
      __syncthreads();
      continue;
    }

    // ---- 3. pack pass --------------------------------------------------------------------------------------------------------
    const bool all_ties = cnt == static_cast<unsigned>(need);
    const int wpw = (words + WARPS - 1) / WARPS;
    const int w0 = min(words, warp * wpw), w1 = min(words, w0 + wpw);
    unsigned tie_base = 0;
    if (!all_ties) {   // the keys equal to the k-th one are taken in column order: count them per warp range first
      unsigned t = 0;
      for (int w = w0; w < w1; ++w) {
        const int c2 = 32 * w + lane;
        const bool tie = c2 < n_cols && (score_ord(x[c2]) >> shift) == pfx;
        t += __popc(__ballot_sync(0xffffffffu, tie));
      }
      if (lane == 0) warp_ties[warp] = t;
      __syncthreads();
      for (int w = 0; w < warp; ++w) tie_base += warp_ties[w];
    }
    const unsigned lt_mask = (1u << lane) - 1u;
    for (int w = w0; w < w1; ++w) {
      const int c2 = 32 * w + lane;
      const bool valid = c2 < n_cols;
      const uint32_t hi = valid ? (score_ord(x[c2]) >> shift) : 0u;
      const bool tie = valid && hi == pfx;
      const unsigned tb = __ballot_sync(0xffffffffu, tie);
      bool sel = valid && hi > pfx;
      if (tie) sel = all_ties || tie_base + __popc(tb & lt_mask) < static_cast<unsigned>(need);
      tie_base += __popc(tb);
      const unsigned word = __ballot_sync(0xffffffffu, sel);
      if (lane == 0) {
        out[w] = word;
        ones += __popc(word);
      }
    }
    __syncthreads();   // the next row overwrites the stage and the histograms
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ones += __shfl_xor_sync(0xffffffffu, ones, o);
  if (lane == 0 && ones) atomicAdd(count, ones);
}

template <typename T>
static int topk_pack_impl(const char* what, const T* d_scores, int64_t rows, int n_cols, int64_t ld, const int32_t* d_k,
                          uint32_t* d_bits, int64_t words_per_row, unsigned long long* d_count, int32_t* d_status, void* stream) {
  char msg[160];
  if (rows < 0 || n_cols < 1 || ld < n_cols || words_per_row < (static_cast<int64_t>(n_cols) + 31) / 32) {
    snprintf(msg, sizeof msg, "%s: bad shape", what);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  if (n_cols > MAX_COLS) {
    snprintf(msg, sizeof msg, "%s: n_cols above 2^20", what);
    return sdrm_fail(SDRM_ERR_UNSUPPORTED, msg);
  }
  if (rows == 0) return SDRM_OK;
  if (!d_scores || !d_k || !d_bits || !d_count || !d_status) {
    snprintf(msg, sizeof msg, "%s: null pointer", what);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  const int staged = static_cast<int64_t>(n_cols) * static_cast<int64_t>(sizeof(T)) <= STAGE_BYTES ? 1 : 0;
  const int smem = staged ? ((n_cols * static_cast<int>(sizeof(T)) + 15) & ~15) : 0;
  static bool attr_done[64] = {false};   // once per device: allow the largest stage (the 48 KB default covers less)
  int dev = 0, sms = 148, per_sm = 1;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (!(dev < 64 && attr_done[dev])) {
    SDRM_CUDA(cudaFuncSetAttribute(topk_pack_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, STAGE_BYTES));
    if (dev < 64) attr_done[dev] = true;
  }
  SDRM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  SDRM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, topk_pack_kernel<T>, THREADS, smem));
  // one resident wave of CTAs, each looping over rows (row stride = the grid)
  const long long wave = static_cast<long long>(sms) * (per_sm > 0 ? per_sm : 1);
  const long long grid = rows < wave ? rows : wave;
  topk_pack_kernel<T><<<static_cast<unsigned>(grid), THREADS, smem, static_cast<cudaStream_t>(stream)>>>(
      d_scores, rows, n_cols, ld, d_k, d_bits, words_per_row, d_count, d_status, staged);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

}  // namespace sdrm_sel

extern "C" {

int sdrm_topk_pack(const float* d_scores, int64_t rows, int n_cols, int64_t ld, const int32_t* d_k, uint32_t* d_bits,
                   int64_t words_per_row, unsigned long long* d_count, int32_t* d_status, void* stream) {
  return sdrm_sel::topk_pack_impl<float>("sdrm_topk_pack", d_scores, rows, n_cols, ld, d_k, d_bits, words_per_row, d_count, d_status,
                                         stream);
}

int sdrm_topk_pack_bf16(const uint16_t* d_scores, int64_t rows, int n_cols, int64_t ld, const int32_t* d_k, uint32_t* d_bits,
                        int64_t words_per_row, unsigned long long* d_count, int32_t* d_status, void* stream) {
  return sdrm_sel::topk_pack_impl<uint16_t>("sdrm_topk_pack_bf16", d_scores, rows, n_cols, ld, d_k, d_bits, words_per_row, d_count,
                                            d_status, stream);
}

}  // extern "C"
