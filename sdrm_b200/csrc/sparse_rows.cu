// K10 — bit-packed binary rows -> CSR (indptr int64[rows + 1], indices int32[nnz]) on the device.
//
// Input: sdrm_threshold_pack's layout (bit j of word w of a row is column 32 w + j, words_ld words per row); bits at or past
// n_cols are masked off, whatever the padding holds.
//
//   indptr:  count_scan_kernel (a warp per row: popcount of the row's words; the block's 128 counts scanned in shared memory,
//            the block total to the workspace), block_offsets_kernel (one block scans the block totals), add_offsets_kernel.
//            Integer sums: the result does not depend on the launch shape, and the same bits give the same indptr every call.
//   indices: a warp per row, lane i owns word 32 c + i of chunk c; a warp scan of the lanes' popcounts gives each lane's write
//            offset inside the chunk, the lanes write their column indices (ascending by construction) to a shared-memory
//            staging buffer, and the warp copies the chunk to global memory with contiguous stores.
// Both passes read the bits once; the work per byte is a popcount and a few shuffles, so they are memory-bound.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/sdrm_b200.h"
#include "host_util.h"

namespace sdrm_csr {

constexpr int THREADS = 256;
constexpr int WARPS = THREADS / 32;
constexpr int SCAN_ROWS = 128;                       // rows per block of the counting pass (one workspace entry each)
constexpr int ROWS_PER_WARP = SCAN_ROWS / WARPS;
constexpr int OFFSET_THREADS = 1024;

// the row's word w with the bits at or past n_cols cleared
__device__ __forceinline__ uint32_t row_word(const uint32_t* row, int64_t w, int64_t n_words, int tail_bits) {
  if (w >= n_words) return 0u;
  uint32_t v = __ldg(row + w);
  if (w == n_words - 1 && tail_bits) v &= (1u << tail_bits) - 1u;
  return v;
}

__global__ void __launch_bounds__(THREADS) count_scan_kernel(const uint32_t* __restrict__ words, int64_t words_ld, int64_t rows,
                                                             int n_cols, int64_t* __restrict__ indptr,
                                                             int64_t* __restrict__ block_sums) {
  __shared__ int64_t counts[SCAN_ROWS];
  __shared__ int64_t warp_tot[SCAN_ROWS / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n_words = (static_cast<int64_t>(n_cols) + 31) / 32;
  const int tail_bits = n_cols & 31;
  const int64_t n_full = tail_bits ? n_words - 1 : n_words;   // words with no bit at or past n_cols
  const int64_t row0 = static_cast<int64_t>(blockIdx.x) * SCAN_ROWS;
  for (int i = 0; i < ROWS_PER_WARP; ++i) {
    const int local = warp * ROWS_PER_WARP + i;
    const int64_t r = row0 + local;
    int64_t c = 0;
    if (r < rows) {
      const uint32_t* row = words + r * words_ld;
      int64_t w = lane;
      // four independent loads in flight per lane, on full words only; the rest (and the masked last word) one at a time
      for (; w + 96 < n_full; w += 128)
        c += __popc(__ldg(row + w)) + __popc(__ldg(row + w + 32)) + __popc(__ldg(row + w + 64)) + __popc(__ldg(row + w + 96));
      for (; w < n_words; w += 32) c += __popc(row_word(row, w, n_words, tail_bits));
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) counts[local] = c;
  }
  __syncthreads();
  // inclusive scan of the 128 counts: threads 0..127, one warp scan each, then the four warp totals
  int64_t v = 0;
  if (threadIdx.x < SCAN_ROWS) {
    v = counts[threadIdx.x];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    if (lane == 31) warp_tot[warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < SCAN_ROWS) {
    for (int k = 0; k < warp; ++k) v += warp_tot[k];
    const int64_t r = row0 + threadIdx.x;
    if (r < rows) indptr[r + 1] = v;
    if (threadIdx.x == SCAN_ROWS - 1) block_sums[blockIdx.x] = v;
  }
}

// exclusive scan of the block totals in place (one block, chunks of 1024 with a running carry)
__global__ void __launch_bounds__(OFFSET_THREADS) block_offsets_kernel(int64_t* __restrict__ block_sums, int64_t n_blocks) {
  __shared__ int64_t warp_tot[OFFSET_THREADS / 32];
  __shared__ int64_t carry;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < n_blocks; base += OFFSET_THREADS) {
    const int64_t i = base + threadIdx.x;
    const int64_t x = i < n_blocks ? block_sums[i] : 0;
    int64_t v = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    if (warp == 0) {
      int64_t t = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int64_t u = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += u;
      }
      warp_tot[lane] = t;   // inclusive over warps
    }
    __syncthreads();
    const int64_t c = carry;
    const int64_t incl = v + (warp ? warp_tot[warp - 1] : 0);
    if (i < n_blocks) block_sums[i] = c + incl - x;
    __syncthreads();
    if (threadIdx.x == OFFSET_THREADS - 1) carry = c + incl;
    __syncthreads();
  }
}

__global__ void add_offsets_kernel(int64_t* __restrict__ indptr, int64_t rows, const int64_t* __restrict__ block_offsets) {
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows; r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t b = r / SCAN_ROWS;
    if (b) indptr[r + 1] += block_offsets[b];
  }
}

__global__ void __launch_bounds__(THREADS) indices_kernel(const uint32_t* __restrict__ words, int64_t words_ld, int64_t rows, int n_cols,
                                                          const int64_t* __restrict__ indptr, int32_t* __restrict__ indices) {
  __shared__ int32_t stage[WARPS][32 * 32];          // one chunk of 32 words holds at most 1024 ones
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int32_t* buf = stage[warp];
  const int64_t n_words = (static_cast<int64_t>(n_cols) + 31) / 32;
  const int tail_bits = n_cols & 31;
  const int64_t warp_step = static_cast<int64_t>(gridDim.x) * WARPS;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * WARPS + warp; r < rows; r += warp_step) {
    const uint32_t* row = words + r * words_ld;
    int32_t* out = indices + indptr[r];
    for (int64_t w0 = 0; w0 < n_words; w0 += 32) {
      const int64_t w = w0 + lane;
      uint32_t bits = row_word(row, w, n_words, tail_bits);
      const int c = __popc(bits);
      int off = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, off, o);
        if (lane >= o) off += u;
      }
      const int total = __shfl_sync(0xffffffffu, off, 31);
      if (total == 0) continue;
      off -= c;
      const int32_t col0 = static_cast<int32_t>(w * 32);    // < n_cols <= 2^31 - 1 whenever the word has a bit left
      while (bits) {
        buf[off++] = col0 + (__ffs(bits) - 1);
        bits &= bits - 1u;
      }
      __syncwarp();
      for (int k = lane; k < total; k += 32) out[k] = buf[k];
      __syncwarp();
      out += total;
    }
  }
}

inline int64_t scan_blocks(int64_t rows) { return rows > 0 ? (rows + SCAN_ROWS - 1) / SCAN_ROWS : 0; }

int check_shape(const char* what, const uint32_t* d_words, int64_t words_ld, int64_t rows, int n_cols) {
  char msg[192];
  if (rows < 0 || n_cols < 1) {
    snprintf(msg, sizeof msg, "%s: bad shape (rows = %lld, n_cols = %d; rows >= 0 and n_cols >= 1)", what, static_cast<long long>(rows), n_cols);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  if (words_ld < (static_cast<int64_t>(n_cols) + 31) / 32) {
    snprintf(msg, sizeof msg, "%s: words_ld = %lld < ceil(n_cols / 32) = %lld", what, static_cast<long long>(words_ld),
             static_cast<long long>((static_cast<int64_t>(n_cols) + 31) / 32));
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  if (rows > 0 && !d_words) {
    snprintf(msg, sizeof msg, "%s: null pointer (d_words)", what);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  return SDRM_OK;
}

}  // namespace sdrm_csr

using namespace sdrm_csr;

extern "C" {

size_t sdrm_packed_csr_workspace_bytes(int64_t rows) { return static_cast<size_t>(scan_blocks(rows)) * sizeof(int64_t); }

int sdrm_packed_csr_indptr(const uint32_t* d_words, int64_t words_ld, int64_t rows, int n_cols, int64_t* d_indptr, void* d_workspace,
                           size_t workspace_bytes, void* stream) {
  if (!d_indptr) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_packed_csr_indptr: null pointer (d_indptr)");
  const int rc = check_shape("sdrm_packed_csr_indptr", d_words, words_ld, rows, n_cols);
  if (rc != SDRM_OK) return rc;
  const int64_t blocks = scan_blocks(rows);
  if (rows > 0 && !d_workspace) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_packed_csr_indptr: null pointer (d_workspace)");
  if (workspace_bytes < static_cast<size_t>(blocks) * sizeof(int64_t))
    return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_packed_csr_indptr: workspace smaller than sdrm_packed_csr_workspace_bytes(rows)");
  if (blocks > 0x7fffffffLL) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_packed_csr_indptr: too many rows for one launch");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaMemsetAsync(d_indptr, 0, sizeof(int64_t), s));
  if (rows == 0) return SDRM_OK;
  int64_t* sums = static_cast<int64_t*>(d_workspace);
  count_scan_kernel<<<static_cast<unsigned>(blocks), THREADS, 0, s>>>(d_words, words_ld, rows, n_cols, d_indptr, sums);
  SDRM_CUDA(cudaGetLastError());
  if (blocks > 1) {
    block_offsets_kernel<<<1, OFFSET_THREADS, 0, s>>>(sums, blocks);
    SDRM_CUDA(cudaGetLastError());
    const int64_t grid = (rows + 255) / 256;
    add_offsets_kernel<<<static_cast<unsigned>(grid < 65536 ? grid : 65536), 256, 0, s>>>(d_indptr, rows, sums);
    SDRM_CUDA(cudaGetLastError());
  }
  return SDRM_OK;
}

int sdrm_packed_csr_indices(const uint32_t* d_words, int64_t words_ld, int64_t rows, int n_cols, const int64_t* d_indptr,
                            int32_t* d_indices, void* stream) {
  const int rc = check_shape("sdrm_packed_csr_indices", d_words, words_ld, rows, n_cols);
  if (rc != SDRM_OK) return rc;
  if (rows > 0 && (!d_indptr || !d_indices)) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_packed_csr_indices: null pointer (d_indptr / d_indices)");
  if (rows == 0) return SDRM_OK;
  const int64_t want = (rows + WARPS - 1) / WARPS;
  const unsigned grid = static_cast<unsigned>(want < (1 << 20) ? want : (1 << 20));
  indices_kernel<<<grid, THREADS, 0, static_cast<cudaStream_t>(stream)>>>(d_words, words_ld, rows, n_cols, d_indptr, d_indices);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

}  // extern "C"
