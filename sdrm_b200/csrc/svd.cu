// K11 — products of binary CSR rows with a skinny fp64 matrix: Y[r, :] = sum over j in row r of X[j, :], w <= 32 columns.
//
// The randomized truncated SVD of the SVD evaluator (sdrm_b200/svd.py) runs every product of its power iterations through
// this kernel: A·Q on the CSR of A, Aᵀ·Q on the CSR of Aᵀ, and the scoring product X_test·VTᵀ.
//
//   spmm_chunk_kernel: the nnz entries are cut into fixed chunks of CHUNK entries, one warp per chunk, lane l owns column l.
//            A chunk may hold the end of one row, whole rows and the start of another.  The warp finds the row of its first
//            entry by a binary search of indptr, then walks the entries in order: 32 indices are loaded by the lanes at once
//            and broadcast one by one with a shuffle; the gathered X rows are loaded 16 at a time (16 loads in flight per
//            lane) and added in entry order.  A row that lies inside the chunk is written to Y; the partial sum of the row
//            the chunk starts in goes to first[chunk], that of the row it ends in to last[chunk].
//   spmm_fixup_kernel: one warp per row.  Checks the row's indptr pair, writes 0 for an empty row, and for a row that
//            crosses chunk boundaries sums last[c0] + first[c0 + 1] + ... + first[c1] in that order.
// Every sum has a fixed order that depends on the data only, never on the launch or on scheduling (no atomics on values),
// so the same inputs give bit-identical Y on every call.  A popular item with thousands of users (a long row of Aᵀ) is
// split over many warps instead of serialising on one.  An index outside [0, n_x) contributes nothing and ORs
// SDRM_SPMM_BAD_INDEX into the status word; a bad indptr pair zeroes its row and ORs SDRM_SPMM_BAD_INDPTR.  Neither faults.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/sdrm_b200.h"
#include "host_util.h"

namespace sdrm_spmm {

constexpr int CHUNK = 256;                 // entries per warp of the chunk pass
constexpr int WARPS = 4;
constexpr int THREADS = WARPS * 32;
constexpr int LOADS = 16;                  // gathered X loads in flight per lane

inline int64_t n_chunks(int64_t nnz) { return nnz > 0 ? (nnz + CHUNK - 1) / CHUNK : 0; }

__global__ void __launch_bounds__(THREADS) spmm_chunk_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                             int64_t rows, int64_t nnz, const double* __restrict__ x, int64_t n_x,
                                                             int w, int64_t ldx, double* __restrict__ y, int64_t ldy,
                                                             double* __restrict__ first, double* __restrict__ last,
                                                             int32_t* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  const int64_t g = static_cast<int64_t>(blockIdx.x) * WARPS + (threadIdx.x >> 5);
  const int64_t c_beg = g * CHUNK;
  if (c_beg >= nnz) return;
  const int64_t c_end = c_beg + CHUNK < nnz ? c_beg + CHUNK : nnz;
  // the last row r with indptr[r] <= c_beg (a non-empty row when indptr is valid)
  int64_t lo = 0, hi = rows - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (__ldg(indptr + mid) <= c_beg) lo = mid; else hi = mid - 1;
  }
  const bool col = lane < w;
  const double* xl = x + lane;
  int64_t p = c_beg;
  for (int64_t r = lo; p < c_end && r < rows; ++r) {
    const int64_t rs = __ldg(indptr + r), re = __ldg(indptr + r + 1);
    if (re <= p) continue;                 // empty row (or an inconsistent pair, which the fix-up pass reports)
    const int64_t seg_end = re < c_end ? re : c_end;
    double acc = 0.0;
    for (int64_t base = p; base < seg_end; base += 32) {
      const int n = seg_end - base < 32 ? static_cast<int>(seg_end - base) : 32;
      int j = lane < n ? __ldg(indices + base + lane) : 0;
      const bool bad = lane < n && (j < 0 || static_cast<int64_t>(j) >= n_x);
      if (bad) atomicOr(status, SDRM_SPMM_BAD_INDEX);
      if (bad) j = -1;                     // gathers nothing
      if (n == 32) {
#pragma unroll
        for (int k0 = 0; k0 < 32; k0 += LOADS) {
          double v[LOADS];
#pragma unroll
          for (int u = 0; u < LOADS; ++u) {
            const int jk = __shfl_sync(0xffffffffu, j, k0 + u);
            v[u] = (col && jk >= 0) ? __ldg(xl + static_cast<int64_t>(jk) * ldx) : 0.0;
          }
#pragma unroll
          for (int u = 0; u < LOADS; ++u) acc += v[u];
        }
      } else {
        for (int k = 0; k < n; ++k) {
          const int jk = __shfl_sync(0xffffffffu, j, k);
          acc += (col && jk >= 0) ? __ldg(xl + static_cast<int64_t>(jk) * ldx) : 0.0;
        }
      }
    }
    if (col) {
      if (rs >= c_beg && re <= c_end) {
        y[r * ldy + lane] = acc;
      } else {
        if (rs < c_beg) first[g * w + lane] = acc;
        if (re > c_end) last[g * w + lane] = acc;
      }
    }
    p = seg_end;
  }
}

__global__ void __launch_bounds__(THREADS) spmm_fixup_kernel(const int64_t* __restrict__ indptr, int64_t rows, int64_t nnz, int w,
                                                             double* __restrict__ y, int64_t ldy, const double* __restrict__ first,
                                                             const double* __restrict__ last, int32_t* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  const int64_t r = static_cast<int64_t>(blockIdx.x) * WARPS + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int64_t rs = indptr[r], re = indptr[r + 1];
  const bool bad = rs < 0 || re < rs || re > nnz || (r == 0 && rs != 0) || (r == rows - 1 && re != nnz);
  if (bad && lane == 0) atomicOr(status, SDRM_SPMM_BAD_INDPTR);
  if (lane >= w) return;
  double* out = y + r * ldy + lane;
  if (bad || re == rs) {
    *out = 0.0;
    return;
  }
  const int64_t c0 = rs / CHUNK, c1 = (re - 1) / CHUNK;
  if (c0 == c1) return;                    // written by the chunk pass
  double acc = last[c0 * w + lane];
  for (int64_t c = c0 + 1; c <= c1; ++c) acc += first[c * w + lane];
  *out = acc;
}

}  // namespace sdrm_spmm

using namespace sdrm_spmm;

extern "C" {

size_t sdrm_spmm_binary_workspace_bytes(int64_t nnz, int w) {
  if (w < 1 || w > 32) return 0;
  return static_cast<size_t>(n_chunks(nnz)) * 2u * static_cast<size_t>(w) * sizeof(double);
}

int sdrm_spmm_binary(const int64_t* d_indptr, const int32_t* d_indices, int64_t rows, int64_t nnz, const double* d_x, int64_t n_x,
                     int w, int64_t ldx, double* d_y, int64_t ldy, int32_t* d_status, void* d_workspace, size_t workspace_bytes,
                     void* stream) {
  char msg[224];
  if (rows < 0 || nnz < 0 || n_x < 0 || w < 1 || ldx < w || ldy < w) {
    snprintf(msg, sizeof msg, "sdrm_spmm_binary: bad shape (rows = %lld, nnz = %lld, n_x = %lld, w = %d, ldx = %lld, ldy = %lld)",
             static_cast<long long>(rows), static_cast<long long>(nnz), static_cast<long long>(n_x), w,
             static_cast<long long>(ldx), static_cast<long long>(ldy));
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  if (w > 32) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_spmm_binary: w > 32");
  if (rows == 0 && nnz > 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_spmm_binary: nnz > 0 with rows = 0");
  if (rows == 0) return SDRM_OK;
  if (!d_indptr || !d_y || !d_status || (nnz > 0 && (!d_indices || !d_x)))
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_spmm_binary: null pointer (d_indptr / d_indices / d_x / d_y / d_status)");
  const size_t need = sdrm_spmm_binary_workspace_bytes(nnz, w);
  if (need > 0 && !d_workspace) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_spmm_binary: null pointer (d_workspace)");
  if (workspace_bytes < need)
    return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_spmm_binary: workspace smaller than sdrm_spmm_binary_workspace_bytes(nnz, w)");
  const int64_t chunks = n_chunks(nnz);
  const int64_t chunk_blocks = (chunks + WARPS - 1) / WARPS, row_blocks = (rows + WARPS - 1) / WARPS;
  if (chunk_blocks > 0x7fffffffLL || row_blocks > 0x7fffffffLL)
    return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_spmm_binary: too many rows or entries for one launch");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  double* first = static_cast<double*>(d_workspace);
  double* last = first + chunks * w;
  if (chunks > 0) {
    spmm_chunk_kernel<<<static_cast<unsigned>(chunk_blocks), THREADS, 0, s>>>(d_indptr, d_indices, rows, nnz, d_x, n_x, w, ldx, d_y,
                                                                               ldy, first, last, d_status);
    SDRM_CUDA(cudaGetLastError());
  }
  spmm_fixup_kernel<<<static_cast<unsigned>(row_blocks), THREADS, 0, s>>>(d_indptr, rows, nnz, w, d_y, ldy, first, last, d_status);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

}  // extern "C"
