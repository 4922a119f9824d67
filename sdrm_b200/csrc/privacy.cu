// K8 — nearest rows by Jaccard similarity between two binary row sets (the distance-to-closest-record audit of synthetic
// rows against the real rows the generator was trained on).
//
//   c = |q & r| for every (query, reference) pair is an integer matrix product of the 0/1 operand images: tcgen05.mma
//   kind::i8 (u8 x u8 -> s32 in TMEM), exact because counts are integers <= n_items.  The per-row top-k by
//   J = c / u, u = a + b - c (a = |q|, b = |r|), is fused into the epilogue and compared exactly: c1 * u2 > c2 * u1 in 64 bits.
//
// Operand images: uint8 0/1, K-major, row pitch a multiple of 128 bytes with zero padding (prep kernels below), loaded with TMA
// in 128B-swizzled k-blocks of 128 columns (4 UMMAs of K = 32 each).
//
// Structure (K5's pipeline on one CTA): a CTA owns 128 query rows (TMEM lane = query row) and a contiguous range of reference
// tiles of 256 rows.  warp 0 = TMA producer, warp 1 = UMMA issuer + TMEM allocation, warps 2-9 = epilogue (two per TMEM lane
// quarter, alternating 16-column groups); two 256-column accumulators so the epilogue of tile j overlaps the UMMAs of tile j+1.
// Each epilogue thread keeps the running top-k of its query row over its column groups in registers; the per-pair path is
// u = a + b - c and one cross-multiplied compare against the current k-th entry, insertion is rare.  When there are fewer
// query tiles than SMs, the reference tiles are split over several CTAs per query tile.  Every (CTA, epilogue warp) writes a
// partial list; a merge kernel combines them by (J desc, index asc), so the result does not depend on the split.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/sdrm_b200.h"
#include "host_util.h"
#include "ptx_sm100.cuh"

namespace sdrm_priv {

using namespace sdrm;

constexpr int BM = 128;                 // query rows per CTA (UMMA M, TMEM lanes)
constexpr int BN = 256;                 // reference rows per tile (UMMA N)
constexpr int KB = 128;                 // columns (bytes) per k-block: one 128-byte swizzle row
constexpr int NSTG = 4;
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 64 + 32 * EPI_WARPS;
constexpr int LISTS_PER_CTA = EPI_WARPS / 4;   // partial lists per query row and CTA (one per epilogue warp of a quarter)
constexpr uint32_t A_BYTES = BM * KB;
constexpr uint32_t B_BYTES = BN * KB;
constexpr uint32_t STG_BYTES = A_BYTES + B_BYTES;
constexpr uint32_t SCRATCH_BYTES = EPI_WARPS * 32 * 16 * 4;   // counts of a 16-column group, for the rare insertion path
constexpr int SMEM_BYTES = NSTG * STG_BYTES + SCRATCH_BYTES + 1024 + 256;
constexpr int MAX_K = 16;
constexpr int MAX_ITEMS = 1 << 20;
enum : int { WD_P_PRODUCER = 801, WD_P_MMA_FULL = 802, WD_P_MMA_ACC = 803, WD_P_EPI = 804 };

struct Entry {   // one neighbour of a partial list: 16 bytes so a list entry is one vector store
  int idx, c, u, pad;
};

struct Params {
  CUtensorMap tmQ;            // dims {pitch, n}, box {128, 128}
  CUtensorMap tmR;            // dims {pitch, m}, box {128, 256}
  const int* q_ones;
  const int* r_ones;          // 16-byte aligned
  int n, m, kblocks;
  int r_tiles, tiles_per_split, splits;
  long long q_offset;         // global index of query row 0 (exclusion)
  int exclude;
  Entry* partial;             // [splits * LISTS_PER_CTA, n, K]
  int* err_word;
};

// (c1, u1) has the strictly higher J than (c2, u2); u >= 1 on real entries, a sentinel is (-1, 0) and loses to every one
__device__ __forceinline__ bool j_greater(int c1, int u1, int c2, int u2) {
  return static_cast<long long>(c1) * u2 > static_cast<long long>(c2) * u1;
}

// a candidate known to beat li/lc/lu[K - 1] goes in after the entries it does not beat (they hold lower indices on ties)
template <int K>
__device__ __forceinline__ void list_insert(int (&li)[K], int (&lc)[K], int (&lu)[K], int idx, int c, int u) {
  bool placed = false;
#pragma unroll
  for (int i = K - 1; i > 0; --i) {
    if (!placed) {
      if (j_greater(c, u, lc[i - 1], lu[i - 1])) {
        li[i] = li[i - 1]; lc[i] = lc[i - 1]; lu[i] = lu[i - 1];
      } else {
        li[i] = idx; lc[i] = c; lu[i] = u;
        placed = true;
      }
    }
  }
  if (!placed) { li[0] = idx; lc[0] = c; lu[0] = u; }
}

template <int K>
__global__ void __launch_bounds__(THREADS, 1) nearest_kernel(const __grid_constant__ Params P) {
  extern __shared__ uint8_t sm_raw[];
  const uint32_t raw_addr = smem_u32(sm_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  const uint32_t scratch_addr = base + NSTG * STG_BYTES;
  const uint32_t bar_base = scratch_addr + SCRATCH_BYTES;
  auto a_addr = [&](uint32_t s) { return base + s * STG_BYTES; };
  auto b_addr = [&](uint32_t s) { return base + s * STG_BYTES + A_BYTES; };
  auto bar_full = [&](uint32_t s) { return bar_base + 8u * s; };
  auto bar_empty = [&](uint32_t s) { return bar_base + 8u * (NSTG + s); };
  auto bar_acc_full = [&](uint32_t b) { return bar_base + 8u * (2 * NSTG + b); };
  auto bar_acc_empty = [&](uint32_t b) { return bar_base + 8u * (2 * NSTG + 2 + b); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(sm_raw + (bar_base - raw_addr) + 8 * (2 * NSTG + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  int* err = P.err_word;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < NSTG; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_acc_full(b), 1);
      mbar_init(bar_acc_empty(b), EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int qt = blockIdx.x / P.splits;
  const int split = blockIdx.x % P.splits;
  const int t0 = split * P.tiles_per_split;
  const int t1 = min(P.r_tiles, t0 + P.tiles_per_split);

  if (warp == 0) {
    // ================================ TMA producer ================================
    const uint64_t pol = l2_policy_evict_last();
    uint32_t stage = 0, sphase = 0;
    for (int t = t0; t < t1; ++t) {
      for (int kb = 0; kb < P.kblocks; ++kb) {
        mbar_wait(bar_empty(stage), sphase ^ 1u, err, WD_P_PRODUCER);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_full(stage), STG_BYTES);   // rows past n / m are zero-filled and still counted
          tma_load_2d_hint(a_addr(stage), &P.tmQ, kb * KB, qt * BM, bar_full(stage), pol);
          tma_load_2d_hint(b_addr(stage), &P.tmR, kb * KB, t * BN, bar_full(stage), pol);
        }
        __syncwarp();
        if (++stage == NSTG) { stage = 0; sphase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ================================ UMMA issuer ================================
    uint32_t stage = 0, sphase = 0, cc = 0;
    constexpr uint32_t idesc = umma_idesc_u8(BM, BN);
    for (int t = t0; t < t1; ++t, ++cc) {
      const uint32_t buf = cc & 1u;
      mbar_wait(bar_acc_empty(buf), ((cc >> 1) & 1u) ^ 1u, err, WD_P_MMA_ACC);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + buf * BN;
      for (int kb = 0; kb < P.kblocks; ++kb) {
        mbar_wait(bar_full(stage), sphase, err, WD_P_MMA_FULL);
        tc_fence_after();
        const uint64_t ad = umma_desc_sw128(a_addr(stage)), bd = umma_desc_sw128(b_addr(stage));
        if (elect_one()) {
          // +32 B along K inside the swizzle row = +2 in the 16-byte address field
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) umma_u8_ss(d_tmem, ad + 2u * k, bd + 2u * k, idesc, (kb > 0) | k);
          umma_commit(bar_empty(stage));
        }
        __syncwarp();
        if (++stage == NSTG) { stage = 0; sphase ^= 1u; }
      }
      if (elect_one()) umma_commit(bar_acc_full(buf));
      __syncwarp();
    }
  } else {
    // ================================ epilogue warps ================================
    const int q = warp & 3;                  // TMEM lane quarter this warp may read
    const int sub = (warp - 2) >> 2;         // owns the column groups g = sub (mod 2)
    const int r = q * 32 + lane;
    const int row = qt * BM + r;
    const bool row_ok = row < P.n;
    const int a = row_ok ? __ldg(P.q_ones + row) : 1;
    const long long qg = P.q_offset + row;   // global index of this query row
    const int self = (P.exclude && qg >= 0 && qg < P.m) ? static_cast<int>(qg) : -1;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    // this thread's slots of the scratch area: [e][thread] so the rare path's stores and loads are conflict-free
    int* scratch = reinterpret_cast<int*>(sm_raw + (scratch_addr - raw_addr)) + (warp - 2) * 32 * 16 + lane;

    int li[K], lc[K], lu[K];
#pragma unroll
    for (int i = 0; i < K; ++i) { li[i] = -1; lc[i] = -1; lu[i] = 0; }

    uint32_t cc = 0;
    for (int t = t0; t < t1; ++t, ++cc) {
      const uint32_t buf = cc & 1u;
      const int r_end = min(P.m, (t + 1) * BN);
      mbar_wait(bar_acc_full(buf), (cc >> 1) & 1u, err, WD_P_EPI);
      tc_fence_after();
      const uint32_t t_tile = tmem_base + lane_addr + buf * BN;
      uint32_t v[16];
      tmem_ld16(t_tile + sub * 16u, v);
      for (int g = sub; g < BN / 16; g += 2) {
        const int col0 = t * BN + g * 16;
        __syncwarp();
        tmem_ld_wait();
        int cv[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) cv[e] = static_cast<int>(v[e]);
        if (g + 2 < BN / 16 && col0 + 32 < r_end) tmem_ld16(t_tile + (g + 2) * 16u, v);   // (warp-uniform condition)
        if (col0 >= r_end) break;
        if (!row_ok) continue;   // (rows past n: the warp reconverges at the loop head before the next collective load)
        const bool full = col0 + 16 <= r_end;
        const bool fast = full && a > 0 && static_cast<unsigned>(self - col0) >= 16u;
        uint32_t mask = 0;
        if (fast) {
          int b[16];
          const int4* bp = reinterpret_cast<const int4*>(P.r_ones + col0);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int4 w = __ldg(bp + j);
            b[4 * j] = w.x; b[4 * j + 1] = w.y; b[4 * j + 2] = w.z; b[4 * j + 3] = w.w;
          }
          const int kc = lc[K - 1], ku = lu[K - 1];
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const int u = a + b[e] - cv[e];
            if (j_greater(cv[e], u, kc, ku)) mask |= 1u << e;
          }
        } else {
          mask = (1u << min(16, r_end - col0)) - 1u;   // ragged tile end, the excluded column or an empty query row:
          if (static_cast<unsigned>(self - col0) < 16u) mask &= ~(1u << (self - col0));   // every column is re-tested below
        }
        if (mask) {
#pragma unroll
          for (int e = 0; e < 16; ++e) scratch[e * 32] = cv[e];
          while (mask) {
            const int e = __ffs(mask) - 1;
            mask &= mask - 1u;
            const int c = scratch[e * 32];
            const int b = __ldg(P.r_ones + col0 + e);
            // an empty query row: c = 0 and J = 1 against an empty reference row, else 0 (kept as (1, 1) or (0, b))
            const int cj = a > 0 ? c : (b == 0 ? 1 : 0);
            const int uj = a > 0 ? a + b - c : max(b, 1);
            if (j_greater(cj, uj, lc[K - 1], lu[K - 1])) list_insert<K>(li, lc, lu, col0 + e, cj, uj);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty(buf));
    }
    if (row_ok) {
      Entry* out = P.partial + (static_cast<long long>(split * LISTS_PER_CTA + sub) * P.n + row) * K;
#pragma unroll
      for (int i = 0; i < K; ++i) out[i] = Entry{li[i], lc[i], lu[i], 0};
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// Merge the partial lists of every query row: (J desc, index asc); then the first k entries with the raw counts
template <int K>
__global__ void merge_kernel(const Entry* __restrict__ partial, int lists, int n, int k, const int* __restrict__ q_ones,
                             const int* __restrict__ r_ones, int64_t* __restrict__ idx_out, int* __restrict__ inter_out,
                             int* __restrict__ union_out) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  int li[K], lc[K], lu[K];
#pragma unroll
  for (int i = 0; i < K; ++i) { li[i] = -1; lc[i] = -1; lu[i] = 0; }
  for (int p = 0; p < lists; ++p) {
    const Entry* src = partial + (static_cast<long long>(p) * n + row) * K;
    for (int i = 0; i < K; ++i) {
      const Entry x = src[i];
      if (x.idx < 0) break;   // sentinels only follow
      // x beats the k-th entry: higher J, or equal J and a lower index (a sentinel k-th entry loses to any x)
      const long long l = static_cast<long long>(x.c) * lu[K - 1], rr = static_cast<long long>(lc[K - 1]) * x.u;
      if (!(l > rr || (l == rr && (li[K - 1] < 0 || x.idx < li[K - 1])))) continue;
      bool placed = false;
#pragma unroll
      for (int j = K - 1; j > 0; --j) {
        if (!placed) {
          const long long l2 = static_cast<long long>(x.c) * lu[j - 1], r2 = static_cast<long long>(lc[j - 1]) * x.u;
          if (l2 > r2 || (l2 == r2 && (li[j - 1] < 0 || x.idx < li[j - 1]))) {
            li[j] = li[j - 1]; lc[j] = lc[j - 1]; lu[j] = lu[j - 1];
          } else {
            li[j] = x.idx; lc[j] = x.c; lu[j] = x.u;
            placed = true;
          }
        }
      }
      if (!placed) { li[0] = x.idx; lc[0] = x.c; lu[0] = x.u; }
    }
  }
  const int a = q_ones[row];
#pragma unroll
  for (int i = 0; i < K; ++i) {
    if (i < k) {
      const long long o = static_cast<long long>(row) * k + i;
      const int j = li[i];
      idx_out[o] = j;
      // an empty query row kept (J numerator, denominator) = (b == 0, max(b, 1)); its true counts are c = 0, u = b
      inter_out[o] = j < 0 ? 0 : (a > 0 ? lc[i] : 0);
      union_out[o] = j < 0 ? 0 : (a > 0 ? lu[i] : r_ones[j]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// operand images
// ---------------------------------------------------------------------------------------------------------------------
constexpr int PREP_THREADS = 128;

__device__ __forceinline__ int block_sum(int v, int* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  int s = 0;
  for (int w = 0; w < PREP_THREADS / 32; ++w) s += red[w];
  return s;
}

// 4 bits -> 4 bytes of 0/1
__device__ __forceinline__ uint32_t nibble_bytes(uint32_t x) {
  return (x & 1u) | ((x & 2u) << 7) | ((x & 4u) << 14) | ((x & 8u) << 21);
}

__global__ void __launch_bounds__(PREP_THREADS) bits_image_kernel(const uint32_t* __restrict__ words, long long words_ld,
                                                                  int n_cols, uint8_t* __restrict__ image, long long pitch,
                                                                  int* __restrict__ ones) {
  __shared__ int red[PREP_THREADS / 32];
  const long long row = blockIdx.x;
  const int wpr = (n_cols + 31) >> 5;
  const int wpitch = static_cast<int>(pitch >> 5);
  int cnt = 0;
  for (int w = threadIdx.x; w < wpitch; w += PREP_THREADS) {
    uint32_t x = 0;
    if (w < wpr) {
      x = words[row * words_ld + w];
      const int valid = n_cols - 32 * w;   // bits past n_cols are not columns, whatever the caller left there
      if (valid < 32) x &= (1u << valid) - 1u;
    }
    cnt += __popc(x);
    uint4* dst = reinterpret_cast<uint4*>(image + row * pitch + 32ll * w);
    dst[0] = make_uint4(nibble_bytes(x), nibble_bytes(x >> 4), nibble_bytes(x >> 8), nibble_bytes(x >> 12));
    dst[1] = make_uint4(nibble_bytes(x >> 16), nibble_bytes(x >> 20), nibble_bytes(x >> 24), nibble_bytes(x >> 28));
  }
  const int s = block_sum(cnt, red);
  if (threadIdx.x == 0) ones[row] = s;
}

__global__ void __launch_bounds__(PREP_THREADS) csr_image_kernel(const int64_t* __restrict__ indptr,
                                                                 const int64_t* __restrict__ indices,
                                                                 const float* __restrict__ values, long long nnz, int n_cols,
                                                                 uint8_t* __restrict__ image, long long pitch,
                                                                 int* __restrict__ ones, int* __restrict__ status) {
  __shared__ int red[PREP_THREADS / 32];
  const long long row = blockIdx.x;
  uint8_t* dst = image + row * pitch;
  for (long long o = 16ll * threadIdx.x; o < pitch; o += 16ll * PREP_THREADS) *reinterpret_cast<uint4*>(dst + o) = make_uint4(0, 0, 0, 0);
  __syncthreads();
  long long s = indptr[row], e = indptr[row + 1];
  if (s < 0 || e < s || e > nnz) {
    if (threadIdx.x == 0) atomicOr(status, SDRM_PRIVACY_BAD_INDPTR);
    s = e = 0;
  }
  for (long long p = s + threadIdx.x; p < e; p += PREP_THREADS) {
    const long long j = indices[p];
    if (j < 0 || j >= n_cols) atomicOr(status, SDRM_PRIVACY_BAD_INDEX);
    else if (!values || values[p] != 0.0f) dst[j] = 1;   // explicit stored zeros are not interactions; duplicates set the same byte
  }
  __syncthreads();
  int cnt = 0;
  for (long long o = 4ll * threadIdx.x; o < pitch; o += 4ll * PREP_THREADS) cnt += __popc(*reinterpret_cast<const uint32_t*>(dst + o));
  const int sum = block_sum(cnt, red);
  if (threadIdx.x == 0) ones[row] = sum;
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
static_assert(KB == 128, "make_u8_map (host_util.h) loads boxes of 128 columns");

static int k_lists(int k) { return k <= 1 ? 1 : k <= 2 ? 2 : k <= 4 ? 4 : k <= 8 ? 8 : 16; }

// Reference tiles per query tile and CTA: one CTA per SM (the two accumulators take all 512 TMEM columns), so pick the split
// that minimises waves x (tiles per CTA + 1), the +1 standing for a CTA's fixed cost (set-up, pipeline fill, list write).
static int auto_splits(int q_tiles, int r_tiles, int sms) {
  int best = 1;
  long long best_cost = -1;
  for (int s = 1; s <= r_tiles; ++s) {
    const int tps = (r_tiles + s - 1) / s;
    if ((r_tiles + tps - 1) / tps != s) continue;   // only splits whose every part is non-empty
    const long long waves = (static_cast<long long>(q_tiles) * s + sms - 1) / sms;
    const long long cost = waves * (tps + 1);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = s; }
  }
  return best;
}

static int resolve_splits(int64_t n, int64_t m, int splits, int* out) {
  const int q_tiles = static_cast<int>((n + BM - 1) / BM), r_tiles = static_cast<int>((m + BN - 1) / BN);
  if (splits < 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy: splits must be >= 0");
  if (splits == 0) {
    int dev = 0, sms = 0;
    SDRM_CUDA(cudaGetDevice(&dev));
    SDRM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    splits = auto_splits(q_tiles, r_tiles, sms);
  }
  splits = splits > r_tiles ? r_tiles : splits;
  const int tps = (r_tiles + splits - 1) / splits;
  *out = (r_tiles + tps - 1) / tps;
  return SDRM_OK;
}

constexpr size_t WS_HEADER = 256;   // watchdog word

template <int K>
static int launch(const Params& P, int q_tiles, int k, const int* q_ones, const int* r_ones, int64_t* idx_out, int* inter_out,
                  int* union_out, cudaStream_t st) {
  static bool attr_done[64] = {false};
  int dev = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (!(dev < 64 && attr_done[dev])) {
    SDRM_CUDA(cudaFuncSetAttribute(nearest_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    if (dev < 64) attr_done[dev] = true;
  }
  nearest_kernel<K><<<static_cast<unsigned>(q_tiles * P.splits), THREADS, SMEM_BYTES, st>>>(P);
  SDRM_CUDA(cudaGetLastError());
  merge_kernel<K><<<static_cast<unsigned>((P.n + 127) / 128), 128, 0, st>>>(P.partial, P.splits * LISTS_PER_CTA, P.n, k, q_ones,
                                                                               r_ones, idx_out, inter_out, union_out);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

}  // namespace sdrm_priv

extern "C" {

int64_t sdrm_privacy_image_pitch(int n_items) {
  if (n_items < 1) return 0;
  return (static_cast<int64_t>(n_items) + 127) / 128 * 128;
}

int sdrm_privacy_image_bits(const uint32_t* d_words, int64_t words_ld, int64_t rows, int n_cols, uint8_t* d_image, int64_t pitch,
                            int32_t* d_ones, void* stream) {
  using namespace sdrm_priv;
  if ((rows > 0 && (!d_words || !d_image || !d_ones)) || rows < 0 || n_cols < 1 || words_ld < (n_cols + 31) / 32)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_image_bits: null pointer or bad shape");
  if (n_cols > MAX_ITEMS) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_privacy_image_bits: n_cols above 2^20");
  if (pitch != sdrm_privacy_image_pitch(n_cols) || (reinterpret_cast<uintptr_t>(d_image) & 15))
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_image_bits: pitch must be sdrm_privacy_image_pitch(n_cols), image 16-byte aligned");
  if (rows > 0x7FFFFFFFLL) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_privacy_image_bits: more than 2^31 - 1 rows");
  if (rows == 0) return SDRM_OK;
  bits_image_kernel<<<static_cast<unsigned>(rows), PREP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(d_words, words_ld, n_cols,
                                                                                                         d_image, pitch, d_ones);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_privacy_image_csr(const int64_t* d_indptr, const int64_t* d_indices, const float* d_values, int64_t nnz, int64_t rows,
                           int n_cols, uint8_t* d_image, int64_t pitch, int32_t* d_ones, int32_t* d_status, void* stream) {
  using namespace sdrm_priv;
  if ((rows > 0 && (!d_indptr || !d_image || !d_ones || !d_status)) || (nnz > 0 && !d_indices) || rows < 0 || nnz < 0 || n_cols < 1)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_image_csr: null pointer or bad shape");
  if (n_cols > MAX_ITEMS) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_privacy_image_csr: n_cols above 2^20");
  if (pitch != sdrm_privacy_image_pitch(n_cols) || (reinterpret_cast<uintptr_t>(d_image) & 15))
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_image_csr: pitch must be sdrm_privacy_image_pitch(n_cols), image 16-byte aligned");
  if (rows > 0x7FFFFFFFLL) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_privacy_image_csr: more than 2^31 - 1 rows");
  if (rows == 0) return SDRM_OK;
  csr_image_kernel<<<static_cast<unsigned>(rows), PREP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      d_indptr, d_indices, d_values, nnz, n_cols, d_image, pitch, d_ones, d_status);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

size_t sdrm_privacy_workspace_bytes(int64_t n, int64_t m, int k, int splits) {
  using namespace sdrm_priv;
  if (n < 1 || m < 1 || k < 1 || k > MAX_K) return 0;
  int s = 0;
  if (resolve_splits(n, m, splits, &s)) return 0;
  return WS_HEADER + static_cast<size_t>(s) * LISTS_PER_CTA * static_cast<size_t>(n) * k_lists(k) * sizeof(Entry);
}

int sdrm_privacy_nearest(const uint8_t* d_q_image, const int32_t* d_q_ones, int64_t n, const uint8_t* d_r_image,
                         const int32_t* d_r_ones, int64_t m, int n_items, int64_t pitch, int k, int exclude_same_index,
                         int64_t q_index_offset, int splits, int64_t* d_idx_out, int32_t* d_inter_out, int32_t* d_union_out,
                         void* d_workspace, size_t workspace_bytes, void* stream) {
  using namespace sdrm_priv;
  if (!d_q_image || !d_q_ones || !d_r_image || !d_r_ones || !d_idx_out || !d_inter_out || !d_union_out || !d_workspace)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_nearest: null pointer");
  if (n < 1 || m < 1 || n_items < 1 || q_index_offset < 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_nearest: bad shape");
  if (n_items > MAX_ITEMS) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_privacy_nearest: n_items above 2^20");
  if (n > 0x7FFFFFFFLL - BM || m > 0x7FFFFFFFLL - BN) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_privacy_nearest: more than 2^31 - 257 rows");
  if (pitch != sdrm_privacy_image_pitch(n_items)) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_nearest: pitch must be sdrm_privacy_image_pitch(n_items)");
  if (k < 1 || k > MAX_K || k > m) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_privacy_nearest: k must be in [1, min(16, m)]");
  if ((reinterpret_cast<uintptr_t>(d_q_image) | reinterpret_cast<uintptr_t>(d_r_image) | reinterpret_cast<uintptr_t>(d_r_ones) |
       reinterpret_cast<uintptr_t>(d_workspace)) & 15)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_privacy_nearest: images, reference ones and workspace must be 16-byte aligned");
  { int wrc = sdrm::apply_watchdog_env(); if (wrc) return wrc; }
  int s = 0;
  { int rc = resolve_splits(n, m, splits, &s); if (rc) return rc; }
  const size_t need = sdrm_privacy_workspace_bytes(n, m, k, s);
  if (workspace_bytes < need) return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_privacy_nearest: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  Params P;
  { int rc = make_u8_map(&P.tmQ, d_q_image, n, pitch, BM); if (rc) return rc; }
  { int rc = make_u8_map(&P.tmR, d_r_image, m, pitch, BN); if (rc) return rc; }
  P.q_ones = d_q_ones;
  P.r_ones = d_r_ones;
  P.n = static_cast<int>(n);
  P.m = static_cast<int>(m);
  P.kblocks = static_cast<int>(pitch / KB);
  P.r_tiles = static_cast<int>((m + BN - 1) / BN);
  P.splits = s;
  P.tiles_per_split = (P.r_tiles + s - 1) / s;
  P.q_offset = q_index_offset;
  P.exclude = exclude_same_index ? 1 : 0;
  P.err_word = static_cast<int*>(d_workspace);
  P.partial = reinterpret_cast<Entry*>(static_cast<uint8_t*>(d_workspace) + WS_HEADER);
  SDRM_CUDA(cudaMemsetAsync(d_workspace, 0, WS_HEADER, st));
  const int q_tiles = static_cast<int>((n + BM - 1) / BM);
  switch (k_lists(k)) {
    case 1: return launch<1>(P, q_tiles, k, d_q_ones, d_r_ones, d_idx_out, d_inter_out, d_union_out, st);
    case 2: return launch<2>(P, q_tiles, k, d_q_ones, d_r_ones, d_idx_out, d_inter_out, d_union_out, st);
    case 4: return launch<4>(P, q_tiles, k, d_q_ones, d_r_ones, d_idx_out, d_inter_out, d_union_out, st);
    case 8: return launch<8>(P, q_tiles, k, d_q_ones, d_r_ones, d_idx_out, d_inter_out, d_union_out, st);
    default: return launch<16>(P, q_tiles, k, d_q_ones, d_r_ones, d_idx_out, d_inter_out, d_union_out, st);
  }
}

}  // extern "C"
