// K9 — pairwise item correlation of two binary row sets (the fidelity audit of synthetic rows against the real rows).
//
//   For one set with U users, item counts a_i and pair counts c_ij = |users holding i and j|, the phi coefficient (Pearson
//   correlation of the 0/1 item columns) is phi_ij = (U c_ij - a_i a_j) / (sqrt(v_i) sqrt(v_j)), v_i = a_i (U - a_i), and 0 when
//   an item is constant in the set (v = 0).  K9 returns, over the pairs i < j, the six fp64 sums of d^2 (d = phiR - phiS), phiR,
//   phiS, phiR^2, phiS^2 and phiR phiS; the I x I matrices are never stored.
//
// Operand images: item-major uint8 0/1 [items, pitch], pitch = sdrm_privacy_image_pitch(users) (K8's image rules with items as
// rows and users as columns), written by the two prep kernels below with the item and user popcounts.
//
// Structure (K8's pipeline): a persistent CTA walks the upper-triangle tiles of 128 x 128 items.  warp 0 = TMA producer (for
// each tile the real images' k-blocks of 128 users, then the synthetic ones), warp 1 = UMMA issuer + TMEM allocation
// (tcgen05.mma kind::i8, u8 x u8 -> s32, M = N = 128), warps 2-9 = epilogue.  TMEM holds two tiles x two sets x 128 columns, so
// the epilogue of tile t overlaps the products of the CTA's next tile.  Each tile's six partial sums go to a workspace slot
// indexed by tile; a one-block kernel adds the slots in a fixed order, so the result does not depend on the grid.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/sdrm_b200.h"
#include "host_util.h"
#include "ptx_sm100.cuh"

namespace sdrm_fid {

using namespace sdrm;

constexpr int BT = 128;                 // items per tile side (UMMA M = N, TMEM lanes)
constexpr int KB = 128;                 // users (bytes) per k-block: one 128-byte swizzle row
constexpr int NSTG = 6;
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 64 + 32 * EPI_WARPS;
constexpr uint32_t OP_BYTES = BT * KB;
constexpr uint32_t STG_BYTES = 2 * OP_BYTES;
constexpr uint32_t RED_BYTES = 2 * EPI_WARPS * 6 * 8;   // per-warp partial sums, double-buffered by tile parity
constexpr int SMEM_BYTES = NSTG * STG_BYTES + RED_BYTES + 1024 + 256;
constexpr int MAX_USERS = 1 << 20;
constexpr int MAX_ITEMS = 1 << 20;
constexpr int NSUMS = 6;
constexpr size_t WS_HEADER = 256;       // watchdog word
enum : int { WD_F_PRODUCER = 901, WD_F_MMA_FULL = 902, WD_F_MMA_ACC = 903, WD_F_EPI = 904 };
static_assert(KB == 128, "make_u8_map (host_util.h) loads boxes of 128 columns");

struct ItemStat {   // per item and set: a and 1 / sqrt(v) (0 for a constant item, so its phi is 0)
  double a_r, inv_r, a_s, inv_s;
};

struct Params {
  CUtensorMap tmR;            // real image:      dims {pitch_r, n_items}, box {128, 128}
  CUtensorMap tmS;            // synthetic image: dims {pitch_s, n_items}, box {128, 128}
  const ItemStat* stats;
  double u_r, u_s;
  int n_items, kb_r, kb_s, t_side, n_tiles;
  double* slots;              // [n_tiles, 6]
  int* err_word;
};

// the CTA's next upper-triangle tile: row ti holds the tiles tj = ti .. T - 1 (tiles numbered row by row)
__device__ __forceinline__ void tile_advance(int step, int T, int& ti, int& tj) {
  tj += step;
  while (tj >= T) { ++ti; tj = tj - T + ti; }
}

// phi of one set; the same instruction sequence for both sets, so identical sets give bit-identical phi.  The numerator is
// exact: U c and a_i a_j are integers below 2^41.
__device__ __forceinline__ double phi(double U, int c, double ai, double aj, double inv_i, double inv_j) {
  const double num = fma(U, static_cast<double>(c), -(ai * aj));
  return num * inv_i * inv_j;
}

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory"); }

__global__ void __launch_bounds__(THREADS, 1) pair_stats_kernel(const __grid_constant__ Params P) {
  extern __shared__ uint8_t sm_raw[];
  const uint32_t raw_addr = smem_u32(sm_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  const uint32_t red_addr = base + NSTG * STG_BYTES;
  const uint32_t bar_base = red_addr + RED_BYTES;
  auto a_addr = [&](uint32_t s) { return base + s * STG_BYTES; };
  auto b_addr = [&](uint32_t s) { return base + s * STG_BYTES + OP_BYTES; };
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
  const int T = P.t_side;
  const int G = static_cast<int>(gridDim.x);

  if (warp == 0) {
    // ================================ TMA producer ================================
    const uint64_t pol = l2_policy_evict_last();
    uint32_t stage = 0, sphase = 0;
    int ti = 0, tj = 0;
    tile_advance(blockIdx.x, T, ti, tj);
    for (int t = blockIdx.x; t < P.n_tiles; t += G) {
      for (int set = 0; set < 2; ++set) {
        const CUtensorMap* tm = set ? &P.tmS : &P.tmR;
        const int kbs = set ? P.kb_s : P.kb_r;
        for (int kb = 0; kb < kbs; ++kb) {
          mbar_wait(bar_empty(stage), sphase ^ 1u, err, WD_F_PRODUCER);
          if (elect_one()) {
            mbar_arrive_expect_tx(bar_full(stage), STG_BYTES);   // item rows past n_items are zero-filled (masked later)
            tma_load_2d_hint(a_addr(stage), tm, kb * KB, ti * BT, bar_full(stage), pol);
            tma_load_2d_hint(b_addr(stage), tm, kb * KB, tj * BT, bar_full(stage), pol);
          }
          __syncwarp();
          if (++stage == NSTG) { stage = 0; sphase ^= 1u; }
        }
      }
      if (t + G < P.n_tiles) tile_advance(G, T, ti, tj);
    }
  } else if (warp == 1) {
    // ================================ UMMA issuer ================================
    uint32_t stage = 0, sphase = 0, cc = 0;
    constexpr uint32_t idesc = umma_idesc_u8(BT, BT);
    for (int t = blockIdx.x; t < P.n_tiles; t += G, ++cc) {
      const uint32_t buf = cc & 1u;
      mbar_wait(bar_acc_empty(buf), ((cc >> 1) & 1u) ^ 1u, err, WD_F_MMA_ACC);
      tc_fence_after();
      for (int set = 0; set < 2; ++set) {
        const uint32_t d_tmem = tmem_base + buf * (2 * BT) + set * BT;
        const int kbs = set ? P.kb_s : P.kb_r;
        for (int kb = 0; kb < kbs; ++kb) {
          mbar_wait(bar_full(stage), sphase, err, WD_F_MMA_FULL);
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
      }
      if (elect_one()) umma_commit(bar_acc_full(buf));
      __syncwarp();
    }
  } else {
    // ================================ epilogue warps ================================
    const int ew = warp - 2;
    const int q = warp & 3;                  // TMEM lane quarter this warp may read
    const int sub = ew >> 2;                 // owns the column groups g = sub (mod 2)
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    double* red = reinterpret_cast<double*>(sm_raw + (red_addr - raw_addr));
    const double2* stats2 = reinterpret_cast<const double2*>(P.stats);
    int ti = 0, tj = 0;
    tile_advance(blockIdx.x, T, ti, tj);
    uint32_t cc = 0;
    for (int t = blockIdx.x; t < P.n_tiles; t += G, ++cc) {
      const uint32_t buf = cc & 1u;
      const int i = ti * BT + q * 32 + lane;
      const double2 si0 = __ldg(stats2 + 2 * min(i, P.n_items - 1)), si1 = __ldg(stats2 + 2 * min(i, P.n_items - 1) + 1);
      double s_dd = 0.0, s_r = 0.0, s_s = 0.0, s_rr = 0.0, s_ss = 0.0, s_rs = 0.0;
      mbar_wait(bar_acc_full(buf), (cc >> 1) & 1u, err, WD_F_EPI);
      tc_fence_after();
      const uint32_t t_tile = tmem_base + lane_addr + buf * (2 * BT);
      for (int g = sub; g < BT / 16; g += 2) {
        const int col0 = tj * BT + g * 16;
        if (col0 >= P.n_items) break;        // (warp-uniform)
        uint32_t vr[16], vs[16];
        tmem_ld16(t_tile + g * 16u, vr);
        tmem_ld16(t_tile + BT + g * 16u, vs);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const int j = col0 + e;
          const int jl = min(j, P.n_items - 1);
          const double2 sj0 = __ldg(stats2 + 2 * jl), sj1 = __ldg(stats2 + 2 * jl + 1);
          const double pr = phi(P.u_r, static_cast<int>(vr[e]), si0.x, sj0.x, si0.y, sj0.y);
          const double ps = phi(P.u_s, static_cast<int>(vs[e]), si1.x, sj1.x, si1.y, sj1.y);
          if (j > i && j < P.n_items) {      // pairs i < j only; zero-filled rows and columns past n_items never count
            const double d = pr - ps;
            s_dd = fma(d, d, s_dd);
            s_r += pr;
            s_s += ps;
            s_rr = fma(pr, pr, s_rr);
            s_ss = fma(ps, ps, s_ss);
            s_rs = fma(pr, ps, s_rs);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty(buf));
      double s[NSUMS] = {s_dd, s_r, s_s, s_rr, s_ss, s_rs};
#pragma unroll
      for (int k = 0; k < NSUMS; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
      }
      double* rb = red + buf * (EPI_WARPS * NSUMS);
      if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NSUMS; ++k) rb[ew * NSUMS + k] = s[k];
      }
      // (rb of this parity is rewritten two tiles later, after the next barrier, which its reader reaches only after reading)
      epi_bar();
      if (ew == 0 && lane < NSUMS) {
        double acc = 0.0;
        for (int w = 0; w < EPI_WARPS; ++w) acc += rb[w * NSUMS + lane];
        P.slots[static_cast<long long>(t) * NSUMS + lane] = acc;
      }
      if (t + G < P.n_tiles) tile_advance(G, T, ti, tj);
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

__global__ void item_stats_kernel(const int* __restrict__ a_r, const int* __restrict__ a_s, int u_r, int u_s, int n,
                                  ItemStat* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int ar = a_r[i], as = a_s[i];
  const long long vr = static_cast<long long>(ar) * (u_r - ar), vs = static_cast<long long>(as) * (u_s - as);
  out[i] = ItemStat{static_cast<double>(ar), vr > 0 ? 1.0 / sqrt(static_cast<double>(vr)) : 0.0, static_cast<double>(as),
                    vs > 0 ? 1.0 / sqrt(static_cast<double>(vs)) : 0.0};
}

// the tile slots added in a fixed order (strided per thread, then a fixed tree): the same bits for any grid of K9
constexpr int RED_THREADS = 256;
__global__ void __launch_bounds__(RED_THREADS) reduce_slots_kernel(const double* __restrict__ slots, long long n_tiles,
                                                                   double* __restrict__ out) {
  __shared__ double red[RED_THREADS];
  for (int k = 0; k < NSUMS; ++k) {
    double acc = 0.0;
    for (long long t = threadIdx.x; t < n_tiles; t += RED_THREADS) acc += slots[t * NSUMS + k];
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = RED_THREADS / 2; o > 0; o >>= 1) {
      if (static_cast<int>(threadIdx.x) < o) red[threadIdx.x] += red[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) out[k] = red[0];
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// item-major operand images
// ---------------------------------------------------------------------------------------------------------------------
constexpr int TP_WARPS = 8;                   // bits: a block = 32 * TP_WARPS users x TP_WORDS * 32 items
constexpr int TP_WORDS = 8;
constexpr int PREP_THREADS = 128;             // CSR: one block per user row / item row

// 4 bits -> 4 bytes of 0/1
__device__ __forceinline__ uint32_t nibble_bytes(uint32_t x) {
  return (x & 1u) | ((x & 2u) << 7) | ((x & 4u) << 14) | ((x & 8u) << 21);
}

__device__ __forceinline__ int block_sum(int v, int* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  int s = 0;
  for (int w = 0; w < PREP_THREADS / 32; ++w) s += red[w];
  return s;
}

// Bit-packed user rows -> item-major image.  Each warp reads one word (32 items) of 32 users and transposes the 32 x 32 bit
// block with 32 ballots: lane j then holds item 32 w + j's bits over the warp's users, written as 32 bytes of its image row.
// item_ones and user_ones are zeroed by the caller and collect one atomic add per block and item / user.
__global__ void __launch_bounds__(32 * TP_WARPS) bits_item_image_kernel(const uint32_t* __restrict__ words, long long words_ld,
                                                                        int users, int n_items, uint8_t* __restrict__ image,
                                                                        long long pitch, int* __restrict__ item_ones,
                                                                        int* __restrict__ user_ones) {
  __shared__ int red[TP_WARPS][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long u0 = static_cast<long long>(blockIdx.x) * (32 * TP_WARPS) + 32 * warp;   // this warp's first user
  const long long u = u0 + lane;
  const int wpr = (n_items + 31) >> 5;
  const int w0 = blockIdx.y * TP_WORDS, w1 = min(wpr, w0 + TP_WORDS);
  int ucnt = 0;
  for (int w = w0; w < w1; ++w) {
    uint32_t x = 0;
    if (u < users) {
      x = words[u * words_ld + w];
      const int valid = n_items - 32 * w;   // bits past n_items are not items, whatever the caller left there
      if (valid < 32) x &= (1u << valid) - 1u;
    }
    ucnt += __popc(x);
    uint32_t col = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const uint32_t b = __ballot_sync(0xffffffffu, (x >> j) & 1u);
      if (lane == j) col = b;
    }
    const int item = 32 * w + lane;
    if (u0 < pitch && item < n_items) {   // users past `users` are zero columns up to the pitch
      uint4* dst = reinterpret_cast<uint4*>(image + item * pitch + u0);
      dst[0] = make_uint4(nibble_bytes(col), nibble_bytes(col >> 4), nibble_bytes(col >> 8), nibble_bytes(col >> 12));
      dst[1] = make_uint4(nibble_bytes(col >> 16), nibble_bytes(col >> 20), nibble_bytes(col >> 24), nibble_bytes(col >> 28));
    }
    red[warp][lane] = __popc(col);
    __syncthreads();
    if (warp == 0) {
      int s = 0;
      for (int k = 0; k < TP_WARPS; ++k) s += red[k][lane];
      if (s && item < n_items) atomicAdd(item_ones + item, s);
    }
    __syncthreads();
  }
  if (ucnt) atomicAdd(user_ones + u, ucnt);
}

// CSR user rows -> item-major image (zeroed by the caller).  The first store of a (user, item) byte counts for the user: an
// atomic OR on the byte's word tells which store that was, so a repeated column counts once.
__global__ void __launch_bounds__(PREP_THREADS) csr_item_image_kernel(const int64_t* __restrict__ indptr,
                                                                      const int64_t* __restrict__ indices,
                                                                      const float* __restrict__ values, long long nnz,
                                                                      int n_items, uint8_t* __restrict__ image, long long pitch,
                                                                      int* __restrict__ user_ones, int* __restrict__ status) {
  __shared__ int red[PREP_THREADS / 32];
  const long long row = blockIdx.x;
  long long s = indptr[row], e = indptr[row + 1];
  if (s < 0 || e < s || e > nnz) {
    if (threadIdx.x == 0) atomicOr(status, SDRM_PRIVACY_BAD_INDPTR);
    s = e = 0;
  }
  uint32_t* col_word = reinterpret_cast<uint32_t*>(image + (row & ~3ll));
  const uint32_t bit = 1u << (8 * (row & 3));
  int cnt = 0;
  for (long long p = s + threadIdx.x; p < e; p += PREP_THREADS) {
    const long long j = indices[p];
    if (j < 0 || j >= n_items) atomicOr(status, SDRM_PRIVACY_BAD_INDEX);
    else if (!values || values[p] != 0.0f)   // explicit stored zeros are not interactions
      if (!(atomicOr(col_word + j * (pitch >> 2), bit) & bit)) ++cnt;
  }
  const int sum = block_sum(cnt, red);
  if (threadIdx.x == 0) user_ones[row] = sum;
}

__global__ void __launch_bounds__(PREP_THREADS) row_ones_kernel(const uint8_t* __restrict__ image, long long pitch,
                                                                int* __restrict__ ones) {
  __shared__ int red[PREP_THREADS / 32];
  const uint8_t* src = image + blockIdx.x * pitch;
  int cnt = 0;
  for (long long o = 16ll * threadIdx.x; o < pitch; o += 16ll * PREP_THREADS) {
    const uint4 v = *reinterpret_cast<const uint4*>(src + o);
    cnt += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
  }
  const int sum = block_sum(cnt, red);
  if (threadIdx.x == 0) ones[blockIdx.x] = sum;
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
static long long n_tiles_of(int n_items) {
  const long long T = (n_items + BT - 1) / BT;
  return T * (T + 1) / 2;
}

static size_t stats_bytes(int n_items) { return (static_cast<size_t>(n_items) * sizeof(ItemStat) + 255) / 256 * 256; }

static int check_image_args(const char* who, int64_t users, int n_items, const uint8_t* d_image, int64_t pitch) {
  char msg[160];
  if (users < 1 || users > MAX_USERS || n_items < 1 || n_items > MAX_ITEMS) {
    snprintf(msg, sizeof msg, "%s: users and n_items must lie in [1, 2^20]", who);
    return sdrm_fail(SDRM_ERR_UNSUPPORTED, msg);
  }
  if (pitch != sdrm_privacy_image_pitch(static_cast<int>(users)) || (reinterpret_cast<uintptr_t>(d_image) & 15)) {
    snprintf(msg, sizeof msg, "%s: pitch must be sdrm_privacy_image_pitch(users), image 16-byte aligned", who);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  return SDRM_OK;
}

}  // namespace sdrm_fid

extern "C" {

int sdrm_fidelity_item_image_bits(const uint32_t* d_words, int64_t words_ld, int64_t users, int n_items, uint8_t* d_image,
                                  int64_t pitch, int32_t* d_item_ones, int32_t* d_user_ones, void* stream) {
  using namespace sdrm_fid;
  if (!d_words || !d_image || !d_item_ones || !d_user_ones || words_ld < (static_cast<int64_t>(n_items) + 31) / 32)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_fidelity_item_image_bits: null pointer or words_ld below the words of a row");
  { int rc = check_image_args("sdrm_fidelity_item_image_bits", users, n_items, d_image, pitch); if (rc) return rc; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaMemsetAsync(d_item_ones, 0, sizeof(int32_t) * n_items, st));
  SDRM_CUDA(cudaMemsetAsync(d_user_ones, 0, sizeof(int32_t) * users, st));
  const int wpr = (n_items + 31) / 32;
  const dim3 grid(static_cast<unsigned>((pitch + 32 * TP_WARPS - 1) / (32 * TP_WARPS)), static_cast<unsigned>((wpr + TP_WORDS - 1) / TP_WORDS));
  bits_item_image_kernel<<<grid, 32 * TP_WARPS, 0, st>>>(d_words, words_ld, static_cast<int>(users), n_items, d_image, pitch,
                                                         d_item_ones, d_user_ones);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_fidelity_item_image_csr(const int64_t* d_indptr, const int64_t* d_indices, const float* d_values, int64_t nnz,
                                 int64_t users, int n_items, uint8_t* d_image, int64_t pitch, int32_t* d_item_ones,
                                 int32_t* d_user_ones, int32_t* d_status, void* stream) {
  using namespace sdrm_fid;
  if (!d_indptr || !d_image || !d_item_ones || !d_user_ones || !d_status || (nnz > 0 && !d_indices) || nnz < 0)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_fidelity_item_image_csr: null pointer or bad shape");
  { int rc = check_image_args("sdrm_fidelity_item_image_csr", users, n_items, d_image, pitch); if (rc) return rc; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaMemsetAsync(d_image, 0, static_cast<size_t>(n_items) * pitch, st));
  csr_item_image_kernel<<<static_cast<unsigned>(users), PREP_THREADS, 0, st>>>(d_indptr, d_indices, d_values, nnz, n_items, d_image,
                                                                                pitch, d_user_ones, d_status);
  SDRM_CUDA(cudaGetLastError());
  row_ones_kernel<<<static_cast<unsigned>(n_items), PREP_THREADS, 0, st>>>(d_image, pitch, d_item_ones);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

size_t sdrm_fidelity_workspace_bytes(int n_items) {
  using namespace sdrm_fid;
  if (n_items < 1 || n_items > MAX_ITEMS) return 0;
  return WS_HEADER + stats_bytes(n_items) + static_cast<size_t>(n_tiles_of(n_items)) * NSUMS * sizeof(double);
}

int sdrm_fidelity_pair_stats(const uint8_t* d_real_image, const int32_t* d_real_item_ones, int64_t real_users, int64_t real_pitch,
                             const uint8_t* d_synth_image, const int32_t* d_synth_item_ones, int64_t synth_users,
                             int64_t synth_pitch, int n_items, double* d_sums_out, void* d_workspace, size_t workspace_bytes,
                             void* stream) {
  using namespace sdrm_fid;
  if (!d_real_image || !d_real_item_ones || !d_synth_image || !d_synth_item_ones || !d_sums_out || !d_workspace)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_fidelity_pair_stats: null pointer");
  { int rc = check_image_args("sdrm_fidelity_pair_stats (real)", real_users, n_items, d_real_image, real_pitch); if (rc) return rc; }
  { int rc = check_image_args("sdrm_fidelity_pair_stats (synthetic)", synth_users, n_items, d_synth_image, synth_pitch); if (rc) return rc; }
  if ((reinterpret_cast<uintptr_t>(d_workspace) & 15) || (reinterpret_cast<uintptr_t>(d_sums_out) & 7))
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_fidelity_pair_stats: workspace must be 16-byte aligned, sums 8-byte aligned");
  if (workspace_bytes < sdrm_fidelity_workspace_bytes(n_items))
    return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_fidelity_pair_stats: workspace too small");
  { int wrc = sdrm::apply_watchdog_env(); if (wrc) return wrc; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  Params P;
  { int rc = make_u8_map(&P.tmR, d_real_image, n_items, real_pitch, BT); if (rc) return rc; }
  { int rc = make_u8_map(&P.tmS, d_synth_image, n_items, synth_pitch, BT); if (rc) return rc; }
  uint8_t* ws = static_cast<uint8_t*>(d_workspace);
  ItemStat* stats = reinterpret_cast<ItemStat*>(ws + WS_HEADER);
  P.stats = stats;
  P.u_r = static_cast<double>(real_users);
  P.u_s = static_cast<double>(synth_users);
  P.n_items = n_items;
  P.kb_r = static_cast<int>(real_pitch / KB);
  P.kb_s = static_cast<int>(synth_pitch / KB);
  P.t_side = (n_items + BT - 1) / BT;
  P.n_tiles = static_cast<int>(n_tiles_of(n_items));
  P.slots = reinterpret_cast<double*>(ws + WS_HEADER + stats_bytes(n_items));
  P.err_word = static_cast<int*>(d_workspace);

  static bool attr_done[64] = {false};
  int dev = 0, sms = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  SDRM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (!(dev < 64 && attr_done[dev])) {
    SDRM_CUDA(cudaFuncSetAttribute(pair_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    if (dev < 64) attr_done[dev] = true;
  }
  SDRM_CUDA(cudaMemsetAsync(d_workspace, 0, WS_HEADER, st));
  item_stats_kernel<<<static_cast<unsigned>((n_items + 255) / 256), 256, 0, st>>>(d_real_item_ones, d_synth_item_ones,
                                                                                   static_cast<int>(real_users),
                                                                                   static_cast<int>(synth_users), n_items, stats);
  SDRM_CUDA(cudaGetLastError());
  const int grid = P.n_tiles < sms ? P.n_tiles : sms;   // one CTA per SM: the four accumulators take all 512 TMEM columns
  pair_stats_kernel<<<static_cast<unsigned>(grid), THREADS, SMEM_BYTES, st>>>(P);
  SDRM_CUDA(cudaGetLastError());
  reduce_slots_kernel<<<1, RED_THREADS, 0, st>>>(P.slots, P.n_tiles, d_sums_out);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

}  // extern "C"
