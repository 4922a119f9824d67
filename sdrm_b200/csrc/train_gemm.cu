// Host side of K5: the dense products of the diffusion TRAINING step on the tcgen05 GEMM (gemm_x3_kernel.cuh).
//
// Reference: the three denoiser forwards of score_matching_loss and their autograd backward
// (train_SDRM.py:191-199, 331-337; SDRM.forward 97-103).  The three forwards are batched as one [rows = 3B, L] problem (rows
// are independent, so this is the same arithmetic), every Linear is one GEMM launch with its bias / PReLU / tanh fused into
// the epilogue, the backward is one data-gradient GEMM (PReLU' fused) and one split-K weight-gradient GEMM per layer; the
// shared hidden Linear (train_SDRM.py:94) accumulates its gradient over its nh applications in ONE slab reduction.
//
// Exports: sdrm_denoiser_train_workspace_bytes / sdrm_denoiser_fwd / sdrm_denoiser_bwd (SURVEY.md §8b) and the plain product
// sdrm_gemm (the three products of a Linear layer and its autograd: MultiVAE++ training step, unit tests).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "../../include/sdrm_b200.h"
#include "gemm_x3_kernel.cuh"
#include "host_util.h"

namespace sdrm {

// ------------------------------------------------------------------------------------------------
// operand preparation: fp32 matrix (optionally transformed) -> bf16 hi / lo images, row-major and / or transposed
// ------------------------------------------------------------------------------------------------
enum PrepMode : int { PREP_IDENT = 0, PREP_PRELU = 1, PREP_TANH_BWD = 2 };

struct PrepParams {
  const float* src; long long ld_src;      // [R, C]
  const float* src2; long long ld_src2;    // TANH_BWD: the tanh OUTPUT (v = src * (1 - src2^2))
  const float* slope;                      // PRELU: device scalar
  long long R; int C; int mode;
  __nv_bfloat16 *rm_hi, *rm_lo; long long ld_rm;   // [R, ld_rm] or nullptr
  __nv_bfloat16 *tr_hi, *tr_lo; long long ld_tr;   // [C, ld_tr] or nullptr
  double* colsum;                                   // [C], accumulated, or nullptr
};

// One block = a 64-row x 32-column tile.  Reads are coalesced along the columns, the transposed image is written from a
// shared-memory tile with bf16x2 stores coalesced along the (source) rows.  Rows >= R of the last tile are written as zeros
// into the transposed image (the GEMM's TMA zero-fills whatever lies beyond the logical extent anyway).
__global__ void __launch_bounds__(256) operand_prep_kernel(const PrepParams P) {
  __shared__ float tile[64][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long r0 = static_cast<long long>(blockIdx.y) * 64;
  const int c0 = blockIdx.x * 32;
  const int c = c0 + lane;
  const float slope = (P.mode == PREP_PRELU) ? __ldg(P.slope) : 0.0f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int rr = warp + 8 * i;
    const long long r = r0 + rr;
    float v = 0.0f;
    if (r < P.R && c < P.C) {
      v = P.src[r * P.ld_src + c];
      if (P.mode == PREP_PRELU) v = v > 0.0f ? v : slope * v;
      else if (P.mode == PREP_TANH_BWD) {
        const float o = P.src2[r * P.ld_src2 + c];
        v = v * (1.0f - o * o);
      }
      if (P.rm_hi) {
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        P.rm_hi[r * P.ld_rm + c] = h;
        P.rm_lo[r * P.ld_rm + c] = __float2bfloat16_rn(v - __bfloat162float(h));
      }
    }
    tile[rr][lane] = v;
  }
  __syncthreads();
  if (P.colsum) {
    // warp w sums columns 4w .. 4w+3 of the tile: lane l adds rows l and l + 32
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cc = 4 * warp + j;
      double s = static_cast<double>(tile[lane][cc]) + static_cast<double>(tile[lane + 32][cc]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0 && c0 + cc < P.C) atomicAdd(P.colsum + c0 + cc, s);
    }
  }
  if (P.tr_hi) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cc = warp + 8 * j;
      if (c0 + cc >= P.C) continue;
      const float v0 = tile[2 * lane][cc], v1 = tile[2 * lane + 1][cc];
      const float h0 = bf16_round(v0), h1 = bf16_round(v1);
      const long long off = static_cast<long long>(c0 + cc) * P.ld_tr + r0 + 2 * lane;
      if (r0 + 2 * lane + 1 < P.ld_tr) {
        *reinterpret_cast<uint32_t*>(P.tr_hi + off) = pack_bf16x2(h0, h1);
        *reinterpret_cast<uint32_t*>(P.tr_lo + off) = pack_bf16x2(v0 - h0, v1 - h1);
      }
    }
  }
}

// out[m, n] = sum_s slab[s][m, n]   (split-K partial products; also sums the nh applications of the shared hidden layer)
__global__ void slab_reduce_kernel(const float* __restrict__ slabs, long long slab_stride, int n_slabs, long long ld_slab, int M, int N,
                                   float* __restrict__ out, long long ld_out) {
  const long long total = static_cast<long long>(M) * N;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int m = static_cast<int>(i / N), n = static_cast<int>(i - static_cast<long long>(m) * N);
    float acc = 0.0f;
    for (int s = 0; s < n_slabs; ++s) acc += slabs[s * slab_stride + m * ld_slab + n];
    out[m * ld_out + n] = acc;
  }
}

// gTable[i, n] = sum over the rows r with t[r] == i of G0[r, n]  (gradient of the hoisted time-embedding bias rows).  The rows
// come bucketed by t (order / offsets from the host), so the sum is deterministic and every read is coalesced along n.
__global__ void table_grad_kernel(const float* __restrict__ G, long long ld_g, const long long* __restrict__ order,
                                  const long long* __restrict__ offsets, int D, float* __restrict__ out, long long ld_out) {
  const int i = blockIdx.x;
  const int n = blockIdx.y * blockDim.x + threadIdx.x;
  if (n >= D) return;
  float acc = 0.0f;
  for (long long p = offsets[i]; p < offsets[i + 1]; ++p) acc += G[order[p] * ld_g + n];
  out[i * ld_out + n] = acc;
}

__global__ void finish_sums_kernel(const double* __restrict__ src, int n, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = static_cast<float>(src[i]);
}

}  // namespace sdrm

using namespace sdrm;

static thread_local long long g_train_launches = 0;   // kernels of this file launched by the calling thread (bench bookkeeping)

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------
// bf16 matrix [rows, cols] with row pitch ld (elements, multiple of 8): box = 64 columns x box_rows rows, SWIZZLE_128B
static int make_bf16_map(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld, unsigned box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return sdrm_fail(SDRM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  const cuuint32_t box[2] = {64, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char msg[160];
    snprintf(msg, sizeof msg, "cuTensorMapEncodeTiled (bf16) failed (%d) rows=%lld cols=%lld ld=%lld box_rows=%u", static_cast<int>(r), rows, cols, ld, box_rows);
    return sdrm_fail(SDRM_ERR_CUDA, msg);
  }
  return SDRM_OK;
}

struct Bf16Mat {   // hi / lo images of one fp32 matrix
  __nv_bfloat16* hi = nullptr;
  __nv_bfloat16* lo = nullptr;
  long long rows = 0, cols = 0, ld = 0;
};


static int gemm_clusters(int* out) {
  { int wrc = apply_watchdog_env(); if (wrc) return wrc; }
  static int cached[64];
  static bool have[64] = {false};
  int dev = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && have[dev]) { *out = cached[dev]; return SDRM_OK; }
  SDRM_CUDA(cudaFuncSetAttribute(sdrm_gemm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  int sms = 0;
  SDRM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(sms / 2 * 2));
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = GEMM_SMEM_BYTES;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  int n = 0;
  SDRM_CUDA(cudaOccupancyMaxActiveClusters(&n, sdrm_gemm_pair_kernel, &cfg));
  if (n <= 0) return sdrm_fail(SDRM_ERR_CUDA, "gemm: no resident cluster");
  if (dev < 64) { cached[dev] = n; have[dev] = true; }
  *out = n;
  return SDRM_OK;
}

static int tile_width(int N, int* n_tiles) {
  *n_tiles = (N + 255) / 256;
  const int per = (N + *n_tiles - 1) / *n_tiles;
  return std::max(16, (per + 15) / 16 * 16);
}

// split-K factor of a weight-gradient product: enough work items to occupy the resident clusters
static int wgrad_splits(long long M, int N, long long K, int clusters) {
  int nt;
  tile_width(N, &nt);
  const long long tiles = ((M + 255) / 256) * nt;
  const long long kb = (K + 63) / 64;
  long long s = std::max<long long>(1, clusters / std::max<long long>(1, tiles));
  s = std::min<long long>(s, std::min<long long>(kb, 8));
  const long long per = (kb + s - 1) / s;
  return static_cast<int>((kb + per - 1) / per);
}

struct GemmCall {
  Bf16Mat A, B;            // A [M, K], B [N, K]
  float* C = nullptr; long long ldc = 0;
  int splits = 1; long long slab_stride = 0;
  const float* bias = nullptr;
  const float* bias_table = nullptr; const long long* bias_rows = nullptr; long long bias_ld = 0;
  int epi = GEMM_EPI_STORE;
  const float* slope = nullptr;
  Bf16Mat O;               // bf16 outputs
  const float* aux = nullptr; long long ld_aux = 0;
  double* slope_grad = nullptr;
  int passes = 3;
};

static int launch_gemm(const GemmCall& g, int* err_word, cudaStream_t st) {
  if (g.A.cols != g.B.cols) return sdrm_fail(SDRM_ERR_BAD_ARG, "gemm: K mismatch");
  GemmParams P;
  memset(&P, 0, sizeof P);
  P.M = static_cast<int>(g.A.rows); P.N = static_cast<int>(g.B.rows); P.K = static_cast<int>(g.A.cols);
  P.BN = tile_width(P.N, &P.n_tiles);
  P.m_tiles = (P.M + 255) / 256;
  P.kb_total = (P.K + 63) / 64;
  P.splits = std::max(1, std::min(g.splits, P.kb_total));
  P.kb_per_split = (P.kb_total + P.splits - 1) / P.splits;
  P.splits = (P.kb_total + P.kb_per_split - 1) / P.kb_per_split;
  P.passes = g.passes == 1 ? 1 : 3;
  int rc;
  if ((rc = make_bf16_map(&P.tmA[0], g.A.hi, g.A.rows, g.A.cols, g.A.ld, 128))) return rc;
  if ((rc = make_bf16_map(&P.tmA[1], g.A.lo, g.A.rows, g.A.cols, g.A.ld, 128))) return rc;
  if ((rc = make_bf16_map(&P.tmB[0], g.B.hi, g.B.rows, g.B.cols, g.B.ld, P.BN / 2))) return rc;
  if ((rc = make_bf16_map(&P.tmB[1], g.B.lo, g.B.rows, g.B.cols, g.B.ld, P.BN / 2))) return rc;
  P.C = g.C; P.ldc = g.ldc; P.slab_stride = g.slab_stride;
  P.bias = g.bias; P.bias_table = g.bias_table; P.bias_rows = g.bias_rows; P.bias_ld = g.bias_ld;
  P.epi = g.epi; P.slope = g.slope;
  P.o_hi = g.O.hi; P.o_lo = g.O.lo; P.ldo = g.O.ld;
  P.aux = g.aux; P.ld_aux = g.ld_aux; P.slope_grad = g.slope_grad;
  P.err_word = err_word;
  int clusters = 0;
  if ((rc = gemm_clusters(&clusters))) return rc;
  const long long work = static_cast<long long>(P.m_tiles) * P.n_tiles * P.splits;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(2 * std::min<long long>(work, clusters)));
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = GEMM_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  SDRM_CUDA(cudaLaunchKernelEx(&cfg, sdrm_gemm_pair_kernel, P));
  ++g_train_launches;
  return SDRM_OK;
}

static int launch_prep(const float* src, long long ld_src, long long R, int C, int mode, const float* src2, long long ld_src2,
                       const float* slope, const Bf16Mat* rm, const Bf16Mat* tr, double* colsum, cudaStream_t st) {
  PrepParams P;
  memset(&P, 0, sizeof P);
  P.src = src; P.ld_src = ld_src; P.src2 = src2; P.ld_src2 = ld_src2; P.slope = slope; P.R = R; P.C = C; P.mode = mode;
  if (rm) { P.rm_hi = rm->hi; P.rm_lo = rm->lo; P.ld_rm = rm->ld; }
  if (tr) { P.tr_hi = tr->hi; P.tr_lo = tr->lo; P.ld_tr = tr->ld; }
  P.colsum = colsum;
  dim3 grid(static_cast<unsigned>((C + 31) / 32), static_cast<unsigned>((R + 63) / 64));
  if (grid.y > 65535) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "operand_prep: more than 4 M rows");
  operand_prep_kernel<<<grid, 256, 0, st>>>(P);
  SDRM_CUDA(cudaGetLastError());
  ++g_train_launches;
  return SDRM_OK;
}

static long long up64(long long x) { return (x + 63) / 64 * 64; }

// ------------------------------------------------------------------------------------------------
// workspace of one training step (forward activations are kept for the backward)
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int MAX_TRAIN_LAYERS = 8;   // 1 + nh hidden PReLU layers, nh <= 6 (the output layer keeps nothing but `out`)
struct TrainLayout {
  long long R, L, D, nh, Rp, Lp, Dp, Wp, Wmax;
  int splits_h, splits_o, splits_0, n_slabs;
  size_t head, x, pre[MAX_TRAIN_LAYERS], h[MAX_TRAIN_LAYERS], w0, wh, wo, wht, wot, g_f32[2], g_bf[2], gt, xt, colsum, slabs, total;
  size_t slab_elems;
};
size_t bf_pair_bytes(long long rows, long long ld) { return (static_cast<size_t>(rows) * ld * 2 * 2 + 255) & ~static_cast<size_t>(255); }
int make_layout(long long R, int L, int D, int nh, int clusters, TrainLayout* t) {
  if (R <= 0 || L <= 0 || D <= 0 || nh < 0 || nh + 1 > MAX_TRAIN_LAYERS) return sdrm_fail(SDRM_ERR_BAD_ARG, "denoiser train: bad shape");
  t->R = R; t->L = L; t->D = D; t->nh = nh;
  t->Rp = up64(R); t->Lp = up64(L); t->Dp = up64(D); t->Wp = std::max(t->Lp, t->Dp); t->Wmax = std::max(L, D);
  t->splits_h = wgrad_splits(D, D, R, clusters);
  t->splits_o = wgrad_splits(L, D, R, clusters);
  t->splits_0 = wgrad_splits(D, L, R, clusters);
  t->n_slabs = std::max({std::max(nh, 1) * t->splits_h, t->splits_o, t->splits_0});
  t->slab_elems = static_cast<size_t>(t->Wmax) * t->Wp;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~static_cast<size_t>(255); return o; };
  t->head = take(256);
  t->x = take(bf_pair_bytes(R, t->Lp));
  for (int l = 0; l <= nh; ++l) {
    t->pre[l] = take(static_cast<size_t>(R) * t->Dp * 4);
    t->h[l] = take(bf_pair_bytes(R, t->Dp));
  }
  t->w0 = take(bf_pair_bytes(D, t->Lp));
  t->wh = take(bf_pair_bytes(D, t->Dp));
  t->wo = take(bf_pair_bytes(L, t->Dp));
  t->wht = take(bf_pair_bytes(D, t->Dp));
  t->wot = take(bf_pair_bytes(D, t->Lp));
  for (int b = 0; b < 2; ++b) {
    t->g_f32[b] = take(static_cast<size_t>(R) * t->Wp * 4);
    t->g_bf[b] = take(bf_pair_bytes(R, t->Wp));
  }
  t->gt = take(bf_pair_bytes(t->Wmax, t->Rp));
  t->xt = take(bf_pair_bytes(t->Wmax, t->Rp));
  t->colsum = take(static_cast<size_t>(t->Wp) * 8 * 2);
  t->slabs = take(static_cast<size_t>(t->n_slabs) * t->slab_elems * 4);
  t->total = off;
  return SDRM_OK;
}
Bf16Mat mat_at(uint8_t* ws, size_t off, long long rows, long long cols, long long ld) {
  Bf16Mat m;
  m.hi = reinterpret_cast<__nv_bfloat16*>(ws + off);
  m.lo = m.hi + static_cast<size_t>(rows) * ld;
  m.rows = rows; m.cols = cols; m.ld = ld;
  return m;
}
}  // namespace

extern "C" {

// automatic split-K factor (splits == 0): enough work items for the resident clusters when the output has few tiles
static int auto_splits(int64_t M, int N, int64_t K) {
  int clusters = 0;
  if (gemm_clusters(&clusters)) return 1;
  return wgrad_splits(M, N, K, clusters);
}

size_t sdrm_gemm_workspace_bytes(int64_t M, int N, int64_t K, int splits) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if (splits == 0) splits = 8;   // upper bound of the automatic choice
  const long long Kp = up64(K);
  return 256 + bf_pair_bytes(M, Kp) + bf_pair_bytes(N, Kp) + (splits > 1 ? static_cast<size_t>(splits) * M * up64(N) * 4 : 0) + 1024;
}

int sdrm_gemm(const float* d_A, int64_t lda, int trans_a, const float* d_B, int64_t ldb, int trans_b, const float* d_bias, float* d_C,
              int64_t ldc, int64_t M, int N, int64_t K, int passes, int splits, void* d_workspace, size_t workspace_bytes, void* stream) {
  if (!d_A || !d_B || !d_C || !d_workspace) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_gemm: null pointer");
  if (M <= 0 || N <= 0 || K <= 0 || ldc < N || lda < (trans_a ? M : K) || ldb < (trans_b ? N : K))
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_gemm: bad shape / leading dimension");
  if (K > 0x7fffffffLL || M > 0x7fffffffLL) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_gemm: dimension above 2^31");
  if (splits < 0) splits = 1;
  if (workspace_bytes < sdrm_gemm_workspace_bytes(M, N, K, splits)) return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_gemm: workspace too small");
  if (splits == 0) splits = auto_splits(M, N, K);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(d_workspace);
  const long long Kp = up64(K), Np = up64(N);
  SDRM_CUDA(cudaMemsetAsync(ws, 0, 256, st));
  size_t off = 256;
  Bf16Mat A = mat_at(ws, off, M, K, Kp); off += bf_pair_bytes(M, Kp);
  Bf16Mat B = mat_at(ws, off, N, K, Kp); off += bf_pair_bytes(N, Kp);
  float* slabs = reinterpret_cast<float*>(ws + off);
  int rc;
  // an operand given transposed ([K, M] / [K, N] in memory) goes through the transposing path of the operand preparation
  if (trans_a) rc = launch_prep(d_A, lda, K, static_cast<int>(M), PREP_IDENT, nullptr, 0, nullptr, nullptr, &A, nullptr, st);
  else rc = launch_prep(d_A, lda, M, static_cast<int>(K), PREP_IDENT, nullptr, 0, nullptr, &A, nullptr, nullptr, st);
  if (rc) return rc;
  if (trans_b) rc = launch_prep(d_B, ldb, K, N, PREP_IDENT, nullptr, 0, nullptr, nullptr, &B, nullptr, st);
  else rc = launch_prep(d_B, ldb, N, static_cast<int>(K), PREP_IDENT, nullptr, 0, nullptr, &B, nullptr, nullptr, st);
  if (rc) return rc;
  GemmCall g;
  g.A = A; g.B = B; g.passes = passes;
  const int kb = static_cast<int>((K + 63) / 64);
  int eff = std::max(1, std::min(splits, kb));
  const int per = (kb + eff - 1) / eff;
  eff = (kb + per - 1) / per;   // what launch_gemm uses
  if (eff > 1) {
    g.C = slabs; g.ldc = Np; g.splits = eff; g.slab_stride = static_cast<long long>(M) * Np;
  } else {
    g.C = d_C; g.ldc = ldc; g.bias = d_bias;
  }
  if ((rc = launch_gemm(g, reinterpret_cast<int*>(ws), st))) return rc;
  if (eff > 1) {
    if (d_bias) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_gemm: bias with split-K");
    slab_reduce_kernel<<<296, 256, 0, st>>>(slabs, g.slab_stride, eff, Np, static_cast<int>(M), N, d_C, ldc); ++g_train_launches;
    SDRM_CUDA(cudaGetLastError());
  }
  return SDRM_OK;
}

size_t sdrm_denoiser_train_workspace_bytes(int64_t rows, int L, int D, int nh) {
  int clusters = 0;
  if (gemm_clusters(&clusters)) return 0;
  TrainLayout t;
  if (make_layout(rows, L, D, nh, clusters, &t)) return 0;
  return t.total;
}

int sdrm_denoiser_fwd(const float* d_x, const int64_t* d_t, const float* d_table, int64_t ld_table, const float* d_W0, int64_t ldw0,
                      const float* d_a0, const float* d_Wh, const float* d_bh, const float* d_ah, const float* d_Wo, const float* d_bo,
                      int64_t rows, int L, int D, int nh, int passes, float* d_out, void* d_workspace, size_t workspace_bytes,
                      void* stream) {
  if (!d_x || !d_t || !d_table || !d_W0 || !d_a0 || !d_Wo || !d_bo || !d_out || !d_workspace)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_fwd: null pointer");
  if (nh > 0 && (!d_Wh || !d_bh || !d_ah)) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_fwd: nh > 0 needs Wh, bh, ah");
  if (ldw0 < L || ld_table < D) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_fwd: leading dimension");
  int clusters = 0, rc;
  if ((rc = gemm_clusters(&clusters))) return rc;
  TrainLayout t;
  if ((rc = make_layout(rows, L, D, nh, clusters, &t))) return rc;
  if (workspace_bytes < t.total) return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_denoiser_fwd: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(d_workspace);
  int* err = reinterpret_cast<int*>(ws + t.head);
  SDRM_CUDA(cudaMemsetAsync(ws + t.head, 0, 256, st));
  Bf16Mat X = mat_at(ws, t.x, rows, L, t.Lp);
  Bf16Mat W0 = mat_at(ws, t.w0, D, L, t.Lp), Wh = mat_at(ws, t.wh, D, D, t.Dp), Wo = mat_at(ws, t.wo, L, D, t.Dp);
  if ((rc = launch_prep(d_x, L, rows, L, PREP_IDENT, nullptr, 0, nullptr, &X, nullptr, nullptr, st))) return rc;
  if ((rc = launch_prep(d_W0, ldw0, D, L, PREP_IDENT, nullptr, 0, nullptr, &W0, nullptr, nullptr, st))) return rc;
  if (nh > 0 && (rc = launch_prep(d_Wh, D, D, D, PREP_IDENT, nullptr, 0, nullptr, &Wh, nullptr, nullptr, st))) return rc;
  if ((rc = launch_prep(d_Wo, D, L, D, PREP_IDENT, nullptr, 0, nullptr, &Wo, nullptr, nullptr, st))) return rc;
  // layer 0: pre_0 = x W0[:, :L]^T + table[t]   (the table row holds W0[:, L:] emb(t) + b0, train_SDRM.py:98-101)
  Bf16Mat Hprev = X;
  for (int l = 0; l <= nh; ++l) {
    GemmCall g;
    g.A = Hprev; g.B = (l == 0) ? W0 : Wh; g.passes = passes;
    g.C = reinterpret_cast<float*>(ws + t.pre[l]); g.ldc = t.Dp;
    if (l == 0) { g.bias_table = d_table; g.bias_rows = reinterpret_cast<const long long*>(d_t); g.bias_ld = ld_table; }
    else g.bias = d_bh;
    g.epi = GEMM_EPI_PRELU_SPLIT;
    g.slope = (l == 0) ? d_a0 : d_ah;
    g.O = mat_at(ws, t.h[l], rows, D, t.Dp);
    if ((rc = launch_gemm(g, err, st))) return rc;
    Hprev = g.O;
  }
  GemmCall g;
  g.A = Hprev; g.B = Wo; g.passes = passes;
  g.C = d_out; g.ldc = L; g.bias = d_bo; g.epi = GEMM_EPI_TANH;
  return launch_gemm(g, err, st);
}

int sdrm_denoiser_bwd(const float* d_g_out, const float* d_out, const float* d_x, const int64_t* d_order, const int64_t* d_offsets, int T,
                      const float* d_a0, const float* d_Wh, const float* d_ah, const float* d_Wo, int64_t rows, int L, int D, int nh,
                      int passes, float* d_gW0, float* d_gTable, float* d_ga0, float* d_gWh, float* d_gbh, float* d_gah,
                      float* d_gWo, float* d_gbo, void* d_workspace, size_t workspace_bytes, void* stream) {
  if (!d_g_out || !d_out || !d_x || !d_order || !d_offsets || !d_a0 || !d_Wo || !d_gW0 || !d_gTable || !d_ga0 || !d_gWo || !d_gbo || !d_workspace)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_bwd: null pointer");
  if (nh > 0 && (!d_Wh || !d_ah || !d_gWh || !d_gbh || !d_gah)) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_bwd: nh > 0 needs the hidden-layer pointers");
  int clusters = 0, rc;
  if ((rc = gemm_clusters(&clusters))) return rc;
  TrainLayout t;
  if ((rc = make_layout(rows, L, D, nh, clusters, &t))) return rc;
  if (workspace_bytes < t.total) return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_denoiser_bwd: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(d_workspace);
  int* err = reinterpret_cast<int*>(ws + t.head);
  double* slope_g = reinterpret_cast<double*>(ws + t.head + 64);   // [0] = d a0, [1] = d ah (zeroed by the forward's head memset... and here)
  SDRM_CUDA(cudaMemsetAsync(ws + t.head + 64, 0, 64, st));
  double* colsum = reinterpret_cast<double*>(ws + t.colsum);
  float* slabs = reinterpret_cast<float*>(ws + t.slabs);
  auto pre = [&](int l) { return reinterpret_cast<float*>(ws + t.pre[l]); };
  auto slope_of = [&](int l) { return l == 0 ? d_a0 : d_ah; };
  // transposed weights: B operands of the data-gradient products
  Bf16Mat WoT = mat_at(ws, t.wot, D, L, t.Lp), WhT = mat_at(ws, t.wht, D, D, t.Dp);
  if ((rc = launch_prep(d_Wo, D, L, D, PREP_IDENT, nullptr, 0, nullptr, nullptr, &WoT, nullptr, st))) return rc;
  if (nh > 0 && (rc = launch_prep(d_Wh, D, D, D, PREP_IDENT, nullptr, 0, nullptr, nullptr, &WhT, nullptr, st))) return rc;

  // ---- output layer: G = g_out * (1 - out^2)
  int cur = 0;
  Bf16Mat G = mat_at(ws, t.g_bf[cur], rows, L, t.Wp);
  Bf16Mat GT = mat_at(ws, t.gt, L, rows, t.Rp);
  SDRM_CUDA(cudaMemsetAsync(colsum, 0, sizeof(double) * t.Wp, st));
  if ((rc = launch_prep(d_g_out, L, rows, L, PREP_TANH_BWD, d_out, L, nullptr, &G, &GT, colsum, st))) return rc;
  finish_sums_kernel<<<(L + 255) / 256, 256, 0, st>>>(colsum, L, d_gbo); ++g_train_launches;
  // dWo = G^T H_nh^T^T   (A = G^T [L, rows], B = H_nh^T [D, rows])
  Bf16Mat XT = mat_at(ws, t.xt, D, rows, t.Rp);
  if ((rc = launch_prep(pre(nh), t.Dp, rows, D, PREP_PRELU, nullptr, 0, slope_of(nh), nullptr, &XT, nullptr, st))) return rc;
  {
    GemmCall g;
    g.A = GT; g.B = XT; g.passes = passes; g.C = slabs; g.ldc = t.Wp; g.splits = t.splits_o; g.slab_stride = static_cast<long long>(t.slab_elems);
    if ((rc = launch_gemm(g, err, st))) return rc;
    slab_reduce_kernel<<<296, 256, 0, st>>>(slabs, g.slab_stride, wgrad_splits(L, D, rows, clusters), t.Wp, L, D, d_gWo, D); ++g_train_launches;
  }
  // dH_nh = G Wo, then through PReLU'(pre_nh): the new G
  {
    GemmCall g;
    g.A = G; g.B = WoT; g.passes = passes;
    g.C = reinterpret_cast<float*>(ws + t.g_f32[cur ^ 1]); g.ldc = t.Wp;
    g.epi = GEMM_EPI_DPRELU; g.slope = slope_of(nh); g.aux = pre(nh); g.ld_aux = t.Dp; g.slope_grad = slope_g + (nh == 0 ? 0 : 1);
    g.O = mat_at(ws, t.g_bf[cur ^ 1], rows, D, t.Wp);
    if ((rc = launch_gemm(g, err, st))) return rc;
    cur ^= 1;
  }
  // ---- hidden layers nh .. 1 (all applications of the ONE shared Linear, train_SDRM.py:94)
  if (nh > 0) SDRM_CUDA(cudaMemsetAsync(colsum, 0, sizeof(double) * t.Wp, st));
  for (int j = nh; j >= 1; --j) {
    G = mat_at(ws, t.g_bf[cur], rows, D, t.Wp);
    const float* Gf = reinterpret_cast<const float*>(ws + t.g_f32[cur]);
    GT = mat_at(ws, t.gt, D, rows, t.Rp);
    if ((rc = launch_prep(Gf, t.Wp, rows, D, PREP_IDENT, nullptr, 0, nullptr, nullptr, &GT, colsum, st))) return rc;
    XT = mat_at(ws, t.xt, D, rows, t.Rp);
    if ((rc = launch_prep(pre(j - 1), t.Dp, rows, D, PREP_PRELU, nullptr, 0, slope_of(j - 1), nullptr, &XT, nullptr, st))) return rc;
    GemmCall gw;
    gw.A = GT; gw.B = XT; gw.passes = passes; gw.ldc = t.Wp; gw.splits = t.splits_h; gw.slab_stride = static_cast<long long>(t.slab_elems);
    gw.C = slabs + static_cast<size_t>(nh - j) * t.splits_h * t.slab_elems;
    if ((rc = launch_gemm(gw, err, st))) return rc;
    GemmCall gd;
    gd.A = G; gd.B = WhT; gd.passes = passes;
    gd.C = reinterpret_cast<float*>(ws + t.g_f32[cur ^ 1]); gd.ldc = t.Wp;
    gd.epi = GEMM_EPI_DPRELU; gd.slope = slope_of(j - 1); gd.aux = pre(j - 1); gd.ld_aux = t.Dp; gd.slope_grad = slope_g + (j - 1 == 0 ? 0 : 1);
    gd.O = mat_at(ws, t.g_bf[cur ^ 1], rows, D, t.Wp);
    if ((rc = launch_gemm(gd, err, st))) return rc;
    cur ^= 1;
  }
  if (nh > 0) {
    slab_reduce_kernel<<<296, 256, 0, st>>>(slabs, static_cast<long long>(t.slab_elems), nh * wgrad_splits(D, D, rows, clusters), t.Wp, D, D, d_gWh, D); ++g_train_launches;
    finish_sums_kernel<<<(D + 255) / 256, 256, 0, st>>>(colsum, D, d_gbh); ++g_train_launches;
  }
  // ---- layer 0: dW0[:, :L] = G_0^T x, and the gradient of the time-embedding bias rows
  {
    const float* Gf = reinterpret_cast<const float*>(ws + t.g_f32[cur]);
    GT = mat_at(ws, t.gt, D, rows, t.Rp);
    if ((rc = launch_prep(Gf, t.Wp, rows, D, PREP_IDENT, nullptr, 0, nullptr, nullptr, &GT, nullptr, st))) return rc;
    XT = mat_at(ws, t.xt, L, rows, t.Rp);
    if ((rc = launch_prep(d_x, L, rows, L, PREP_IDENT, nullptr, 0, nullptr, nullptr, &XT, nullptr, st))) return rc;
    GemmCall g;
    g.A = GT; g.B = XT; g.passes = passes; g.C = slabs; g.ldc = t.Wp; g.splits = t.splits_0; g.slab_stride = static_cast<long long>(t.slab_elems);
    if ((rc = launch_gemm(g, err, st))) return rc;
    slab_reduce_kernel<<<296, 256, 0, st>>>(slabs, g.slab_stride, wgrad_splits(D, L, rows, clusters), t.Wp, D, L, d_gW0, L); ++g_train_launches;
    dim3 grid(static_cast<unsigned>(T + 1), static_cast<unsigned>((D + 255) / 256));
    table_grad_kernel<<<grid, 256, 0, st>>>(Gf, t.Wp, reinterpret_cast<const long long*>(d_order), reinterpret_cast<const long long*>(d_offsets), D, d_gTable, D); ++g_train_launches;
  }
  finish_sums_kernel<<<1, 32, 0, st>>>(slope_g, 1, d_ga0); ++g_train_launches;
  if (nh > 0) {
    finish_sums_kernel<<<1, 32, 0, st>>>(slope_g + 1, 1, d_gah); ++g_train_launches;
  }
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

long long sdrm_train_launch_count(int reset) {
  const long long n = g_train_launches;
  if (reset) g_train_launches = 0;
  return n;
}

int sdrm_train_check_device_error(const void* d_workspace, void* stream) {
  cudaError_t e = cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
  int word = 0;
  cudaError_t e2 = cudaMemcpy(&word, d_workspace, sizeof(int), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess || e2 != cudaSuccess || word != 0) {
    char msg[200];
    snprintf(msg, sizeof msg, "device error: sync=%s copy=%s watchdog=%d", cudaGetErrorString(e), cudaGetErrorString(e2), word);
    return sdrm_fail(SDRM_ERR_CUDA, msg);
  }
  return SDRM_OK;
}

}  // extern "C"
