// Host side of K1: weight / bias packing kernels and the C-ABI entry points that drive the
// layer engine (sdrm_create, sdrm_denoiser_pack, sdrm_decoder_pack, sdrm_sample, sdrm_probe_linear).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>

#include "../../include/sdrm_b200.h"
#include "host_util.h"
#include "layer_engine.cuh"
#include "layer_engine_kernel.cuh"
#include "ptx_sm100.cuh"
#include "small_chain_kernel.cuh"
#include "engine_launch.cuh"

namespace sdrm {

// ------------------------------------------------------------------------------------------------
// geometry of one dense layer on the engine
// ------------------------------------------------------------------------------------------------
struct Geom {
  int N = 0, K = 0, NCH = 0, NC = 0, Np = 0, KB = 0, kmma_last = 0;
  size_t img_bytes() const { return static_cast<size_t>(NCH) * KB * NC * 128; }  // one image (hi or lo)
};
static Geom make_geom(int N, int K) {
  Geom g;
  g.N = N; g.K = K;
  g.NCH = (N + MAX_NC - 1) / MAX_NC;
  const int per = (N + g.NCH - 1) / g.NCH;
  g.NC = ((per + 15) / 16) * 16;
  g.Np = g.NCH * g.NC;
  g.KB = (K + KBLK - 1) / KBLK;
  const int rem = K - KBLK * (g.KB - 1);
  g.kmma_last = (rem + 15) / 16;
  return g;
}

// Column-split geometry (clusters of SPLIT_S CTAs per row tile, see the kernel): a layer of fewer than SPLIT_S chunks is re-cut
// into SPLIT_S narrower ones, so that every CTA of the cluster owns one -- half the weight bytes and half the epilogue per SM
// of a 4-chunk geometry.  (A UMMA costs ~60 ns whatever its N <= 208, so the narrower chunks do not shorten a layer's tensor
// phase; they shorten everything around it: profiles/k1_split_r02.txt.)
constexpr int SPLIT_S = 8;
static Geom make_geom_split(int N, int K) {
  Geom g = make_geom(N, K);
  if (g.NCH >= SPLIT_S) return g;
  g.NCH = SPLIT_S;
  const int per = (N + g.NCH - 1) / g.NCH;
  g.NC = std::max(16, ((per + 15) / 16) * 16);
  g.Np = g.NCH * g.NC;
  return g;
}
static bool same_geom(const Geom& a, const Geom& b) { return a.NCH == b.NCH && a.NC == b.NC && a.KB == b.KB; }

// ------------------------------------------------------------------------------------------------
// packing kernels
// ------------------------------------------------------------------------------------------------
// W fp32 [N, ldw] (columns col_off .. col_off+K) -> bf16 hi (and lo) tile images
__global__ void pack_weight_kernel(const float* __restrict__ W, int N, int K, long long ldw, int col_off,
                                   uint8_t* __restrict__ img_hi, uint8_t* __restrict__ img_lo, int NCH, int NC, int KB) {
  const long long total = static_cast<long long>(NCH) * KB * NC * 8;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int j = static_cast<int>(idx & 7);
    long long t = idx >> 3;
    const int r = static_cast<int>(t % NC); t /= NC;
    const int kb = static_cast<int>(t % KB);
    const int c = static_cast<int>(t / KB);
    const int n = c * NC + r;
    const int k0 = kb * KBLK + j * 8;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v0 = 0.f, v1 = 0.f;
      if (n < N) {
        if (k0 + 2 * e < K) v0 = W[n * ldw + col_off + k0 + 2 * e];
        if (k0 + 2 * e + 1 < K) v1 = W[n * ldw + col_off + k0 + 2 * e + 1];
      }
      const float h0 = bf16_round(v0), h1 = bf16_round(v1);
      hi[e] = pack_bf16x2(h0, h1);
      lo[e] = pack_bf16x2(v0 - h0, v1 - h1);
    }
    const size_t off = ((static_cast<size_t>(c) * KB + kb) * NC + r) * 128 + ((j ^ (r & 7)) << 4);
    *reinterpret_cast<uint4*>(img_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (img_lo) *reinterpret_cast<uint4*>(img_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// A fp32 [M, K] -> per-tile activation images (hi / lo) for the probe entry
__global__ void pack_act_kernel(const float* __restrict__ A, long long M, int K, uint8_t* __restrict__ scratch,
                                size_t scratch_stride, size_t act_buf_bytes, int KB) {
  const long long n_tiles = (M + TILE_M - 1) / TILE_M;
  const long long total = n_tiles * KB * TILE_M * 8;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int j = static_cast<int>(idx & 7);
    long long t = idx >> 3;
    const int r = static_cast<int>(t % TILE_M); t /= TILE_M;
    const int kb = static_cast<int>(t % KB);
    const long long tile = t / KB;
    const long long row = tile * TILE_M + r;
    const int k0 = kb * KBLK + j * 8;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v0 = 0.f, v1 = 0.f;
      if (row < M) {
        if (k0 + 2 * e < K) v0 = A[row * K + k0 + 2 * e];
        if (k0 + 2 * e + 1 < K) v1 = A[row * K + k0 + 2 * e + 1];
      }
      const float h0 = bf16_round(v0), h1 = bf16_round(v1);
      hi[e] = pack_bf16x2(h0, h1);
      lo[e] = pack_bf16x2(v0 - h0, v1 - h1);
    }
    uint8_t* base = scratch + static_cast<size_t>(tile) * scratch_stride;
    // activation images are LINEAR in global memory ([k block][row][64 bf16]); the TMA load swizzles them (SWIZZLE_128B)
    const size_t off = static_cast<size_t>(kb) * A_TILE_BYTES + r * 128 + (j << 4);
    *reinterpret_cast<uint4*>(base + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(base + act_buf_bytes + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

__global__ void pad_bias_kernel(const float* __restrict__ b, int N, float* __restrict__ out, int Np) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Np; i += gridDim.x * blockDim.x)
    out[i] = (b != nullptr && i < N) ? b[i] : 0.0f;
}

// Hoisted timestep embedding (SDRM.timestep_embedding + emb_layer + the emb columns of dnn.0,
// train_SDRM.py:98-112): bias0[i][n] = b0[n] + sum_t W0[n][L+t] * (be[t] + sum_s We[t][s] temb_i[s]).
// One block per step i in [0, T].
__global__ void bias_table_kernel(const float* __restrict__ We, const float* __restrict__ be,
                                  const float* __restrict__ W0, const float* __restrict__ b0, int T, int L, int D,
                                  float* __restrict__ out, int Np) {
  extern __shared__ float sh[];
  float* temb = sh;       // [T]
  float* emb = sh + T;    // [T]
  const int i = blockIdx.x;
  const int half = T / 2;
  for (int s = threadIdx.x; s < T; s += blockDim.x) {
    float v = 0.0f;
    if (s < 2 * half) {
      const int k = s < half ? s : s - half;
      const float freq = expf(-logf(10000.0f) * static_cast<float>(k) / static_cast<float>(half));
      const float arg = static_cast<float>(i) * freq;
      v = s < half ? cosf(arg) : sinf(arg);
    }
    temb[s] = v;
  }
  __syncthreads();
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    float acc = 0.0f;
    for (int s = 0; s < T; ++s) acc = fmaf(We[static_cast<size_t>(t) * T + s], temb[s], acc);
    emb[t] = acc + be[t];
  }
  __syncthreads();
  for (int n = threadIdx.x; n < Np; n += blockDim.x) {
    float acc = 0.0f;
    if (n < D) {
      const float* w = W0 + static_cast<size_t>(n) * (L + T) + L;
      for (int t = 0; t < T; ++t) acc = fmaf(w[t], emb[t], acc);
      acc += b0[n];
    }
    out[static_cast<size_t>(i) * Np + n] = acc;
  }
}

// K6 images: W fp32 [N, ldw] (columns col_off .. col_off + K) -> zero-padded bf16 hi (and lo) [rows_pad][SMALL_KP]
__global__ void pack_small_weight_kernel(const float* __restrict__ W, int N, int K, long long ldw, int col_off, int rows_pad,
                                         __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const long long total = static_cast<long long>(rows_pad) * SMALL_KP;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total; idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(idx / SMALL_KP), k = static_cast<int>(idx - static_cast<long long>(r) * SMALL_KP);
    const float v = (r < N && k < K) ? W[r * ldw + col_off + k] : 0.0f;
    const float h = bf16_round(v);
    hi[idx] = __float2bfloat16_rn(h);
    if (lo) lo[idx] = __float2bfloat16_rn(v - h);
  }
}
// rows of `cols` floats (pitch src_ld) -> rows of 64 zero-padded floats
__global__ void pad_rows64_kernel(const float* __restrict__ src, long long src_ld, int cols, int rows, float* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * 64) return;
  const int r = i >> 6, c = i & 63;
  dst[i] = (src != nullptr && c < cols) ? src[r * src_ld + c] : 0.0f;
}

// coef[i] = {(1-a_i)/sqrt(1-ab_i), 1/sqrt(a_i), sqrt(b_i)*nd (0 at i=1), 0}  (train_SDRM.py:20-25,56)
__global__ void coef_kernel(const float* __restrict__ sched, int T, float nd, float* __restrict__ coef) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > T) return;
  const float b = sched[i], a = sched[(T + 1) + i], ab = sched[2 * (T + 1) + i];
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i >= 1) {
    c.x = (1.0f - a) / sqrtf(1.0f - ab);
    c.y = 1.0f / sqrtf(a);
    c.z = i > 1 ? sqrtf(b) * nd : 0.0f;
  }
  reinterpret_cast<float4*>(coef)[i] = c;
}

}  // namespace sdrm

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
using namespace sdrm;

struct sdrm_handle {
  int device = 0;
  int num_sms = 0;
  int last_launches = 0;
  int last_cluster = 1;
  int resident[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // resident CTAs per cluster size (1, 2, 4, 8)
  int* err_word = nullptr;        // device view of the watchdog word
  volatile int* err_host = nullptr;   // host view: the word lives in mapped pinned host memory, so it survives a device trap
  // per-handle tuning options (sdrm_set_option); 0 = automatic
  int cluster_override = 0;     // 1 / 2 / 4 / 8
  int subtile_override = 0;     // 1 / 2 row tiles a CTA interleaves
  int no_discard = 0;           // 1 = keep dead activation lines in the L2 (A/B of the discard warp)
  int no_resident = 0;          // 1 = never keep the chain's activation tile in shared memory (A/B of the resident mode)
  int no_split = 0;             // 1 = never split a row tile's N chunks over a cluster (A/B of the column-split mode)
  int split_resident[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // resident CTAs of the column-split kernel per cluster size (2, 4, 8)
  int last_split = 0;           // cluster size of the last launch's column split (0: not split)
  int last_resident = 0;        // what the last sdrm_sample launch did
  int grid_limit = 0;           // cap on the CTAs of an sdrm_sample launch (tests: small inputs exercise the multi-tile loops)
  int debug_flags = 0;          // -DSDRM_PERF_DEBUG builds only
  unsigned long long* trace = nullptr;   // -DSDRM_TRACE builds only
  // denoiser
  bool have_den = false;
  int T = 0, L = 0, D = 0, nh = 0;
  float nd = 1.0f;
  Geom g0, gh, go;
  uint8_t *w0 = nullptr, *wh = nullptr, *wo = nullptr;
  // column-split geometry (8 chunks per layer) and its weight images; packed for every denoiser the tcgen05 engine takes (> 64 wide)
  Geom s0, sh, so, s1, s2;
  uint8_t *w0s = nullptr, *whs = nullptr, *wos = nullptr, *w1s = nullptr, *w2s = nullptr;
  bool split_den = false, split_dec = false;
  int np0 = 0, nph = 0, npo = 0, np1 = 0, np2 = 0;   // padded bias widths (both geometries fit)
  float *bias0 = nullptr, *bh = nullptr, *bo = nullptr, *slopes = nullptr, *coef = nullptr;
  // K6 (small denoisers, small_chain_kernel.cuh): zero-padded bf16 images and 64-wide bias rows, packed when every width <= 64
  bool small_den = false, small_dec = false;
  __nv_bfloat16 *s_den = nullptr;   // w0 | wh | wo, each [64][SMALL_KP]
  __nv_bfloat16 *s_dec1 = nullptr;  // w1 hi | w1 lo
  __nv_bfloat16 *s_dec2 = nullptr;  // w2 hi | w2 lo, each [I rounded up to 64][SMALL_KP]
  float *s_bias = nullptr;          // bias0 [T+1][64] | bh [64] | bo [64]
  float *s_b1 = nullptr;            // b1 [64] | b2 [I rounded up to 64]
  int engine_choice = 0;            // SDRM_OPT_ENGINE: 0 automatic, 1 tcgen05 layer engine, 2 small-chain kernel
  // decoder
  bool have_dec = false;
  int H = 0, I = 0;
  Geom g1, g2;
  uint8_t *w1 = nullptr, *w2 = nullptr;
  float *b1 = nullptr, *b2 = nullptr;
};

static void free_den(sdrm_handle* h) {
  cudaFree(h->w0); cudaFree(h->wh); cudaFree(h->wo);
  cudaFree(h->w0s); cudaFree(h->whs); cudaFree(h->wos);
  h->w0s = h->whs = h->wos = nullptr; h->split_den = false;
  cudaFree(h->bias0); cudaFree(h->bh); cudaFree(h->bo); cudaFree(h->slopes); cudaFree(h->coef);
  cudaFree(h->s_den); cudaFree(h->s_bias);
  h->s_den = nullptr; h->s_bias = nullptr; h->small_den = false;
  h->w0 = h->wh = h->wo = nullptr;
  h->bias0 = h->bh = h->bo = h->slopes = h->coef = nullptr;
  h->have_den = false;
}
static void free_dec(sdrm_handle* h) {
  cudaFree(h->w1); cudaFree(h->w2); cudaFree(h->b1); cudaFree(h->b2);
  cudaFree(h->w1s); cudaFree(h->w2s);
  h->w1s = h->w2s = nullptr; h->split_dec = false;
  cudaFree(h->s_dec1); cudaFree(h->s_dec2); cudaFree(h->s_b1);
  h->s_dec1 = h->s_dec2 = nullptr; h->s_b1 = nullptr; h->small_dec = false;
  h->w1 = h->w2 = nullptr;
  h->b1 = h->b2 = nullptr;
  h->have_dec = false;
}


// run-time watchdog limit of this translation unit's kernels (ptx_sm100.cuh): SDRM_WATCHDOG_MS in the environment, 0 = none
static int apply_watchdog_env_k1() {
  static bool done = false;
  if (done) return SDRM_OK;
  done = true;
  const char* e = getenv("SDRM_WATCHDOG_MS");
  if (!e || !*e) return SDRM_OK;
  const unsigned long long ns = strtoull(e, nullptr, 10) * 1000000ull;
  SDRM_CUDA(cudaMemcpyToSymbol(sdrm::g_sdrm_watchdog_ns, &ns, sizeof ns));
  return SDRM_OK;
}

static int engine_set_smem_attr() {
  { int wrc = apply_watchdog_env_k1(); if (wrc) return wrc; }
  static bool done[64] = {false};
  int dev = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && done[dev]) return SDRM_OK;
  SDRM_CUDA(cudaFuncSetAttribute(sdrm_layer_engine_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
  SDRM_CUDA(cudaFuncSetAttribute(sdrm_layer_engine_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
  SDRM_CUDA(cudaFuncSetAttribute((sdrm_layer_engine_kernel<2, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
  SDRM_CUDA(cudaFuncSetAttribute((sdrm_layer_engine_kernel<1, false, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, ENGINE_SMEM_BYTES));
  if (dev < 64) done[dev] = true;
  return SDRM_OK;
}

// resident CTAs for a cluster size (1 CTA per SM; clusters must fit inside a GPC)
static int max_resident_ctas(int cluster, int num_sms, bool split = false) {
  if (cluster == 1) return num_sms;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(num_sms / cluster * cluster));
  cfg.blockDim = dim3(ENGINE_THREADS);
  cfg.dynamicSmemBytes = ENGINE_SMEM_BYTES;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  int n = 0;
  if (!split && cluster != 2) return 0;
  cudaError_t e = split ? cudaOccupancyMaxActiveClusters(&n, (sdrm_layer_engine_kernel<1, false, true>), &cfg)
                        : cudaOccupancyMaxActiveClusters(&n, sdrm_layer_engine_kernel<2>, &cfg);
  if (e != cudaSuccess) { cudaGetLastError(); return 0; }
  return n * cluster;
}

// ---- TMA tensor maps: a blob of `rows` x 128 bytes, box = `box_rows` rows x `box_bytes`.  Weight maps (pair mode) take no
// swizzle: the weight images are pre-swizzled in global memory, so a box lands in shared memory byte-for-byte like the bulk
// copies of single mode.  The activation load map swizzles (SWIZZLE_128B), the activation store map does not.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
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
static int make_rows_map(CUtensorMap* map, const void* base, unsigned long long rows, unsigned box_rows, unsigned box_bytes = 128,
                         bool swizzle128 = false) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return sdrm_fail(SDRM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t dims[2] = {128, rows};
  const cuuint64_t strides[1] = {128};
  const cuuint32_t box[2] = {box_bytes, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char msg[128];
    snprintf(msg, sizeof msg, "cuTensorMapEncodeTiled failed (%d) rows=%llu box=%u", static_cast<int>(r), rows, box_rows);
    return sdrm_fail(SDRM_ERR_CUDA, msg);
  }
  return SDRM_OK;
}
// Activation scratch maps (every mode): the images are linear rows of 128 bytes; loads take a 128-row box and swizzle it into the
// UMMA operand layout, the epilogue stores 32 rows x 32 bytes (one warp's 16-column group) from a dense shared-memory box
static int fill_act_maps(ChainParams& P, size_t workspace_bytes) {
  int rc = make_rows_map(&P.tm_act, P.scratch, workspace_bytes / 128, TILE_M, 128, true);
  if (rc) return rc;
  return make_rows_map(&P.tm_act_st, P.scratch, workspace_bytes / 128, 32, 32, false);
}
static int fill_pair_maps(ChainParams& P, size_t workspace_bytes, int cluster) {
  auto w_rows = [](const LayerDesc& d) {
    return static_cast<unsigned long long>(d.passes == 3 ? 2 : 1) * d.NCH * d.KB * d.NC;
  };
  for (int l = 0; l < P.n_step; ++l) {
    int rc = make_rows_map(&P.tm_step_w[l], P.step[l].w_img, w_rows(P.step[l]), P.step[l].NC / cluster);
    if (rc) return rc;
  }
  for (int l = 0; l < P.n_dec; ++l) {
    int rc = make_rows_map(&P.tm_dec_w[l], P.dec[l].w_img, w_rows(P.dec[l]), P.dec[l].NC / cluster);
    if (rc) return rc;
  }
  (void)workspace_bytes;
  return SDRM_OK;
}

// The bfloat16-logits instantiations (sdrm_sample_bf16) are compiled in engine_bf16.cu: in this translation unit they would
// perturb how the compiler optimises the fp32 kernels, whose code stays as it is.
static int launch_engine(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split = 0, bool bf16 = false) {
  return bf16 ? launch_engine_bf16(P, grid, cluster, st, split) : launch_engine_t<false>(P, grid, cluster, st, split);
}

static void launch_pack_weight(const float* W, int N, int K, long long ldw, int col_off, uint8_t* hi, uint8_t* lo,
                               const Geom& g, cudaStream_t st) {
  const long long total = static_cast<long long>(g.NCH) * g.KB * g.NC * 8;
  const int blocks = static_cast<int>(std::min<long long>((total + 255) / 256, 4096));
  pack_weight_kernel<<<blocks, 256, 0, st>>>(W, N, K, ldw, col_off, hi, lo, g.NCH, g.NC, g.KB);
}

extern "C" {

int sdrm_version(void) { return 100; }

int sdrm_create(sdrm_handle** out, int device) {
  if (!out) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_create: out is null");
  SDRM_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SDRM_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    char msg[160];
    snprintf(msg, sizeof msg, "sdrm_create: device %d is sm_%d%d; this library is built for sm_100a only", device,
             prop.major, prop.minor);
    return sdrm_fail(SDRM_ERR_UNSUPPORTED, msg);
  }
  sdrm_handle* h = new sdrm_handle();
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  {
    // the watchdog word is zero-copy host memory: a trapped kernel leaves the context unusable, but the role code it wrote
    // can still be read and reported (sdrm_check_device_error)
    void* hp = nullptr;
    SDRM_CUDA(cudaHostAlloc(&hp, 8 * sizeof(int), cudaHostAllocMapped));
    memset(hp, 0, 8 * sizeof(int));
    void* dp = nullptr;
    SDRM_CUDA(cudaHostGetDevicePointer(&dp, hp, 0));
    h->err_host = static_cast<volatile int*>(hp);
    h->err_word = static_cast<int*>(dp);
  }
  if (engine_set_smem_attr() != SDRM_OK) { delete h; return SDRM_ERR_CUDA; }
  h->resident[1] = h->num_sms;
  h->resident[2] = max_resident_ctas(2, h->num_sms);
  for (int cs = 2; cs <= 8; cs *= 2) h->split_resident[cs] = max_resident_ctas(cs, h->num_sms, true);
  *out = h;
  return SDRM_OK;
}

int sdrm_destroy(sdrm_handle* h) {
  if (!h) return SDRM_OK;
  cudaSetDevice(h->device);
  free_den(h);
  free_dec(h);
  if (h->err_host) cudaFreeHost(const_cast<int*>(h->err_host));
  delete h;
  return SDRM_OK;
}

int sdrm_denoiser_pack(sdrm_handle* h, const float* d_We, const float* d_be, const float* d_W0, const float* d_b0,
                       const float* d_a0, const float* d_Wh, const float* d_bh, const float* d_ah, const float* d_Wo,
                       const float* d_bo, const float* d_sched, int T, int L, int D, int nh, float noise_divider,
                       void* stream) {
  if (!h || !d_We || !d_be || !d_W0 || !d_b0 || !d_a0 || !d_Wo || !d_bo || !d_sched)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_pack: null pointer");
  if (nh > 0 && (!d_Wh || !d_bh || !d_ah)) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_pack: nh>0 needs Wh,bh,ah");
  if (T < 1 || L < 1 || D < 1 || nh < 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_denoiser_pack: bad shape");
  if (2 + nh > MAX_STEP_LAYERS) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_denoiser_pack: nh > 6");
  if (L > MAX_ACT_CHUNKS * MAX_NC || D > MAX_ACT_CHUNKS * MAX_NC)
    return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_denoiser_pack: latent / hidden width above 8 x 256");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaSetDevice(h->device));
  const bool same = h->have_den && h->T == T && h->L == L && h->D == D && h->nh == nh;
  if (!same) {
    free_den(h);
    h->T = T; h->L = L; h->D = D; h->nh = nh;
    h->g0 = make_geom(D, L);
    h->gh = make_geom(D, D);
    h->go = make_geom(L, D);
    h->s0 = make_geom_split(D, L);
    h->sh = make_geom_split(D, D);
    h->so = make_geom_split(L, D);
    h->np0 = std::max(h->g0.Np, h->s0.Np); h->nph = std::max(h->gh.Np, h->sh.Np); h->npo = std::max(h->go.Np, h->so.Np);
    SDRM_CUDA(cudaMalloc(&h->w0, h->g0.img_bytes()));
    SDRM_CUDA(cudaMalloc(&h->wh, h->gh.img_bytes()));
    SDRM_CUDA(cudaMalloc(&h->wo, h->go.img_bytes()));
    // a second set of images in the column-split geometry (every layer re-cut into 8 chunks), unless it is the normal one
    h->split_den = std::max(L, D) > SMALL_MAX &&   // (narrower denoisers run on the small-chain kernel)
                   !(same_geom(h->g0, h->s0) && same_geom(h->gh, h->sh) && same_geom(h->go, h->so));
    if (h->split_den) {
      SDRM_CUDA(cudaMalloc(&h->w0s, h->s0.img_bytes()));
      SDRM_CUDA(cudaMalloc(&h->whs, h->sh.img_bytes()));
      SDRM_CUDA(cudaMalloc(&h->wos, h->so.img_bytes()));
    }
    SDRM_CUDA(cudaMalloc(&h->bias0, sizeof(float) * (T + 1) * h->np0));
    SDRM_CUDA(cudaMalloc(&h->bh, sizeof(float) * h->nph));
    SDRM_CUDA(cudaMalloc(&h->bo, sizeof(float) * h->npo));
    SDRM_CUDA(cudaMalloc(&h->slopes, sizeof(float) * 2));
    SDRM_CUDA(cudaMalloc(&h->coef, sizeof(float) * 4 * (T + 1)));
  }
  h->nd = noise_divider;
  launch_pack_weight(d_W0, D, L, L + T, 0, h->w0, nullptr, h->g0, st);
  if (nh > 0) launch_pack_weight(d_Wh, D, D, D, 0, h->wh, nullptr, h->gh, st);
  launch_pack_weight(d_Wo, L, D, D, 0, h->wo, nullptr, h->go, st);
  if (h->split_den) {
    launch_pack_weight(d_W0, D, L, L + T, 0, h->w0s, nullptr, h->s0, st);
    if (nh > 0) launch_pack_weight(d_Wh, D, D, D, 0, h->whs, nullptr, h->sh, st);
    launch_pack_weight(d_Wo, L, D, D, 0, h->wos, nullptr, h->so, st);
  }
  bias_table_kernel<<<T + 1, 256, sizeof(float) * 2 * T, st>>>(d_We, d_be, d_W0, d_b0, T, L, D, h->bias0, h->np0);
  pad_bias_kernel<<<(h->nph + 255) / 256, 256, 0, st>>>(nh > 0 ? d_bh : nullptr, D, h->bh, h->nph);
  pad_bias_kernel<<<(h->npo + 255) / 256, 256, 0, st>>>(d_bo, L, h->bo, h->npo);
  SDRM_CUDA(cudaMemcpyAsync(h->slopes, d_a0, sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (nh > 0) SDRM_CUDA(cudaMemcpyAsync(h->slopes + 1, d_ah, sizeof(float), cudaMemcpyDeviceToDevice, st));
  coef_kernel<<<(T + 1 + 127) / 128, 128, 0, st>>>(d_sched, T, noise_divider, h->coef);
  SDRM_CUDA(cudaGetLastError());
  if (L <= SMALL_MAX && D <= SMALL_MAX) {   // K6 images
    const size_t img = static_cast<size_t>(64) * SMALL_KP;
    if (!h->s_den) {
      SDRM_CUDA(cudaMalloc(&h->s_den, 3 * img * sizeof(__nv_bfloat16)));
      SDRM_CUDA(cudaMalloc(&h->s_bias, sizeof(float) * 64 * (T + 3)));
    }
    pack_small_weight_kernel<<<18, 256, 0, st>>>(d_W0, D, L, L + T, 0, 64, h->s_den, nullptr);
    pack_small_weight_kernel<<<18, 256, 0, st>>>(nh > 0 ? d_Wh : d_Wo, nh > 0 ? D : 0, nh > 0 ? D : 0, D, 0, 64, h->s_den + img, nullptr);
    pack_small_weight_kernel<<<18, 256, 0, st>>>(d_Wo, L, D, D, 0, 64, h->s_den + 2 * img, nullptr);
    pad_rows64_kernel<<<(64 * (T + 1) + 255) / 256, 256, 0, st>>>(h->bias0, h->np0, D, T + 1, h->s_bias);
    pad_rows64_kernel<<<1, 64, 0, st>>>(nh > 0 ? d_bh : nullptr, 0, D, 1, h->s_bias + 64 * (T + 1));
    pad_rows64_kernel<<<1, 64, 0, st>>>(d_bo, 0, L, 1, h->s_bias + 64 * (T + 2));
    SDRM_CUDA(cudaGetLastError());
    h->small_den = true;
  } else {
    h->small_den = false;
  }
  h->have_den = true;
  return SDRM_OK;
}

int sdrm_decoder_pack(sdrm_handle* h, const float* d_W1, const float* d_b1, const float* d_W2, const float* d_b2,
                      int L, int H, int I, void* stream) {
  if (!h || !d_W1 || !d_b1 || !d_W2 || !d_b2) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_decoder_pack: null pointer");
  if (L < 1 || H < 1 || I < 1) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_decoder_pack: bad shape");
  if (H > MAX_ACT_CHUNKS * MAX_NC) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_decoder_pack: VAE hidden width above 8 x 256");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaSetDevice(h->device));
  const bool same = h->have_dec && h->g1.K == L && h->H == H && h->I == I;
  if (!same) {
    free_dec(h);
    h->H = H; h->I = I;
    h->g1 = make_geom(H, L);
    h->g2 = make_geom(I, H);
    h->s1 = make_geom_split(H, L);
    h->s2 = make_geom_split(I, H);
    h->np1 = std::max(h->g1.Np, h->s1.Np); h->np2 = std::max(h->g2.Np, h->s2.Np);
    SDRM_CUDA(cudaMalloc(&h->w1, 2 * h->g1.img_bytes()));
    SDRM_CUDA(cudaMalloc(&h->w2, 2 * h->g2.img_bytes()));
    h->split_dec = L > SMALL_MAX;   // the denoiser this decoder follows may take the column split
    if (h->split_dec) {
      if (!same_geom(h->g1, h->s1)) SDRM_CUDA(cudaMalloc(&h->w1s, 2 * h->s1.img_bytes()));
      if (!same_geom(h->g2, h->s2)) SDRM_CUDA(cudaMalloc(&h->w2s, 2 * h->s2.img_bytes()));
    }
    SDRM_CUDA(cudaMalloc(&h->b1, sizeof(float) * h->np1));
    SDRM_CUDA(cudaMalloc(&h->b2, sizeof(float) * h->np2));
  }
  launch_pack_weight(d_W1, H, L, L, 0, h->w1, h->w1 + h->g1.img_bytes(), h->g1, st);
  launch_pack_weight(d_W2, I, H, H, 0, h->w2, h->w2 + h->g2.img_bytes(), h->g2, st);
  if (h->w1s) launch_pack_weight(d_W1, H, L, L, 0, h->w1s, h->w1s + h->s1.img_bytes(), h->s1, st);
  if (h->w2s) launch_pack_weight(d_W2, I, H, H, 0, h->w2s, h->w2s + h->s2.img_bytes(), h->s2, st);
  pad_bias_kernel<<<(h->np1 + 255) / 256, 256, 0, st>>>(d_b1, H, h->b1, h->np1);
  pad_bias_kernel<<<(h->np2 + 255) / 256, 256, 0, st>>>(d_b2, I, h->b2, h->np2);
  SDRM_CUDA(cudaGetLastError());
  if (L <= SMALL_MAX && H <= SMALL_MAX) {   // K6 images
    const size_t img = static_cast<size_t>(64) * SMALL_KP;
    const int I_pad = (I + 63) / 64 * 64;
    const size_t img2 = static_cast<size_t>(I_pad) * SMALL_KP;
    if (!h->s_dec1) {
      SDRM_CUDA(cudaMalloc(&h->s_dec1, 2 * img * sizeof(__nv_bfloat16)));
      SDRM_CUDA(cudaMalloc(&h->s_dec2, 2 * img2 * sizeof(__nv_bfloat16)));
      SDRM_CUDA(cudaMalloc(&h->s_b1, sizeof(float) * (64 + I_pad)));
    }
    pack_small_weight_kernel<<<18, 256, 0, st>>>(d_W1, H, L, L, 0, 64, h->s_dec1, h->s_dec1 + img);
    pack_small_weight_kernel<<<static_cast<int>(std::min<size_t>((img2 + 255) / 256, 2048)), 256, 0, st>>>(d_W2, I, H, H, 0, I_pad, h->s_dec2, h->s_dec2 + img2);
    pad_rows64_kernel<<<1, 64, 0, st>>>(d_b1, 0, H, 1, h->s_b1);
    pad_bias_kernel<<<(I_pad + 255) / 256, 256, 0, st>>>(d_b2, I, h->s_b1 + 64, I_pad);
    SDRM_CUDA(cudaGetLastError());
    h->small_dec = true;
  } else {
    h->small_dec = false;
  }
  h->have_dec = true;
  return SDRM_OK;
}

static int kb_max_of(const sdrm_handle* h) {
  int kb = 1;
  const Geom* gs[5] = {&h->g0, &h->gh, &h->go, &h->g1, &h->g2};
  const Geom* ss[4] = {&h->s0, &h->sh, &h->so, &h->s1};
  for (int i = 0; i < 4; ++i) {  // g2 writes logits, not activations
    kb = std::max(kb, gs[i]->KB);
    kb = std::max(kb, (gs[i]->Np + KBLK - 1) / KBLK);
    if (h->split_den && h->split_dec) kb = std::max(kb, (ss[i]->Np + KBLK - 1) / KBLK);   // (the column-split geometry pads wider)
  }
  kb = std::max(kb, h->g2.KB);
  return kb;
}

static void sample_geometry(const sdrm_handle* h, int64_t n, int* grid, size_t* act_bytes, size_t* stride, size_t* mask_off = nullptr,
                            int* mask_pitch = nullptr) {
  const long long n_tiles = (n + TILE_M - 1) / TILE_M;
  // upper bound over every cluster choice (a cluster launch rounds the grid up to a multiple of the cluster size)
  *grid = static_cast<int>(std::max<long long>(8, std::min<long long>((n_tiles + 7) / 8 * 8, (h->num_sms + 7) / 8 * 8)));
  *act_bytes = static_cast<size_t>(kb_max_of(h)) * A_TILE_BYTES;
  const int Lg16 = (h->L + 15) / 16;
  const size_t xs = static_cast<size_t>(Lg16) * 4 * TILE_M * 16;
  const int pitch = 16 * ((Lg16 + 7) / 8);   // one 128-bit Philox block of keep bits per 128 columns
  if (mask_off) *mask_off = NUM_ACT_BUFS * (*act_bytes) + xs;
  if (mask_pitch) *mask_pitch = pitch;
  *stride = NUM_ACT_BUFS * (*act_bytes) + xs + static_cast<size_t>(TILE_M) * pitch;
  // a CTA that owns two or more row tiles interleaves them in pairs: one scratch slot per sub-tile
  int min_res = h->num_sms;
  if (h->resident[2] > 0) min_res = std::min(min_res, h->resident[2]);
  if (n_tiles > min_res) *grid *= MAX_SUB;
}

size_t sdrm_sample_workspace_bytes(const sdrm_handle* h, int64_t n) {
  if (!h || !h->have_den || !h->have_dec || n <= 0) return 0;
  int grid; size_t act, stride;
  sample_geometry(h, n, &grid, &act, &stride);
  return static_cast<size_t>(grid) * stride;
}

}  // extern "C"

// sdrm_sample and sdrm_sample_bf16: d_logits holds fp32 or (bf16) bfloat16 logits, ld_logits counts elements either way
static int sample_impl(sdrm_handle* h, int64_t n, int64_t row_offset, const int32_t* d_t_start, const int32_t* d_row_ids,
                       uint64_t seed, float* d_x0_out, void* d_logits, int64_t ld_logits, bool bf16, const float* d_inj_xT,
                       const float* d_inj_z, const uint8_t* d_inj_mask, void* d_workspace, size_t workspace_bytes, void* stream) {
  if (!h) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_sample: null handle");
  if (!h->have_den || !h->have_dec) return sdrm_fail(SDRM_ERR_STATE, "sdrm_sample: pack denoiser and decoder first");
  if (h->g1.K != h->L) return sdrm_fail(SDRM_ERR_STATE, "sdrm_sample: decoder latent dim != denoiser latent dim");
  if (n <= 0) return SDRM_OK;
  if (!d_logits || ld_logits < h->I) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_sample: logits buffer / ld");
  if (!d_workspace) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_sample: null workspace");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaSetDevice(h->device));
  // ---- small denoisers (every width <= 64): the register / shared-memory resident chain (K6) instead of the tcgen05 engine
  const bool small_ok = h->small_den && h->small_dec && h->D <= SMALL_MAX && h->H <= SMALL_MAX;
  if (h->engine_choice == 2 && !small_ok) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_sample: the small-chain kernel needs every width <= 64");
  if (small_ok && h->engine_choice != 1) {
    SmallParams S;
    memset(&S, 0, sizeof S);
    const size_t img = static_cast<size_t>(64) * SMALL_KP;
    const size_t img2 = static_cast<size_t>((h->I + 63) / 64 * 64) * SMALL_KP;
    S.w0 = h->s_den; S.wh = h->s_den + img; S.wo = h->s_den + 2 * img;
    S.w1_hi = h->s_dec1; S.w1_lo = h->s_dec1 + img;
    S.w2_hi = h->s_dec2; S.w2_lo = h->s_dec2 + img2;
    S.bias0 = h->s_bias; S.bias0_ld = 64;
    S.bh = h->s_bias + 64 * (h->T + 1); S.bo = h->s_bias + 64 * (h->T + 2); S.b1 = h->s_b1; S.b2 = h->s_b1 + 64;
    S.slopes = h->slopes; S.coef = h->coef;
    S.T = h->T; S.L = h->L; S.H = h->H; S.I = h->I; S.nh = h->nh;
    S.n_rows = n; S.row_offset = row_offset; S.ld_logits = ld_logits;
    S.t_start = d_t_start; S.row_ids = d_row_ids; S.x0_out = d_x0_out; S.logits = d_logits;
    S.inj_xT = d_inj_xT; S.inj_z = d_inj_z; S.inj_mask = d_inj_mask; S.seed = seed;
    const int widest = std::max(std::max(h->L, h->D), h->H);
    const int nt = (widest + 7) / 8;
    const long long ctas = (n + 16 * SMALL_WARPS - 1) / (16 * SMALL_WARPS);
    if (ctas > 0x7fffffffLL) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_sample: too many rows for one launch");
    auto launch = [&](auto kernel, int smem) -> int {
      SDRM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      kernel<<<static_cast<unsigned>(ctas), SMALL_THREADS, smem, st>>>(S);
      SDRM_CUDA(cudaGetLastError());
      return SDRM_OK;
    };
    int rc_s;
    if (bf16) {
      rc_s = launch_small_chain_bf16(S, nt, static_cast<unsigned>(ctas), st);
    } else {
      if (nt <= 3) rc_s = launch(sdrm_small_chain_kernel<3>, SmallGeom<3>::SMEM_BYTES);
      else if (nt <= 5) rc_s = launch(sdrm_small_chain_kernel<5>, SmallGeom<5>::SMEM_BYTES);
      else rc_s = launch(sdrm_small_chain_kernel<8>, SmallGeom<8>::SMEM_BYTES);
    }
    if (rc_s) return rc_s;
    h->last_launches = 1;
    h->last_cluster = 0;   // 0 = not the cluster engine
    return SDRM_OK;
  }
  int grid, mask_pitch; size_t act, stride, mask_off;
  sample_geometry(h, n, &grid, &act, &stride, &mask_off, &mask_pitch);
  if (workspace_bytes < static_cast<size_t>(grid) * stride) return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_sample: workspace too small");
  int rc = engine_set_smem_attr();
  if (rc) return rc;

  ChainParams P;
  memset(&P, 0, sizeof P);
  auto fill = [](LayerDesc& d, const uint8_t* w, const float* bias, const float* slope, int bstride, const Geom& g,
                 int passes, int kind, int in_hi, int in_lo, int out_hi, int out_lo) {
    d.w_img = w; d.bias = bias; d.slope = slope; d.bias_step_stride = bstride;
    d.KB = g.KB; d.kmma_last = g.kmma_last; d.passes = passes; d.NCH = g.NCH; d.NC = g.NC; d.kind = kind;
    d.in_hi = in_hi; d.in_lo = in_lo; d.out_hi = out_hi; d.out_lo = out_lo; d.n_valid = g.N;
  };
  // chain layers ping-pong between activation buffers 0/1 (the kernel derives the parity); decoder descriptors name
  // their hi buffers RELATIVE to the chain's last output (0 = that buffer, 1 = the other), lo buffers are 2 and 3
  // Column-split mode (see the kernel): launches of a FEW row tiles (the dataset-sized calls of the reference: the latency
  // regime).  A cluster of S CTAs per tile, CTA j computes the chunks c = j (mod S); one tile per cluster, all clusters resident
  // at once.  Preferred: S = 8 in the 8-chunk geometry (second set of weight images); when 8 CTAs per tile do not fit, the largest
  // S = 4 / 2 that does, in the normal geometry (denoisers of >= 2 chunks).  Measured against the pair flows on every BASELINE
  // configuration and on mid-size launches up to 74 tiles (profiles/k1_split_r02.txt): always faster.
  const long long n_tiles = (n + TILE_M - 1) / TILE_M;
  int split = 0;
  bool split_geom = false;
  {
    int nch_min = std::min(h->g0.NCH, h->go.NCH), nch_max = std::max(h->g0.NCH, h->go.NCH);
    if (h->nh > 0) { nch_min = std::min(nch_min, h->gh.NCH); nch_max = std::max(nch_max, h->gh.NCH); }
    const int ov = h->cluster_override;
    auto fits = [&](int S) {
      return h->split_resident[S] > 0 && n_tiles * S <= h->split_resident[S] && (h->grid_limit == 0 || n_tiles * S <= h->grid_limit);
    };
    // (multi-resolution chains too: the tile's start step is the maximum over its rows in every CTA of the cluster alike)
    if (!h->no_split && (ov == 0 || ov >= 4) && std::max(h->L, h->D) > SMALL_MAX) {
      const bool geom8 = h->split_den && h->split_dec;
      const int s_norm = nch_max <= 2 ? 2 : nch_max <= 4 ? 4 : 8;   // cluster size that gives every chunk of the normal geometry its CTA
      if ((ov == 0 || ov == 8) && fits(8) && (geom8 || nch_max > 4)) { split = 8; split_geom = geom8; }
      else if (ov == 4 && fits(4)) split = 4;
      else if (ov == 0 && nch_min >= 2) {
        // more tiles than clusters of that size fit: smaller clusters, each CTA takes several chunks of a layer (c = j, j + S, ...)
        for (int S = std::min(s_norm, 4); S >= 2 && !split; S >>= 1)
          if (fits(S)) split = S;
      }
    }
  }
  h->last_split = split;
  const Geom& G0 = split_geom ? h->s0 : h->g0;
  const Geom& GH = split_geom ? h->sh : h->gh;
  const Geom& GO = split_geom ? h->so : h->go;
  const Geom& G1 = split_geom ? h->s1 : h->g1;
  const Geom& G2 = split_geom ? h->s2 : h->g2;
  int l = 0;
  fill(P.step[l++], split_geom ? h->w0s : h->w0, h->bias0, h->slopes, h->np0, G0, 1, EPI_PRELU, 0, 0, 0, 0);
  for (int j = 0; j < h->nh; ++j) fill(P.step[l++], split_geom ? h->whs : h->wh, h->bh, h->slopes + 1, 0, GH, 1, EPI_PRELU, 0, 0, 0, 0);
  fill(P.step[l++], split_geom ? h->wos : h->wo, h->bo, nullptr, 0, GO, 1, EPI_POSTERIOR, 0, 0, 0, 0);
  P.n_step = l;
  fill(P.dec[0], (split_geom && h->w1s) ? h->w1s : h->w1, h->b1, nullptr, 0, G1, 3, EPI_TANH_SPLIT, 0, 2, 1, 3);
  fill(P.dec[1], (split_geom && h->w2s) ? h->w2s : h->w2, h->b2, nullptr, 0, G2, 3, EPI_LINEAR_OUT, 1, 3, 0, 0);
  P.n_dec = 2;
  P.T = h->T; P.L = h->L; P.Lg16 = (h->L + 15) / 16;
  P.preloaded_input = 0;
  P.n_rows = n; P.row_offset = row_offset;
  P.coef = h->coef;
  P.t_start = d_t_start;
  P.row_ids = d_row_ids;
  P.x0_out = d_x0_out;
  P.logits = d_logits; P.ld_logits = ld_logits;
  P.inj_xT = d_inj_xT; P.inj_z = d_inj_z; P.inj_mask = d_inj_mask;
  P.seed = seed;
  P.scratch = static_cast<uint8_t*>(d_workspace);
  P.scratch_stride = stride;
  P.act_buf_bytes = act;
  P.mask_off = mask_off;
  P.mask_pitch = mask_pitch;
  P.err_word = h->err_word;
  P.trace = h->trace;
  P.debug_flags = h->debug_flags;
  int cluster = 1;
  // full-resolution chains run on tcgen05 cta_group::2 CTA pairs (fewer weight bytes and more k-blocks in flight per SM);
  // multi-resolution chains (per-tile step counts) and single-tile calls use single-CTA mode
  // (multi-resolution chains too since the third r02 session: a pair runs the longer of its two tiles' chains)
  if (n_tiles >= 2) cluster = 2;
  if (h->cluster_override == 1 || h->cluster_override == 2) cluster = h->cluster_override;
  int launch_grid = 0;
  if (split) { cluster = 1; launch_grid = static_cast<int>(n_tiles) * split; }
  else
  for (; cluster >= 1; cluster >>= 1) {
    const int resident = h->resident[cluster];
    if (resident <= 0) continue;
    const long long want = (n_tiles + cluster - 1) / cluster * cluster;
    launch_grid = static_cast<int>(std::min<long long>(want, resident));
    if (h->grid_limit > 0) launch_grid = std::min(launch_grid, std::max(cluster, h->grid_limit / cluster * cluster));
    break;
  }
  if (launch_grid <= 0 || (split ? n_tiles > grid : launch_grid > grid)) return sdrm_fail(SDRM_ERR_CUDA, "sdrm_sample: no launchable grid");
  h->last_cluster = cluster;
  rc = fill_act_maps(P, static_cast<size_t>(grid) * stride);
  if (rc) return rc;
  if (cluster >= 2) {
    rc = fill_pair_maps(P, static_cast<size_t>(grid) * stride, cluster);
    if (rc) return rc;
  }
  // Sub-tiles: a pair that owns two or more row tiles interleaves two of them layer by layer (see the kernel)
  const long long n_local = split ? 1 : (n_tiles + launch_grid - 1) / launch_grid;
  // Which of the three data flows a pair-mode launch takes (all bit-identical), measured on B200 with tools/shape_probe.py:
  //   * two interleaved sub-tiles per CTA (streaming through the L2): narrow denoisers with several tiles per CTA.  A layer's UMMAs
  //     are short there and the hand-off of a tile's layer hides behind the other tile's work: L = 96 / 128 / 200 / 264 / 300 at
  //     80 000 - 150 000 users: +21 / +18 / +10 / +6.5 / +2.5 % over the best single-tile flow.  From ~320 columns on it loses (the
  //     second tile doubles the scratch and the L2 traffic: cfg-2 widths -5 %, cfg 5 -8 % with the L2 hit rate down from 80 to 67 %);
  //   * resident mode (below): everything else that fits it, except one-tile-per-CTA launches of very narrow denoisers (<= 128
  //     columns: 0.798 vs 0.824 ms, the tile hand-off through the L2 is as fast and the weight stream keeps all 6 stages);
  //   * one streaming tile per CTA: the wide denoisers (cfg 1, cfg 5).
  int w_max = 0;
  for (int j = 0; j < P.n_step; ++j) w_max = std::max(w_max, std::max(P.step[j].KB * KBLK, P.step[j].NCH * P.step[j].NC));
  P.n_sub = 1;
  if (cluster == 2 && n_local >= 2 && P.n_step > 0 && d_t_start == nullptr &&   // (multi-resolution pairs: one tile at a time)
      (h->subtile_override == 2 || (h->subtile_override == 0 && w_max <= 320)))
    P.n_sub = 2;
  // Dead-buffer discard (pair mode, see the kernel's discard warp): whole k-blocks of a chain layer's input image that EVERY
  // chain layer's epilogue rewrites completely (64-column blocks below the narrowest written width), so a partly written
  // last k-block keeps the zero padding it got at kernel start.
  P.discard_kb = 0;
  if (cluster >= 2 && !h->no_discard && h->T >= 2 && d_t_start == nullptr) {   // (the discard warp counts P.T steps per tile)
    const int written = std::min(std::min(h->g0.Np, h->nh > 0 ? h->gh.Np : h->g0.Np), std::min(h->go.Np, P.Lg16 * 16));
    const int kb_read = std::min(std::min(h->g0.KB, h->nh > 0 ? h->gh.KB : h->g0.KB), h->go.KB);
    P.discard_kb = std::max(0, std::min(written / KBLK, kb_read));
  }
  // Resident mode (see the kernel): every chain layer fits one pass of the accumulators (N <= 2 chunks = 512 TMEM columns) and
  // the part of the stage ring the weight stream can spare (<= 8 k-blocks).  Built for the latency regime (one row tile per CTA:
  // cfg 4 1.40 -> 1.31 ms), it also wins when a CTA owns several tiles: at these widths the streaming path is bound by L2 bandwidth
  // (~9 TB/s of activation re-reads, weights, stores and state at 148 CTAs), and the resident tile removes the activation half of it
  // (cfg-2 widths, 100 000 users: 14.91 -> 14.39 ms; cfg-4 widths, 60 000 users: 5.55 -> 5.26 ms).
  P.resident = 0; P.res_nstg = 0;
  if (cluster == 2 && P.n_sub == 1 && P.n_step > 0 && h->no_resident != 1 && d_t_start == nullptr && (n_local >= 2 || w_max > 128)) {
    int kb_max = 0;
    bool ok = true;
    for (int j = 0; j < P.n_step; ++j) {
      const LayerDesc& d = P.step[j];
      ok = ok && d.NCH <= 2 && d.passes == 1;
      kb_max = std::max(kb_max, std::max(d.KB, (d.NCH * d.NC + KBLK - 1) / KBLK));
    }
    if (ok && kb_max <= 8) {
      P.resident = 1;
      P.res_nstg = kb_max <= 6 ? 3 : 2;
      P.discard_kb = 0;
    }
  }
  h->last_resident = P.resident;
  if (split) {
    int nc_max = 16;
    for (int j = 0; j < P.n_step; ++j) nc_max = std::max(nc_max, P.step[j].NC);
    for (int j = 0; j < P.n_dec; ++j) nc_max = std::max(nc_max, P.dec[j].NC);
    P.split_stage_bytes = static_cast<uint32_t>(A_TILE_BYTES + (nc_max * 128 + 1023) / 1024 * 1024);
    P.res_nstg = std::max(1, std::min(6, static_cast<int>(4u * STAGE_BYTES / P.split_stage_bytes)));
  }
  if (static_cast<size_t>(split ? n_tiles : launch_grid) * P.n_sub * stride > workspace_bytes)
    return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_sample: workspace too small for the sub-tile scratch slots");
  rc = launch_engine(P, launch_grid, cluster, st, split, bf16);
  if (rc) return rc;
  h->last_launches = 1;
  return SDRM_OK;
}

extern "C" {

int sdrm_sample(sdrm_handle* h, int64_t n, int64_t row_offset, const int32_t* d_t_start, const int32_t* d_row_ids,
                uint64_t seed,
                float* d_x0_out, float* d_logits, int64_t ld_logits, const float* d_inj_xT, const float* d_inj_z,
                const uint8_t* d_inj_mask, void* d_workspace, size_t workspace_bytes, void* stream) {
  return sample_impl(h, n, row_offset, d_t_start, d_row_ids, seed, d_x0_out, d_logits, ld_logits, false, d_inj_xT, d_inj_z,
                     d_inj_mask, d_workspace, workspace_bytes, stream);
}

int sdrm_sample_bf16(sdrm_handle* h, int64_t n, int64_t row_offset, const int32_t* d_t_start, const int32_t* d_row_ids,
                     uint64_t seed, float* d_x0_out, uint16_t* d_logits, int64_t ld_logits, const float* d_inj_xT,
                     const float* d_inj_z, const uint8_t* d_inj_mask, void* d_workspace, size_t workspace_bytes, void* stream) {
  return sample_impl(h, n, row_offset, d_t_start, d_row_ids, seed, d_x0_out, d_logits, ld_logits, true, d_inj_xT, d_inj_z,
                     d_inj_mask, d_workspace, workspace_bytes, stream);
}

int sdrm_last_launch_count(const sdrm_handle* h) { return h ? h->last_launches : 0; }
int sdrm_last_resident_mode(const sdrm_handle* h) { return h ? h->last_resident : 0; }
int sdrm_last_split_size(const sdrm_handle* h) { return h ? h->last_split : 0; }

int sdrm_check_device_error(sdrm_handle* h, void* stream) {
  if (!h) return sdrm_fail(SDRM_ERR_BAD_ARG, "null handle");
  cudaError_t e = cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
  const int word = h->err_host ? *h->err_host : 0;
  if (e != cudaSuccess || word != 0) {
    char msg[200];
    volatile int* w = h->err_host;
    snprintf(msg, sizeof msg, "device error: sync=%s watchdog=%d (first mbarrier wait that timed out, layer_engine.cuh WD_*; stuck roles: "
             "producers %d, umma %d, epilogue %d, noise %d, discard %d)", cudaGetErrorString(e), word, w[1], w[2], w[3], w[4], w[6]);
    return sdrm_fail(SDRM_ERR_CUDA, msg);
  }
  return SDRM_OK;
}

// ---- probe: one dense layer through the engine -------------------------------------------------
static void probe_geometry(int64_t M, int K, int N, Geom* g, size_t* act, size_t* w_off, size_t* b_off,
                           size_t* s_off, size_t* total) {
  *g = make_geom(N, K);
  *act = static_cast<size_t>(g->KB) * A_TILE_BYTES;
  const long long n_tiles = (M + TILE_M - 1) / TILE_M;
  size_t off = 256;  // err word
  *w_off = off; off += 2 * g->img_bytes();
  *b_off = off; off += sizeof(float) * g->Np; off = (off + 1023) & ~static_cast<size_t>(1023);
  *s_off = off; off += static_cast<size_t>(n_tiles) * 2 * (*act);
  *total = off;
}

int sdrm_set_option(sdrm_handle* h, int option, int64_t value) {
  if (!h) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_option: null handle");
  const int v = static_cast<int>(value);
  switch (option) {
    case SDRM_OPT_NO_SPLIT:
      h->no_split = v != 0;
      return SDRM_OK;
    case SDRM_OPT_CLUSTER:
      if (!(v == 0 || v == 1 || v == 2 || v == 4 || v == 8)) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_option: cluster must be 0 (automatic), 1, 2, or 4 / 8 (column split)");
      h->cluster_override = v;
      return SDRM_OK;
    case SDRM_OPT_SUBTILES:
      if (v < 0 || v > 2) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_option: subtiles must be 0, 1 or 2");
      h->subtile_override = v;
      return SDRM_OK;
    case SDRM_OPT_GRID_LIMIT:
      h->grid_limit = v > 0 ? v : 0;
      return SDRM_OK;
    case SDRM_OPT_NO_DISCARD:
      h->no_discard = v != 0;
      return SDRM_OK;
    case SDRM_OPT_RESIDENT:
      if (v < 0 || v > 1) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_option: resident must be 0 (automatic) or 1 (off)");
      h->no_resident = v;
      return SDRM_OK;
    case SDRM_OPT_ENGINE:
      if (v < 0 || v > 2) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_option: engine must be 0 (auto), 1 (tcgen05 layer engine) or 2 (small-chain kernel)");
      h->engine_choice = v;
      return SDRM_OK;
    case SDRM_OPT_DEBUG_FLAGS:
#ifdef SDRM_PERF_DEBUG
      h->debug_flags = v;
      return SDRM_OK;
#else
      return v == 0 ? SDRM_OK : sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_set_option: debug flags need a -DSDRM_PERF_DEBUG build");
#endif
    case SDRM_OPT_TRACE_BUFFER:
#ifdef SDRM_TRACE
      h->trace = reinterpret_cast<unsigned long long*>(static_cast<uintptr_t>(value));
      return SDRM_OK;
#else
      return value == 0 ? SDRM_OK : sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_set_option: the event timeline needs a -DSDRM_TRACE build");
#endif
    default:
      return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_option: unknown option");
  }
}
int sdrm_resident_ctas(const sdrm_handle* h, int cluster) { return (h && cluster >= 1 && cluster <= 8) ? h->resident[cluster] : 0; }
int sdrm_last_cluster_size(const sdrm_handle* h) { return h ? h->last_cluster : 0; }

int sdrm_layer_geometry(int N, int K, int column_split, int* n_chunks, int* chunk_cols, int* k_blocks) {
  if (N < 1 || K < 1 || !n_chunks || !chunk_cols || !k_blocks) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_layer_geometry: bad argument");
  const Geom g = column_split ? make_geom_split(N, K) : make_geom(N, K);
  *n_chunks = g.NCH; *chunk_cols = g.NC; *k_blocks = g.KB;
  return SDRM_OK;
}

size_t sdrm_probe_linear_workspace_bytes(int64_t M, int K, int N) {
  if (M <= 0 || K <= 0 || N <= 0) return 0;
  Geom g; size_t act, w, b, s, total;
  probe_geometry(M, K, N, &g, &act, &w, &b, &s, &total);
  return total;
}

int sdrm_probe_linear(const float* d_A, const float* d_W, const float* d_bias, float* d_out, int64_t M, int K, int N,
                      int split3, void* d_workspace, size_t workspace_bytes, void* stream) {
  if (!d_A || !d_W || !d_out || !d_workspace) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_probe_linear: null pointer");
  if (M <= 0 || K <= 0 || N <= 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_probe_linear: bad shape");
  Geom g; size_t act, w_off, b_off, s_off, total;
  probe_geometry(M, K, N, &g, &act, &w_off, &b_off, &s_off, &total);
  if (workspace_bytes < total) return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_probe_linear: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = engine_set_smem_attr();
  if (rc) return rc;
  int dev = 0, sms = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  SDRM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  uint8_t* ws = static_cast<uint8_t*>(d_workspace);
  SDRM_CUDA(cudaMemsetAsync(ws, 0, 256, st));
  launch_pack_weight(d_W, N, K, K, 0, ws + w_off, ws + w_off + g.img_bytes(), g, st);
  pad_bias_kernel<<<(g.Np + 255) / 256, 256, 0, st>>>(d_bias, N, reinterpret_cast<float*>(ws + b_off), g.Np);
  const long long n_tiles = (M + TILE_M - 1) / TILE_M;
  {
    const long long total_chunks = n_tiles * g.KB * TILE_M * 8;
    const int blocks = static_cast<int>(std::min<long long>((total_chunks + 255) / 256, 8192));
    pack_act_kernel<<<blocks, 256, 0, st>>>(d_A, M, K, ws + s_off, 2 * act, act, g.KB);
  }
  ChainParams P;
  memset(&P, 0, sizeof P);
  LayerDesc& d = P.dec[0];
  d.w_img = ws + w_off; d.bias = reinterpret_cast<const float*>(ws + b_off); d.slope = nullptr;
  d.bias_step_stride = 0; d.KB = g.KB; d.kmma_last = g.kmma_last; d.passes = split3 ? 3 : 1;
  d.NCH = g.NCH; d.NC = g.NC; d.kind = EPI_LINEAR_OUT; d.in_hi = 0; d.in_lo = 1; d.out_hi = 0; d.out_lo = 0;
  d.n_valid = N;
  P.n_step = 0; P.n_dec = 1; P.T = 0; P.L = K; P.Lg16 = 0; P.preloaded_input = 1; P.n_sub = 1;
  P.n_rows = M; P.row_offset = 0;
  P.logits = d_out; P.ld_logits = N;
  P.scratch = ws + s_off; P.scratch_stride = 2 * act; P.act_buf_bytes = act;
  P.err_word = reinterpret_cast<int*>(ws);
  const int grid = static_cast<int>(std::max<long long>(1, std::min<long long>(n_tiles, sms)));
  rc = fill_act_maps(P, static_cast<size_t>(n_tiles) * 2 * act);
  if (rc) return rc;
  return launch_engine(P, grid, 1, st);
}

}  // extern "C"
