// Host side of K1: weight / bias packing kernels and the C-ABI entry points that drive the
// layer engine (sdrm_create, sdrm_denoiser_pack, sdrm_decoder_pack, sdrm_sample, sdrm_probe_linear).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

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

// Coefficient rows of a step grid (sdrm_set_step_grid) in coef_kernel's layout: row j (1 <= j <= S) is the jump
// tau_j -> tau_{j-1} of the S-step chain, row 0 is zero.  tau [S+1] with tau_0 = 0; sched = b | a | ab as packed.
//   mode 0 (strided DDPM): a span of one step is coef_kernel's row tau_j (same float32 expressions, so the full grid
//     reproduces the packed table bit for bit); a longer span takes a' = prod a_t over (tau_{j-1}, tau_j] in float64 and
//     c0 = (1 - a') / sqrt(1 - ab_{tau_j}), c1 = 1 / sqrt(a'), c2 = sqrt(1 - a') nd, rounded once.
//   mode 1 (DDIM, eta): c1 = sqrt(ab_p / ab_c), c0 = sqrt(1 - ab_c) - sqrt(max(0, 1 - ab_p - sigma^2)) / c1, c2 = sigma nd with
//     sigma = eta sqrt((1 - ab_p) / (1 - ab_c)) sqrt(1 - ab_c / ab_p), ab_p = 1 at tau_0; float64, rounded once.
// The last step (j = 1) draws no noise in either mode.
__global__ void grid_coef_kernel(const float* __restrict__ sched, int T, const int32_t* __restrict__ tau, int S, int mode,
                                 float eta, float nd, float* __restrict__ coef) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > S) return;
  const float *b_t = sched, *a_t = sched + (T + 1), *ab_t = sched + 2 * (T + 1);
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (j >= 1) {
    const int tc = tau[j], tp = tau[j - 1];
    if (mode == 0 && tc - tp == 1) {
      const float b = b_t[tc], a = a_t[tc], ab = ab_t[tc];
      c.x = (1.0f - a) / sqrtf(1.0f - ab);
      c.y = 1.0f / sqrtf(a);
      c.z = j > 1 ? sqrtf(b) * nd : 0.0f;
    } else if (mode == 0) {
      double ap = 1.0;
      for (int t = tp + 1; t <= tc; ++t) ap *= static_cast<double>(a_t[t]);
      c.x = static_cast<float>((1.0 - ap) / sqrt(1.0 - static_cast<double>(ab_t[tc])));
      c.y = static_cast<float>(1.0 / sqrt(ap));
      c.z = j > 1 ? static_cast<float>(sqrt(1.0 - ap) * static_cast<double>(nd)) : 0.0f;
    } else {
      const double abc = ab_t[tc], abp = tp == 0 ? 1.0 : static_cast<double>(ab_t[tp]);
      const double sigma = static_cast<double>(eta) * sqrt((1.0 - abp) / (1.0 - abc)) * sqrt(fmax(0.0, 1.0 - abc / abp));
      const double c1 = sqrt(abp / abc);
      c.x = static_cast<float>(sqrt(1.0 - abc) - sqrt(fmax(0.0, 1.0 - abp - sigma * sigma)) / c1);
      c.y = static_cast<float>(c1);
      c.z = static_cast<float>(sigma * static_cast<double>(nd));
    }
  }
  reinterpret_cast<float4*>(coef)[j] = c;
}

// rows tau_0 .. tau_S of a per-step bias table [T+1][ld] -> rows 0 .. S of the grid's table (same pitch): one block per row
__global__ void grid_bias_kernel(const float* __restrict__ src, int ld, const int32_t* __restrict__ tau, float* __restrict__ dst) {
  const float* s = src + static_cast<size_t>(tau[blockIdx.x]) * ld;
  float* d = dst + static_cast<size_t>(blockIdx.x) * ld;
  for (int c = threadIdx.x; c < ld; c += blockDim.x) d[c] = s[c];
}

static void launch_pack_weight(const float* W, int N, int K, long long ldw, int col_off, uint8_t* hi, uint8_t* lo,
                               const Geom& g, cudaStream_t st) {
  const long long total = static_cast<long long>(g.NCH) * g.KB * g.NC * 8;
  const int blocks = static_cast<int>(std::min<long long>((total + 255) / 256, 4096));
  pack_weight_kernel<<<blocks, 256, 0, st>>>(W, N, K, ldw, col_off, hi, lo, g.NCH, g.NC, g.KB);
}

}  // namespace sdrm

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
using namespace sdrm;

// One dense layer packed for the engine, in the normal geometry [0] and in the 8-chunk geometry of the column split [1].
// img[1] stays null when the split set is not packed or its geometry is the normal one; img[0] then serves.
struct PackedLayer {
  Geom g[2];
  uint8_t* img[2] = {nullptr, nullptr};
  int np = 0;                 // padded bias width (both geometries fit)
  float* bias = nullptr;      // [np]; the first layer's is the per-step table [T+1][np]
  const uint8_t* image(bool split_geom) const { return split_geom && img[1] ? img[1] : img[0]; }
};
enum { LAYER_FIRST, LAYER_HIDDEN, LAYER_OUT, LAYER_DEC1, LAYER_DEC2, N_LAYERS };   // denoiser: FIRST .. OUT, decoder: DEC1, DEC2

// How one sdrm_sample launch runs (every data flow gives bit-identical rows); plan_launch chooses it
struct LaunchPlan {
  bool k6 = false;              // the small-chain kernel instead of the tcgen05 layer engine (K1)
  int cluster = 1;              // K1: CTAs of a tcgen05 tile (1 or 2; 1 for the column split); 0 for K6
  int split = 0;                // K1 column split: CTAs per row tile (8 / 4 / 2), 0 = not split
  bool split_geom = false;      // the column split runs on the 8-chunk images
  int grid = 0;                 // K1 CTAs
  int n_sub = 1;                // row tiles a CTA pair interleaves
  int resident = 0, res_nstg = 0, discard_kb = 0;
  uint32_t split_stage_bytes = 0;
};

struct sdrm_handle {
  int device = 0;
  int num_sms = 0;
  int last_launches = 0;
  LaunchPlan last;              // what the last sdrm_sample launch did
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
  int grid_limit = 0;           // cap on the CTAs of an sdrm_sample launch (tests: small inputs exercise the multi-tile loops)
  int debug_flags = 0;          // -DSDRM_PERF_DEBUG builds only
  unsigned long long* trace = nullptr;   // -DSDRM_TRACE builds only
  PackedLayer layer[N_LAYERS];
  // denoiser
  bool have_den = false;
  int T = 0, L = 0, D = 0, nh = 0;
  float nd = 1.0f;
  float *slopes = nullptr, *coef = nullptr;
  // K6 (small denoisers, small_chain_kernel.cuh): zero-padded bf16 images and 64-wide bias rows, packed when every width <= 64
  bool small_den = false, small_dec = false;
  __nv_bfloat16 *s_den = nullptr;   // w0 | wh | wo, each [64][SMALL_KP]
  __nv_bfloat16 *s_dec1 = nullptr;  // w1 hi | w1 lo
  __nv_bfloat16 *s_dec2 = nullptr;  // w2 hi | w2 lo, each [I rounded up to 64][SMALL_KP]
  float *s_bias = nullptr;          // bias0 [T+1][64] | bh [64] | bo [64]
  float *s_b1 = nullptr;            // b1 [64] | b2 [I rounded up to 64]
  int engine_choice = 0;            // SDRM_OPT_ENGINE: 0 automatic, 1 tcgen05 layer engine, 2 small-chain kernel
  // step grid (sdrm_set_step_grid): grid_S = 0 runs the packed full chain; else the chain has grid_S steps and reads the grid
  // tables below (rows 0 .. grid_S; sized for T + 1 rows)
  int grid_S = 0;
  float* sched = nullptr;           // the packed schedule b | a | ab [3 (T+1)]
  int32_t* grid_tau = nullptr;      // tau_0 = 0, tau_1 .. tau_S
  float *grid_bias0 = nullptr, *grid_coef = nullptr;   // first-layer bias rows tau_j [T+1][np]; coefficients [T+1][4]
  float* grid_s_bias = nullptr;     // K6: bias0 rows tau_j [T+1][64]
  // decoder
  bool have_dec = false;
  int H = 0, I = 0;
};

static void free_layers(sdrm_handle* h, int first, int last) {
  for (int l = first; l <= last; ++l) {
    PackedLayer& p = h->layer[l];
    cudaFree(p.img[0]); cudaFree(p.img[1]); cudaFree(p.bias);
    p = PackedLayer();
  }
}
static void free_den(sdrm_handle* h) {
  free_layers(h, LAYER_FIRST, LAYER_OUT);
  cudaFree(h->slopes); cudaFree(h->coef);
  cudaFree(h->s_den); cudaFree(h->s_bias);
  h->s_den = nullptr; h->s_bias = nullptr; h->small_den = false;
  cudaFree(h->sched); cudaFree(h->grid_tau); cudaFree(h->grid_bias0); cudaFree(h->grid_coef); cudaFree(h->grid_s_bias);
  h->sched = h->grid_bias0 = h->grid_coef = h->grid_s_bias = nullptr; h->grid_tau = nullptr; h->grid_S = 0;
  h->slopes = h->coef = nullptr;
  h->have_den = false;
}
static void free_dec(sdrm_handle* h) {
  free_layers(h, LAYER_DEC1, LAYER_DEC2);
  cudaFree(h->s_dec1); cudaFree(h->s_dec2); cudaFree(h->s_b1);
  h->s_dec1 = h->s_dec2 = nullptr; h->s_b1 = nullptr; h->small_dec = false;
  h->have_dec = false;
}

// The 8-chunk images are packed for a denoiser wider than 64 (narrower ones run on the small-chain kernel) whose layers they
// re-cut, and for a decoder behind a latent wider than 64 (the denoiser it follows may take the column split)
static bool split_set_packed(const sdrm_handle* h, bool decoder) {
  if (decoder) return h->layer[LAYER_DEC1].g[0].K > SMALL_MAX;
  if (std::max(h->L, h->D) <= SMALL_MAX) return false;
  for (int l = LAYER_FIRST; l <= LAYER_OUT; ++l)
    if (!same_geom(h->layer[l].g[0], h->layer[l].g[1])) return true;
  return false;
}

// Layers first .. last, of N x K weights: both geometries, the images (bf16x3: a lo image after the hi one) and the padded bias
// (the first layer's has T + 1 rows).  The 8-chunk image only where the set is packed and the geometry differs.
static int alloc_layers(sdrm_handle* h, int first, int last, const int (*NK)[2], bool bf16x3, int first_bias_rows) {
  for (int l = first; l <= last; ++l) {
    PackedLayer& p = h->layer[l];
    p.g[0] = make_geom(NK[l - first][0], NK[l - first][1]);
    p.g[1] = make_geom_split(NK[l - first][0], NK[l - first][1]);
    p.np = std::max(p.g[0].Np, p.g[1].Np);
  }
  const bool split_set = split_set_packed(h, first == LAYER_DEC1);
  for (int l = first; l <= last; ++l) {
    PackedLayer& p = h->layer[l];
    SDRM_CUDA(cudaMalloc(&p.img[0], (bf16x3 ? 2 : 1) * p.g[0].img_bytes()));
    if (split_set && !same_geom(p.g[0], p.g[1])) SDRM_CUDA(cudaMalloc(&p.img[1], (bf16x3 ? 2 : 1) * p.g[1].img_bytes()));
    SDRM_CUDA(cudaMalloc(&p.bias, sizeof(float) * (l == LAYER_FIRST ? first_bias_rows : 1) * p.np));
  }
  return SDRM_OK;
}

// W fp32 [N, ldw] (columns 0 .. K) -> the layer's images
static void pack_layer(const PackedLayer& p, const float* W, long long ldw, bool bf16x3, cudaStream_t st) {
  for (int s = 0; s < 2; ++s)
    if (p.img[s]) launch_pack_weight(W, p.g[s].N, p.g[s].K, ldw, 0, p.img[s], bf16x3 ? p.img[s] + p.g[s].img_bytes() : nullptr, p.g[s], st);
}

// resident CTAs for a cluster size (1 CTA per SM; clusters must fit inside a GPC)
static int max_resident_ctas(int cluster, int num_sms, bool split = false) {
  if (cluster == 1) return num_sms;
  if (!split && cluster != 2) return 0;
  const EngineClusterConfig c(num_sms / cluster * cluster, cluster, nullptr);
  int n = 0;
  cudaError_t e = cudaOccupancyMaxActiveClusters(&n, engine_kernel<false>(cluster, false, split), &c.cfg);
  if (e != cudaSuccess) { cudaGetLastError(); return 0; }
  return n * cluster;
}

// ---- TMA tensor maps: a blob of `rows` x 128 bytes, box = `box_rows` rows x `box_bytes`.  Weight maps (pair mode) take no
// swizzle: the weight images are pre-swizzled in global memory, so a box lands in shared memory byte-for-byte like the bulk
// copies of single mode.  The activation load map swizzles (SWIZZLE_128B), the activation store map does not.
static int make_rows_map(CUtensorMap* map, const void* base, unsigned long long rows, unsigned box_rows, unsigned box_bytes = 128,
                         bool swizzle128 = false) {
  EncodeTiledFn fn = encode_tiled_fn();
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
static int fill_pair_maps(ChainParams& P, int cluster) {
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
  return SDRM_OK;
}

// The bfloat16-logits instantiations (sdrm_sample_bf16) are compiled in engine_bf16.cu: in this translation unit they would
// perturb how the compiler optimises the fp32 kernels, whose code stays as it is.
static int launch_engine(const ChainParams& P, int grid, int cluster, cudaStream_t st, int split = 0, bool bf16 = false) {
  return bf16 ? launch_engine_bf16(P, grid, cluster, st, split) : launch_engine_t<false>(P, grid, cluster, st, split);
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
  if (engine_setup<false>() != SDRM_OK) { delete h; return SDRM_ERR_CUDA; }
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
    const int NK[3][2] = {{D, L}, {D, D}, {L, D}};   // first, hidden, out
    int rc = alloc_layers(h, LAYER_FIRST, LAYER_OUT, NK, false, T + 1);
    if (rc) return rc;
    SDRM_CUDA(cudaMalloc(&h->slopes, sizeof(float) * 2));
    SDRM_CUDA(cudaMalloc(&h->coef, sizeof(float) * 4 * (T + 1)));
    SDRM_CUDA(cudaMalloc(&h->sched, sizeof(float) * 3 * (T + 1)));
    SDRM_CUDA(cudaMalloc(&h->grid_tau, sizeof(int32_t) * (T + 1)));
    SDRM_CUDA(cudaMalloc(&h->grid_bias0, sizeof(float) * (T + 1) * h->layer[LAYER_FIRST].np));
    SDRM_CUDA(cudaMalloc(&h->grid_coef, sizeof(float) * 4 * (T + 1)));
  }
  h->grid_S = 0;   // new weights or schedule: the full chain until a grid is set again
  h->nd = noise_divider;
  SDRM_CUDA(cudaMemcpyAsync(h->sched, d_sched, sizeof(float) * 3 * (T + 1), cudaMemcpyDeviceToDevice, st));
  const PackedLayer &first = h->layer[LAYER_FIRST], &hidden = h->layer[LAYER_HIDDEN], &out = h->layer[LAYER_OUT];
  pack_layer(first, d_W0, L + T, false, st);
  if (nh > 0) pack_layer(hidden, d_Wh, D, false, st);
  pack_layer(out, d_Wo, D, false, st);
  bias_table_kernel<<<T + 1, 256, sizeof(float) * 2 * T, st>>>(d_We, d_be, d_W0, d_b0, T, L, D, first.bias, first.np);
  pad_bias_kernel<<<(hidden.np + 255) / 256, 256, 0, st>>>(nh > 0 ? d_bh : nullptr, D, hidden.bias, hidden.np);
  pad_bias_kernel<<<(out.np + 255) / 256, 256, 0, st>>>(d_bo, L, out.bias, out.np);
  SDRM_CUDA(cudaMemcpyAsync(h->slopes, d_a0, sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (nh > 0) SDRM_CUDA(cudaMemcpyAsync(h->slopes + 1, d_ah, sizeof(float), cudaMemcpyDeviceToDevice, st));
  coef_kernel<<<(T + 1 + 127) / 128, 128, 0, st>>>(d_sched, T, noise_divider, h->coef);
  SDRM_CUDA(cudaGetLastError());
  if (L <= SMALL_MAX && D <= SMALL_MAX) {   // K6 images
    const size_t img = static_cast<size_t>(64) * SMALL_KP;
    if (!h->s_den) {
      SDRM_CUDA(cudaMalloc(&h->s_den, 3 * img * sizeof(__nv_bfloat16)));
      SDRM_CUDA(cudaMalloc(&h->s_bias, sizeof(float) * 64 * (T + 3)));
      SDRM_CUDA(cudaMalloc(&h->grid_s_bias, sizeof(float) * 64 * (T + 1)));
    }
    pack_small_weight_kernel<<<18, 256, 0, st>>>(d_W0, D, L, L + T, 0, 64, h->s_den, nullptr);
    pack_small_weight_kernel<<<18, 256, 0, st>>>(nh > 0 ? d_Wh : d_Wo, nh > 0 ? D : 0, nh > 0 ? D : 0, D, 0, 64, h->s_den + img, nullptr);
    pack_small_weight_kernel<<<18, 256, 0, st>>>(d_Wo, L, D, D, 0, 64, h->s_den + 2 * img, nullptr);
    pad_rows64_kernel<<<(64 * (T + 1) + 255) / 256, 256, 0, st>>>(first.bias, first.np, D, T + 1, h->s_bias);
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
  const bool same = h->have_dec && h->layer[LAYER_DEC1].g[0].K == L && h->H == H && h->I == I;
  if (!same) {
    free_dec(h);
    h->H = H; h->I = I;
    const int NK[2][2] = {{H, L}, {I, H}};
    int rc = alloc_layers(h, LAYER_DEC1, LAYER_DEC2, NK, true, 1);
    if (rc) return rc;
  }
  const PackedLayer &dec1 = h->layer[LAYER_DEC1], &dec2 = h->layer[LAYER_DEC2];
  pack_layer(dec1, d_W1, L, true, st);
  pack_layer(dec2, d_W2, H, true, st);
  pad_bias_kernel<<<(dec1.np + 255) / 256, 256, 0, st>>>(d_b1, H, dec1.bias, dec1.np);
  pad_bias_kernel<<<(dec2.np + 255) / 256, 256, 0, st>>>(d_b2, I, dec2.bias, dec2.np);
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

// the column split may run on the 8-chunk images when both the denoiser's and the decoder's are packed
static bool geom8_packed(const sdrm_handle* h) { return split_set_packed(h, false) && split_set_packed(h, true); }

// k-blocks of the widest activation image: every layer's input, every output but the logits
static int kb_max_of(const sdrm_handle* h) {
  const bool geom8 = geom8_packed(h);
  int kb = 1;
  for (int l = 0; l < N_LAYERS; ++l) {
    const Geom *g = h->layer[l].g;
    kb = std::max(kb, g[0].KB);
    if (l == LAYER_DEC2) continue;   // writes logits, not activations
    kb = std::max(kb, (g[0].Np + KBLK - 1) / KBLK);
    if (geom8) kb = std::max(kb, (g[1].Np + KBLK - 1) / KBLK);   // (the column-split geometry pads wider)
  }
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

static void fill_desc(LayerDesc& d, const uint8_t* w, const Geom& g, const float* bias, const float* slope, int bstride, int passes,
                      int kind, int in_hi, int in_lo, int out_hi, int out_lo) {
  d.w_img = w; d.bias = bias; d.slope = slope; d.bias_step_stride = bstride;
  d.KB = g.KB; d.kmma_last = g.kmma_last; d.passes = passes; d.NCH = g.NCH; d.NC = g.NC; d.kind = kind;
  d.in_hi = in_hi; d.in_lo = in_lo; d.out_hi = out_hi; d.out_lo = out_lo; d.n_valid = g.N;
}

// the small-chain kernel (K6) takes models whose every width is <= 64
static bool small_ok(const sdrm_handle* h) { return h->small_den && h->small_dec && h->D <= SMALL_MAX && h->H <= SMALL_MAX; }

// The kernel and data flow of a launch of n rows (multires: per-row start steps; steps: reverse steps of the chain), from the
// packed geometries and the handle's options.
static LaunchPlan plan_launch(const sdrm_handle* h, int64_t n, bool multires, int steps) {
  LaunchPlan p;
  // small denoisers (every width <= 64): the register / shared-memory resident chain (K6) instead of the tcgen05 engine
  if (small_ok(h) && h->engine_choice != 1) {
    p.k6 = true;
    p.cluster = 0;   // 0 = not the cluster engine
    return p;
  }
  // the chain's layers (first, hidden when nh > 0, out) in geometry s (1 = 8-chunk)
  auto chain = [h](int s, auto f) {
    for (int l = LAYER_FIRST; l <= LAYER_OUT; ++l)
      if (l != LAYER_HIDDEN || h->nh > 0) f(h->layer[l].g[s]);
  };
  // Column-split mode (see the kernel): launches of a FEW row tiles (the dataset-sized calls of the reference: the latency
  // regime).  A cluster of S CTAs per tile, CTA j computes the chunks c = j (mod S); one tile per cluster, all clusters resident
  // at once.  Preferred: S = 8 in the 8-chunk geometry (second set of weight images); when 8 CTAs per tile do not fit, the largest
  // S = 4 / 2 that does, in the normal geometry (denoisers of >= 2 chunks).  Measured against the pair flows on every BASELINE
  // configuration and on mid-size launches up to 74 tiles (profiles/k1_split_r02.txt): always faster.
  const long long n_tiles = (n + TILE_M - 1) / TILE_M;
  {
    int nch_min = 1 << 30, nch_max = 0;
    chain(0, [&](const Geom& g) { nch_min = std::min(nch_min, g.NCH); nch_max = std::max(nch_max, g.NCH); });
    const int ov = h->cluster_override;
    auto fits = [&](int S) {
      return h->split_resident[S] > 0 && n_tiles * S <= h->split_resident[S] && (h->grid_limit == 0 || n_tiles * S <= h->grid_limit);
    };
    // (multi-resolution chains too: the tile's start step is the maximum over its rows in every CTA of the cluster alike)
    if (!h->no_split && (ov == 0 || ov >= 4) && std::max(h->L, h->D) > SMALL_MAX) {
      const bool geom8 = geom8_packed(h);
      const int s_norm = nch_max <= 2 ? 2 : nch_max <= 4 ? 4 : 8;   // cluster size that gives every chunk of the normal geometry its CTA
      if ((ov == 0 || ov == 8) && fits(8) && (geom8 || nch_max > 4)) { p.split = 8; p.split_geom = geom8; }
      else if (ov == 4 && fits(4)) p.split = 4;
      else if (ov == 0 && nch_min >= 2) {
        // more tiles than clusters of that size fit: smaller clusters, each CTA takes several chunks of a layer (c = j, j + S, ...)
        for (int S = std::min(s_norm, 4); S >= 2 && !p.split; S >>= 1)
          if (fits(S)) p.split = S;
      }
    }
  }
  if (p.split) {
    p.cluster = 1;
    p.grid = static_cast<int>(n_tiles) * p.split;
    int nc_max = 16;
    for (int l = 0; l < N_LAYERS; ++l)
      if (l != LAYER_HIDDEN || h->nh > 0) nc_max = std::max(nc_max, h->layer[l].g[p.split_geom].NC);
    p.split_stage_bytes = static_cast<uint32_t>(A_TILE_BYTES + (nc_max * 128 + 1023) / 1024 * 1024);
    p.res_nstg = std::max(1, std::min(6, static_cast<int>(4u * STAGE_BYTES / p.split_stage_bytes)));
    return p;
  }
  // full-resolution chains run on tcgen05 cta_group::2 CTA pairs (fewer weight bytes and more k-blocks in flight per SM);
  // multi-resolution chains (per-tile step counts) and single-tile calls use single-CTA mode
  // (multi-resolution chains too since the third r02 session: a pair runs the longer of its two tiles' chains)
  int cluster = n_tiles >= 2 ? 2 : 1;
  if (h->cluster_override == 1 || h->cluster_override == 2) cluster = h->cluster_override;
  for (; cluster >= 1; cluster >>= 1) {
    const int resident = h->resident[cluster];
    if (resident <= 0) continue;
    const long long want = (n_tiles + cluster - 1) / cluster * cluster;
    p.grid = static_cast<int>(std::min<long long>(want, resident));
    if (h->grid_limit > 0) p.grid = std::min(p.grid, std::max(cluster, h->grid_limit / cluster * cluster));
    break;
  }
  p.cluster = cluster;
  if (p.grid <= 0) return p;
  // Sub-tiles: a pair that owns two or more row tiles interleaves two of them layer by layer (see the kernel)
  const long long n_local = (n_tiles + p.grid - 1) / p.grid;
  // Which of the three data flows a pair-mode launch takes (all bit-identical), measured on B200 with tools/shape_probe.py:
  //   * two interleaved sub-tiles per CTA (streaming through the L2): narrow denoisers with several tiles per CTA.  A layer's UMMAs
  //     are short there and the hand-off of a tile's layer hides behind the other tile's work: L = 96 / 128 / 200 / 264 / 300 at
  //     80 000 - 150 000 users: +21 / +18 / +10 / +6.5 / +2.5 % over the best single-tile flow.  From ~320 columns on it loses (the
  //     second tile doubles the scratch and the L2 traffic: cfg-2 widths -5 %, cfg 5 -8 % with the L2 hit rate down from 80 to 67 %);
  //   * resident mode (below): everything else that fits it, except one-tile-per-CTA launches of very narrow denoisers (<= 128
  //     columns: 0.798 vs 0.824 ms, the tile hand-off through the L2 is as fast and the weight stream keeps all 6 stages);
  //   * one streaming tile per CTA: the wide denoisers (cfg 1, cfg 5).
  int w_max = 0;
  chain(0, [&](const Geom& g) { w_max = std::max(w_max, std::max(g.KB * KBLK, g.Np)); });
  if (cluster == 2 && n_local >= 2 && !multires &&   // (multi-resolution pairs: one tile at a time)
      (h->subtile_override == 2 || (h->subtile_override == 0 && w_max <= 320)))
    p.n_sub = 2;
  // Dead-buffer discard (pair mode, see the kernel's discard warp): whole k-blocks of a chain layer's input image that EVERY
  // chain layer's epilogue rewrites completely (64-column blocks below the narrowest written width), so a partly written
  // last k-block keeps the zero padding it got at kernel start.
  if (cluster >= 2 && !h->no_discard && steps >= 2 && !multires) {   // (the discard warp counts P.T steps per tile)
    int written = (h->L + 15) / 16 * 16, kb_read = 1 << 30;
    chain(0, [&](const Geom& g) { written = std::min(written, g.Np); kb_read = std::min(kb_read, g.KB); });
    p.discard_kb = std::max(0, std::min(written / KBLK, kb_read));
  }
  // Resident mode (see the kernel): every chain layer fits one pass of the accumulators (N <= 2 chunks = 512 TMEM columns) and
  // the part of the stage ring the weight stream can spare (<= 8 k-blocks).  Built for the latency regime (one row tile per CTA:
  // cfg 4 1.40 -> 1.31 ms), it also wins when a CTA owns several tiles: at these widths the streaming path is bound by L2 bandwidth
  // (~9 TB/s of activation re-reads, weights, stores and state at 148 CTAs), and the resident tile removes the activation half of it
  // (cfg-2 widths, 100 000 users: 14.91 -> 14.39 ms; cfg-4 widths, 60 000 users: 5.55 -> 5.26 ms).
  if (cluster == 2 && p.n_sub == 1 && h->no_resident != 1 && !multires && (n_local >= 2 || w_max > 128)) {
    int kb_max = 0;
    bool ok = true;
    chain(0, [&](const Geom& g) {
      ok = ok && g.NCH <= 2;
      kb_max = std::max(kb_max, std::max(g.KB, (g.Np + KBLK - 1) / KBLK));
    });
    if (ok && kb_max <= 8) {
      p.resident = 1;
      p.res_nstg = kb_max <= 6 ? 3 : 2;
      p.discard_kb = 0;
    }
  }
  return p;
}

// sdrm_sample and sdrm_sample_bf16: d_logits holds fp32 or (bf16) bfloat16 logits, ld_logits counts elements either way
static int sample_impl(sdrm_handle* h, int64_t n, int64_t row_offset, const int32_t* d_t_start, const int32_t* d_row_ids,
                       uint64_t seed, float* d_x0_out, void* d_logits, int64_t ld_logits, bool bf16, const float* d_inj_xT,
                       const float* d_inj_z, const uint8_t* d_inj_mask, void* d_workspace, size_t workspace_bytes, void* stream) {
  if (!h) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_sample: null handle");
  if (!h->have_den || !h->have_dec) return sdrm_fail(SDRM_ERR_STATE, "sdrm_sample: pack denoiser and decoder first");
  if (h->layer[LAYER_DEC1].g[0].K != h->L) return sdrm_fail(SDRM_ERR_STATE, "sdrm_sample: decoder latent dim != denoiser latent dim");
  if (n <= 0) return SDRM_OK;
  if (!d_logits || ld_logits < h->I) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_sample: logits buffer / ld");
  if (!d_workspace) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_sample: null workspace");
  if (h->engine_choice == 2 && !small_ok(h)) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_sample: the small-chain kernel needs every width <= 64");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaSetDevice(h->device));
  const bool on_grid = h->grid_S > 0;
  const int steps = on_grid ? h->grid_S : h->T;   // reverse steps of this launch (t_start entries are clamped to [0, steps])
  const LaunchPlan plan = plan_launch(h, n, d_t_start != nullptr, steps);
  if (plan.k6) {
    const long long ctas = (n + 16 * SMALL_WARPS - 1) / (16 * SMALL_WARPS);
    if (ctas > 0x7fffffffLL) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_sample: too many rows for one launch");
    SmallParams S;
    memset(&S, 0, sizeof S);
    const size_t img = static_cast<size_t>(64) * SMALL_KP;
    const size_t img2 = static_cast<size_t>((h->I + 63) / 64 * 64) * SMALL_KP;
    S.w0 = h->s_den; S.wh = h->s_den + img; S.wo = h->s_den + 2 * img;
    S.w1_hi = h->s_dec1; S.w1_lo = h->s_dec1 + img;
    S.w2_hi = h->s_dec2; S.w2_lo = h->s_dec2 + img2;
    S.bias0 = on_grid ? h->grid_s_bias : h->s_bias; S.bias0_ld = 64;
    S.bh = h->s_bias + 64 * (h->T + 1); S.bo = h->s_bias + 64 * (h->T + 2); S.b1 = h->s_b1; S.b2 = h->s_b1 + 64;
    S.slopes = h->slopes; S.coef = on_grid ? h->grid_coef : h->coef;
    S.T = steps; S.L = h->L; S.H = h->H; S.I = h->I; S.nh = h->nh;
    S.n_rows = n; S.row_offset = row_offset; S.ld_logits = ld_logits;
    S.t_start = d_t_start; S.row_ids = d_row_ids; S.x0_out = d_x0_out; S.logits = d_logits;
    S.inj_xT = d_inj_xT; S.inj_z = d_inj_z; S.inj_mask = d_inj_mask; S.seed = seed;
    const int nt = (std::max(std::max(h->L, h->D), h->H) + 7) / 8;
    const int rc = bf16 ? launch_small_chain_bf16(S, nt, static_cast<unsigned>(ctas), st)
                        : launch_small_chain_t<false>(S, nt, static_cast<unsigned>(ctas), st);
    if (rc) return rc;
    h->last = plan;
    h->last_launches = 1;
    return SDRM_OK;
  }
  int grid, mask_pitch; size_t act, stride, mask_off;
  sample_geometry(h, n, &grid, &act, &stride, &mask_off, &mask_pitch);
  if (workspace_bytes < static_cast<size_t>(grid) * stride) return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_sample: workspace too small");
  const long long n_tiles = (n + TILE_M - 1) / TILE_M;
  if (plan.grid <= 0 || (plan.split ? n_tiles > grid : plan.grid > grid)) return sdrm_fail(SDRM_ERR_CUDA, "sdrm_sample: no launchable grid");
  if (static_cast<size_t>(plan.split ? n_tiles : plan.grid) * plan.n_sub * stride > workspace_bytes)
    return sdrm_fail(SDRM_ERR_WORKSPACE, "sdrm_sample: workspace too small for the sub-tile scratch slots");

  ChainParams P;
  memset(&P, 0, sizeof P);
  // chain layers (first, nh x the shared hidden one, out) ping-pong between activation buffers 0/1 (the kernel derives the
  // parity); decoder descriptors name their hi buffers RELATIVE to the chain's last output (0 = that buffer, 1 = the other),
  // lo buffers are 2 and 3
  const bool sg = plan.split_geom;
  P.n_step = 2 + h->nh;
  for (int j = 0; j < P.n_step; ++j) {
    const int l = j == 0 ? LAYER_FIRST : j <= h->nh ? LAYER_HIDDEN : LAYER_OUT;
    const PackedLayer& q = h->layer[l];
    if (l == LAYER_FIRST)
      fill_desc(P.step[j], q.image(sg), q.g[sg], on_grid ? h->grid_bias0 : q.bias, h->slopes, q.np, 1, EPI_PRELU, 0, 0, 0, 0);
    else if (l == LAYER_HIDDEN)
      fill_desc(P.step[j], q.image(sg), q.g[sg], q.bias, h->slopes + 1, 0, 1, EPI_PRELU, 0, 0, 0, 0);
    else
      fill_desc(P.step[j], q.image(sg), q.g[sg], q.bias, nullptr, 0, 1, EPI_POSTERIOR, 0, 0, 0, 0);
  }
  const PackedLayer &dec1 = h->layer[LAYER_DEC1], &dec2 = h->layer[LAYER_DEC2];
  fill_desc(P.dec[0], dec1.image(sg), dec1.g[sg], dec1.bias, nullptr, 0, 3, EPI_TANH_SPLIT, 0, 2, 1, 3);
  fill_desc(P.dec[1], dec2.image(sg), dec2.g[sg], dec2.bias, nullptr, 0, 3, EPI_LINEAR_OUT, 1, 3, 0, 0);
  P.n_dec = 2;
  P.T = steps; P.L = h->L; P.Lg16 = (h->L + 15) / 16;
  P.preloaded_input = 0;
  P.n_rows = n; P.row_offset = row_offset;
  P.coef = on_grid ? h->grid_coef : h->coef;
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
  P.n_sub = plan.n_sub;
  P.resident = plan.resident;
  P.res_nstg = plan.res_nstg;
  P.discard_kb = plan.discard_kb;
  P.split_stage_bytes = plan.split_stage_bytes;
  int rc = fill_act_maps(P, static_cast<size_t>(grid) * stride);
  if (rc) return rc;
  if (plan.cluster >= 2) {
    rc = fill_pair_maps(P, plan.cluster);
    if (rc) return rc;
  }
  h->last = plan;
  rc = launch_engine(P, plan.grid, plan.cluster, st, plan.split, bf16);
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

int sdrm_set_step_grid(sdrm_handle* h, const int32_t* timesteps, int S, int mode, float eta, void* stream) {
  if (!h) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_step_grid: null handle");
  if (!h->have_den) return sdrm_fail(SDRM_ERR_STATE, "sdrm_set_step_grid: pack the denoiser first");
  if (S < 0 || S > h->T) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_step_grid: S must lie in [0, T]");
  if (mode != 0 && mode != 1) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_step_grid: mode must be 0 (strided DDPM) or 1 (DDIM)");
  if (!(eta >= 0.0f && eta <= 1.0f)) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_step_grid: eta must lie in [0, 1]");
  if (S == 0) { h->grid_S = 0; return SDRM_OK; }
  if (!timesteps) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_step_grid: null timesteps");
  std::vector<int32_t> tau(static_cast<size_t>(S) + 1, 0);
  for (int j = 0; j < S; ++j) {
    if (timesteps[j] < 1 || timesteps[j] > h->T || timesteps[j] <= tau[j])
      return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_set_step_grid: timesteps must increase strictly within [1, T]");
    tau[j + 1] = timesteps[j];
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SDRM_CUDA(cudaSetDevice(h->device));
  // (pageable source: the copy is staged before this call returns)
  SDRM_CUDA(cudaMemcpyAsync(h->grid_tau, tau.data(), sizeof(int32_t) * (S + 1), cudaMemcpyHostToDevice, st));
  grid_coef_kernel<<<(S + 1 + 127) / 128, 128, 0, st>>>(h->sched, h->T, h->grid_tau, S, mode, eta, h->nd, h->grid_coef);
  const PackedLayer& first = h->layer[LAYER_FIRST];
  grid_bias_kernel<<<S + 1, 256, 0, st>>>(first.bias, first.np, h->grid_tau, h->grid_bias0);
  if (h->small_den) grid_bias_kernel<<<S + 1, 64, 0, st>>>(h->s_bias, 64, h->grid_tau, h->grid_s_bias);
  SDRM_CUDA(cudaGetLastError());
  h->grid_S = S;
  return SDRM_OK;
}

int sdrm_step_grid_size(const sdrm_handle* h) { return h ? h->grid_S : 0; }

int sdrm_last_launch_count(const sdrm_handle* h) { return h ? h->last_launches : 0; }
int sdrm_last_resident_mode(const sdrm_handle* h) { return h ? h->last.resident : 0; }
int sdrm_last_split_size(const sdrm_handle* h) { return h ? h->last.split : 0; }

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
int sdrm_last_cluster_size(const sdrm_handle* h) { return h ? h->last.cluster : 0; }

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
  fill_desc(P.dec[0], ws + w_off, g, reinterpret_cast<const float*>(ws + b_off), nullptr, 0, split3 ? 3 : 1, EPI_LINEAR_OUT, 0, 1, 0, 0);
  P.n_step = 0; P.n_dec = 1; P.T = 0; P.L = K; P.Lg16 = 0; P.preloaded_input = 1; P.n_sub = 1;
  P.n_rows = M; P.row_offset = 0;
  P.logits = d_out; P.ld_logits = N;
  P.scratch = ws + s_off; P.scratch_stride = 2 * act; P.act_buf_bytes = act;
  P.err_word = reinterpret_cast<int*>(ws);
  const int grid = static_cast<int>(std::max<long long>(1, std::min<long long>(n_tiles, sms)));
  const int rc = fill_act_maps(P, static_cast<size_t>(n_tiles) * 2 * act);
  if (rc) return rc;
  return launch_engine(P, grid, 1, st);
}

}  // extern "C"
