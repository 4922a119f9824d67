// K6 — register / shared-memory resident reverse-diffusion chain for SMALL denoisers (latent, hidden and VAE hidden width <= 64).
//
// Reference: the same sample_ddpm loop as K1 (train_SDRM.py:27-63; SDRM.forward 97-103; denoise_add_noise 20-25; VAE.decode
// 252-254), for configurations like BASELINE.json's cfg 3 (ADM: L = H = 40, T = 93, 5 hidden layers, 8 582 items, 9 558 users).
// At these widths a 128-row tcgen05 tile does ~50 k MACs per layer: K1 is bound by the ~1 us latency of every layer hand-off
// (651 of them per chain) and keeps 75 of 148 SMs busy (r01: 2.16 ms, 2 % of the HBM logits-write roofline).  Here
//   * the denoiser weights (3 matrices <= 64 x 64, bf16) and the first decoder layer live in SHARED MEMORY for the whole chain
//     (the north star's "weights resident in shared memory across all T timesteps"),
//   * a warp owns 16 rows; the fp32 diffusion state and every activation stay in REGISTERS for all T steps: a layer is
//     NT x KS warp-level mma.sync.m16n8k16 (bf16 operands, fp32 accumulate) whose accumulator fragments are re-packed in place
//     into the next layer's A fragments (no shuffle, no memory round trip),
//   * bias (hoisted time embedding), PReLU / tanh, the always-on dropout, the posterior update and the Philox Gaussian noise
//     are applied on the fragments; the noise / mask streams are the SAME counter streams as K1 (philox.cuh), so a row's
//     random numbers do not depend on which kernel produced it,
//   * the decoder runs as bf16x3 (hi.hi + hi.lo + lo.hi) like K1's; W2 streams through shared memory in 64-item slices
//     (cp.async, double buffered) and the logits go straight from the accumulators to HBM.
// 2 warps (32 rows) per CTA and <= 75 KB of shared memory, so three CTAs fit an SM and ALL CTAs of a dataset-sized launch are
// resident at once (no second wave).  Rows are independent: no inter-CTA communication.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

#include <type_traits>

#include "philox.cuh"
#include "ptx_sm100.cuh"

namespace sdrm {

struct SmallParams {
  const __nv_bfloat16 *w0, *wh, *wo;        // [64][72] zero-padded bf16 images of dnn.0.weight[:, :L], the shared hidden Linear, the output Linear
  const __nv_bfloat16 *w1_hi, *w1_lo;       // [64][72]  decoder[0].weight hi / lo
  const __nv_bfloat16 *w2_hi, *w2_lo;       // [I rounded up to 64][72]  decoder[2].weight hi / lo (zero rows beyond I)
  const float* bias0; int bias0_ld;         // [T+1][64] hoisted time-embedding bias of layer 0, zero padded
  const float *bh, *bo, *b1, *b2;           // bh, bo, b1: 64 zero-padded entries; b2: at least I entries
  const float* slopes;                      // {a0, ah}
  const float* coef;                        // [T+1][4] = c1, c2, sigma * nd, 0
  int T, L, H, I, nh;
  long long n_rows, row_offset, ld_logits;
  const int32_t *t_start, *row_ids;
  float* x0_out;
  void* logits;                             // fp32, or bfloat16 bits (BF16OUT); ld_logits in elements
  const float *inj_xT, *inj_z;
  const uint8_t* inj_mask;
  unsigned long long seed;
};

constexpr int SMALL_WARPS = 2;
constexpr int SMALL_THREADS = 32 * SMALL_WARPS;
constexpr int SMALL_W2_ITEMS = 64;          // items per W2 stage
constexpr int SMALL_KP = 72;                // row pitch (bf16) of every packed small-path weight image
constexpr int SMALL_MAX = 64;               // widest latent / hidden / VAE-hidden dimension this kernel takes

template <int NT>
struct SmallGeom {
  static constexpr int KS = (NT + 1) / 2;            // k16 steps
  static constexpr int KP = SMALL_KP;                 // bf16 per weight row: 64 + 8, the +8 keeps the B-fragment loads conflict-free
  static constexpr int W_ELEMS = 8 * NT * KP;         // the first 8 NT rows of a packed <= 64 x 64 matrix
  static constexpr int STAGE_ELEMS = SMALL_W2_ITEMS * KP;
  static constexpr int SMEM_BYTES = 2 * (5 * W_ELEMS + 4 * STAGE_ELEMS) + 2 * SMALL_W2_ITEMS * 4;   // + the b2 slices of the two stages
};

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// BF16OUT: the logits are stored as bfloat16, the round to nearest even of the fp32 value the fp32 instantiation writes
template <int NT, bool BF16OUT = false>
__global__ void __launch_bounds__(SMALL_THREADS) sdrm_small_chain_kernel(const SmallParams P) {
  using G = SmallGeom<NT>;
  constexpr int KS = G::KS, KP = G::KP;
  extern __shared__ __align__(16) uint8_t ssm_raw[];
  __nv_bfloat16* sW0 = reinterpret_cast<__nv_bfloat16*>(ssm_raw);
  __nv_bfloat16* sWh = sW0 + G::W_ELEMS;
  __nv_bfloat16* sWo = sWh + G::W_ELEMS;
  __nv_bfloat16* sW1h = sWo + G::W_ELEMS;
  __nv_bfloat16* sW1l = sW1h + G::W_ELEMS;
  __nv_bfloat16* sStage = sW1l + G::W_ELEMS;      // [2 buffers][hi, lo][SMALL_W2_ITEMS][KP]
  float* sB2 = reinterpret_cast<float*>(sStage + 4 * G::STAGE_ELEMS);   // [2 buffers][SMALL_W2_ITEMS]

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;

  // ---- weights -> shared memory, once per CTA
  {
    const __nv_bfloat16* src[5] = {P.w0, P.nh > 0 ? P.wh : P.w0, P.wo, P.w1_hi, P.w1_lo};
    constexpr int N16 = G::W_ELEMS * 2 / 16;
    for (int m = 0; m < 5; ++m) {
      const uint4* s = reinterpret_cast<const uint4*>(src[m]);
      uint4* d = reinterpret_cast<uint4*>(sW0 + m * G::W_ELEMS);
      for (int i = threadIdx.x; i < N16; i += SMALL_THREADS) d[i] = __ldg(s + i);
    }
  }
  __syncthreads();

  // ---- the 16 rows of this warp: thread (g, t) holds rows g and g + 8, columns 8 j + 2 t, 8 j + 2 t + 1 of every n-tile j
  const long long tile_row = (static_cast<long long>(blockIdx.x) * SMALL_WARPS + warp) * 16;
  long long prow[2] = {tile_row + g, tile_row + g + 8};
  bool valid[2];
  long long lrow[2];
  unsigned long long grow[2];
  int t_row[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    valid[h] = prow[h] < P.n_rows;
    lrow[h] = (valid[h] && P.row_ids) ? static_cast<long long>(P.row_ids[prow[h]]) : prow[h];
    grow[h] = static_cast<unsigned long long>(P.row_offset + lrow[h]);
    t_row[h] = !valid[h] ? 0 : (P.t_start ? min(max(P.t_start[prow[h]], 0), P.T) : P.T);
  }
  int T_w = max(t_row[0], t_row[1]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) T_w = max(T_w, __shfl_xor_sync(0xffffffffu, T_w, o));
  const PhiloxKeys K = philox_make_keys(P.seed);
  const int L = P.L;

  // N(0,1) draws of (step, n-tile j) for this thread's four state elements: even t computes the Philox call of row g, odd t the
  // one of row g + 8 (columns 8 j + 4 (t >> 1) .. + 3), and the pair swaps halves -- every call is computed exactly once
  auto normals = [&](uint32_t step, int j, float (&z)[4]) {
    float z4[4];
    philox_normal4_keys(K, STREAM_NORMAL, grow[t & 1], step, static_cast<uint32_t>(2 * j + (t >> 1)), z4);
    const float s0 = (t & 1) ? z4[0] : z4[2], s1 = (t & 1) ? z4[1] : z4[3];
    const float r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);
    if (t & 1) { z[0] = r0; z[1] = r1; z[2] = z4[2]; z[3] = z4[3]; }
    else { z[0] = z4[0]; z[1] = z4[1]; z[2] = r0; z[3] = r1; }
  };

  // ---- x_T (train_SDRM.py:51 / 38); padding columns stay exactly 0 for the whole chain
  float x[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    float z[4];
    if (P.inj_xT) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = 8 * j + 2 * t + (e & 1);
        z[e] = (valid[e >> 1] && c < L) ? P.inj_xT[static_cast<size_t>(lrow[e >> 1]) * L + c] : 0.0f;
      }
    } else {
      normals(0u, j, z);
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) x[j][e] = (8 * j + 2 * t + (e & 1) < L) ? z[e] : 0.0f;
  }

  // one dense layer on fragments: acc[j] = sum_s A[s] . W[8 j .. 8 j + 7, 16 s .. 16 s + 15]^T
  auto layer = [&](const uint32_t (&a)[KS][4], const __nv_bfloat16* sW, float (&acc)[NT][4]) {
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.0f;
      const __nv_bfloat16* wrow = sW + (8 * j + g) * KP + 2 * t;
#pragma unroll
      for (int s = 0; s < KS; ++s) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(wrow + 16 * s);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(wrow + 16 * s + 8);
        mma_bf16_16816(acc[j], a[s], b0, b1);
      }
    }
  };
  // accumulator fragments of n-tiles 2 s, 2 s + 1 -> A fragment of k-step s (same thread: no data movement)
  auto to_frags = [&](const float (&v)[NT][4], uint32_t (&a)[KS][4]) {
#pragma unroll
    for (int s = 0; s < KS; ++s) {
      a[s][0] = pack_bf16x2(v[2 * s][0], v[2 * s][1]);
      a[s][1] = pack_bf16x2(v[2 * s][2], v[2 * s][3]);
      if (2 * s + 1 < NT) {
        a[s][2] = pack_bf16x2(v[2 * s + 1][0], v[2 * s + 1][1]);
        a[s][3] = pack_bf16x2(v[2 * s + 1][2], v[2 * s + 1][3]);
      } else {
        a[s][2] = a[s][3] = 0u;
      }
    }
  };

  const float slope0 = __ldg(P.slopes), slopeh = P.nh > 0 ? __ldg(P.slopes + 1) : 0.0f;
  // Step-independent biases live in registers; the step's time-embedding bias row and coefficients are fetched one step ahead
  // (a single warp per scheduler cannot hide a global-load latency per layer: 35 of them per step were 1/3 of the stalls)
  float2 bh2[NT], bo2[NT], b0cur[NT];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    bh2[j] = __ldg(reinterpret_cast<const float2*>(P.bh + 8 * j + 2 * t));
    bo2[j] = __ldg(reinterpret_cast<const float2*>(P.bo + 8 * j + 2 * t));
    b0cur[j] = __ldg(reinterpret_cast<const float2*>(P.bias0 + static_cast<size_t>(T_w) * P.bias0_ld + 8 * j + 2 * t));
  }
  float4 cf = __ldg(reinterpret_cast<const float4*>(P.coef) + T_w);

  // ---- the reverse chain
  for (int i = T_w; i >= 1; --i) {
    float2 b0next[NT];
    const int inext = max(i - 1, 0);
#pragma unroll
    for (int j = 0; j < NT; ++j) b0next[j] = __ldg(reinterpret_cast<const float2*>(P.bias0 + static_cast<size_t>(inext) * P.bias0_ld + 8 * j + 2 * t));
    const float4 cf_next = __ldg(reinterpret_cast<const float4*>(P.coef) + inext);
    // dropout keep bits of this forward (F.dropout p = .5, always on, train_SDRM.py:100): one Philox call per row and step,
    // computed by threads t = 0 (row g) and t = 1 (row g + 8) of the quad
    uint32_t keep[2][2];   // [row half][columns 0..31, 32..63]
    if (!P.inj_mask) {
      const u32x4 m = philox_mask128(K, STREAM_MASK, grow[t & 1], static_cast<uint32_t>(i), 0u);
      const int q0 = lane & ~3;
      keep[0][0] = __shfl_sync(0xffffffffu, m.x, q0);     keep[0][1] = __shfl_sync(0xffffffffu, m.y, q0);
      keep[1][0] = __shfl_sync(0xffffffffu, m.x, q0 | 1); keep[1][1] = __shfl_sync(0xffffffffu, m.y, q0 | 1);
    }
    float v[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = 8 * j + 2 * t + (e & 1), h = e >> 1;
        bool kp;
        if (P.inj_mask) kp = valid[h] && c < L && P.inj_mask[(static_cast<size_t>(i) * P.n_rows + lrow[h]) * L + c] != 0;
        else kp = (keep[h][c >> 5] >> (c & 31)) & 1u;
        v[j][e] = kp ? 2.0f * x[j][e] : 0.0f;
      }
    }
    uint32_t a[KS][4];
    to_frags(v, a);
    float acc[NT][4];
    // layer 0: K = L product + the hoisted time-embedding bias row of step i, PReLU
    layer(a, sW0, acc);
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const float2 bb = b0cur[j];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float hh = acc[j][e] + ((e & 1) ? bb.y : bb.x);
        v[j][e] = hh > 0.0f ? hh : slope0 * hh;
      }
    }
    for (int hl = 0; hl < P.nh; ++hl) {   // the ONE shared hidden Linear + PReLU, nh times (train_SDRM.py:94)
      to_frags(v, a);
      layer(a, sWh, acc);
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        const float2 bb = bh2[j];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float hh = acc[j][e] + ((e & 1) ? bb.y : bb.x);
          v[j][e] = hh > 0.0f ? hh : slopeh * hh;
        }
      }
    }
    to_frags(v, a);
    layer(a, sWo, acc);
    // posterior update (denoise_add_noise, train_SDRM.py:20-25): x <- (x c2 + sigma nd z) - c1 c2 tanh(.)  (K1's operation order)
    const float c12 = cf.x * cf.y;
    const bool act[2] = {valid[0] && i <= t_row[0], valid[1] && i <= t_row[1]};
    // all N(0,1) draws of the step in one unrolled block: NT independent Philox chains the scheduler can interleave
    float z[NT][4];
    if (cf.z != 0.0f && !P.inj_z) {
#pragma unroll
      for (int j = 0; j < NT; ++j) normals(static_cast<uint32_t>(i), j, z[j]);
    } else {
#pragma unroll
      for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int c = 8 * j + 2 * t + (e & 1);
          z[j][e] = (cf.z != 0.0f && valid[e >> 1] && c < L) ? P.inj_z[(static_cast<size_t>(i) * P.n_rows + lrow[e >> 1]) * L + c] : 0.0f;
        }
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const float2 bb = bo2[j];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = 8 * j + 2 * t + (e & 1);
        const float eps = mufu_tanh(acc[j][e] + ((e & 1) ? bb.y : bb.x));
        const float st = fmaf(cf.z, z[j][e], x[j][e] * cf.y);
        const float xn = fmaf(-c12, eps, st);
        if (act[e >> 1] && c < L) x[j][e] = xn;
      }
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) b0cur[j] = b0next[j];
    cf = cf_next;
  }

  // ---- x_0 -> optional latent output
  if (P.x0_out) {
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = 8 * j + 2 * t + (e & 1);
        if (valid[e >> 1] && c < L) P.x0_out[static_cast<size_t>(lrow[e >> 1]) * L + c] = x[j][e];
      }
  }

  // ---- decoder (VAE.decode, train_SDRM.py:252-254) as bf16x3 on fragments
  auto split_frags = [&](const float (&v)[NT][4], uint32_t (&ah)[KS][4], uint32_t (&al)[KS][4]) {
    float hi[NT][4], lo[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        hi[j][e] = bf16_round(v[j][e]);
        lo[j][e] = v[j][e] - hi[j][e];
      }
    to_frags(hi, ah);
    to_frags(lo, al);
  };
  uint32_t ah[KS][4], al[KS][4];
  split_frags(x, ah, al);
  float hdec[NT][4];
  {
    float a1[NT][4], a2[NT][4], a3[NT][4];
    layer(ah, sW1h, a1);
    layer(ah, sW1l, a2);
    layer(al, sW1h, a3);
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const float2 bb = __ldg(reinterpret_cast<const float2*>(P.b1 + 8 * j + 2 * t));
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = 8 * j + 2 * t + (e & 1);
        const float hh = fast_tanh((a1[j][e] + a2[j][e] + a3[j][e]) + ((e & 1) ? bb.y : bb.x));
        hdec[j][e] = c < P.H ? hh : 0.0f;
      }
    }
  }
  split_frags(hdec, ah, al);

  // W2 streams through shared memory: 64 items (rows of decoder[2].weight) per stage, hi and lo images, double buffered
  const int n_stage = (P.I + SMALL_W2_ITEMS - 1) / SMALL_W2_ITEMS;
  auto stage_ptr = [&](int buf, int which) { return sStage + (buf * 2 + which) * G::STAGE_ELEMS; };
  auto fetch = [&](int st, int buf) {
    constexpr int N16 = G::STAGE_ELEMS * 2 / 16;
    const uint4* sh = reinterpret_cast<const uint4*>(P.w2_hi + static_cast<size_t>(st) * G::STAGE_ELEMS);
    const uint4* sl = reinterpret_cast<const uint4*>(P.w2_lo + static_cast<size_t>(st) * G::STAGE_ELEMS);
    const uint32_t dh = smem_u32(stage_ptr(buf, 0)), dl = smem_u32(stage_ptr(buf, 1));
    for (int i = threadIdx.x; i < N16; i += SMALL_THREADS) {
      cp_async16(dh + 16u * i, sh + i);
      cp_async16(dl + 16u * i, sl + i);
    }
    if (threadIdx.x < SMALL_W2_ITEMS / 4)   // the stage's 64 output biases (b2 is padded to a multiple of 64 entries)
      cp_async16(smem_u32(sB2 + buf * SMALL_W2_ITEMS) + 16u * threadIdx.x, P.b2 + static_cast<size_t>(st) * SMALL_W2_ITEMS + 4 * threadIdx.x);
    cp_async_commit();
  };
  fetch(0, 0);
  using OutT = std::conditional_t<BF16OUT, uint16_t, float>;
  const bool pair_ok = ((P.ld_logits & 1) == 0) && ((reinterpret_cast<uintptr_t>(P.logits) & (2 * sizeof(OutT) - 1)) == 0);
  OutT* orow[2] = {static_cast<OutT*>(P.logits) + static_cast<size_t>(lrow[0]) * P.ld_logits,
                   static_cast<OutT*>(P.logits) + static_cast<size_t>(lrow[1]) * P.ld_logits};
  for (int st = 0; st < n_stage; ++st) {
    const int buf = st & 1;
    if (st + 1 < n_stage) { fetch(st + 1, buf ^ 1); cp_async_wait<1>(); }
    else cp_async_wait<0>();
    __syncthreads();
    const __nv_bfloat16* wh_ = stage_ptr(buf, 0);
    const __nv_bfloat16* wl_ = stage_ptr(buf, 1);
    const float* b2s = sB2 + buf * SMALL_W2_ITEMS;
#pragma unroll 2
    for (int jj = 0; jj < SMALL_W2_ITEMS / 8; ++jj) {
      // three independent accumulation chains (hi.hi, hi.lo, lo.hi) instead of one chain of 3 KS dependent MMAs
      float a_hh[4] = {0.f, 0.f, 0.f, 0.f}, a_hl[4] = {0.f, 0.f, 0.f, 0.f}, a_lh[4] = {0.f, 0.f, 0.f, 0.f};
      const __nv_bfloat16* rh = wh_ + (8 * jj + g) * KP + 2 * t;
      const __nv_bfloat16* rl = wl_ + (8 * jj + g) * KP + 2 * t;
#pragma unroll
      for (int s = 0; s < KS; ++s) {
        const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(rh + 16 * s), bh1 = *reinterpret_cast<const uint32_t*>(rh + 16 * s + 8);
        const uint32_t bl0 = *reinterpret_cast<const uint32_t*>(rl + 16 * s), bl1 = *reinterpret_cast<const uint32_t*>(rl + 16 * s + 8);
        mma_bf16_16816(a_hh, ah[s], bh0, bh1);
        mma_bf16_16816(a_hl, ah[s], bl0, bl1);
        mma_bf16_16816(a_lh, al[s], bh0, bh1);
      }
      const int c = st * SMALL_W2_ITEMS + 8 * jj + 2 * t;
      const float2 bb = *reinterpret_cast<const float2*>(b2s + 8 * jj + 2 * t);
      if (c < P.I) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (!valid[h]) continue;
          const float o0 = (a_hh[2 * h] + (a_hl[2 * h] + a_lh[2 * h])) + bb.x, o1 = (a_hh[2 * h + 1] + (a_hl[2 * h + 1] + a_lh[2 * h + 1])) + bb.y;
          if constexpr (BF16OUT) {
            const uint32_t pk = pack_bf16x2(o0, o1);
            if (pair_ok && c + 1 < P.I) __stcs(reinterpret_cast<unsigned int*>(orow[h] + c), pk);
            else {
              orow[h][c] = static_cast<uint16_t>(pk);
              if (c + 1 < P.I) orow[h][c + 1] = static_cast<uint16_t>(pk >> 16);
            }
          } else if (pair_ok && c + 1 < P.I) __stcs(reinterpret_cast<float2*>(orow[h] + c), make_float2(o0, o1));
          else {
            orow[h][c] = o0;
            if (c + 1 < P.I) orow[h][c + 1] = o1;
          }
        }
      }
    }
    __syncthreads();   // every warp is done with this buffer before the fetch after next overwrites it
  }
}

}  // namespace sdrm
