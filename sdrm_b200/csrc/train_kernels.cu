// K2 — fused elementwise kernels of the diffusion training step (reference: train_SDRM.py:321-337,
// perturb_input 202-203, score_matching_loss 191-199).  All three are HBM-bound streaming kernels:
// vectorised (float4) coalesced reads, one pass, fp64 block reductions for the loss statistics.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/sdrm_b200.h"
#include "host_util.h"
#include "philox.cuh"

namespace sdrm {

// The [B, L] latent batch is walked as ONE flat array (row stride == L), so every access is a 16-byte vector whatever L is
// (L = 950 rows are only 8-byte aligned).  A warp owns 512 consecutive elements per iteration: lane l handles the four
// quads j*32 + l (j = 0..3) -> each of its float4 loads / stores is a fully coalesced 512-byte warp access.  Per thread and
// iteration: four Gaussian Philox calls (4 normals each) and ONE call for the 3 x 16 dropout bits.
//   noise   = N(0,1) * nd                                  (train_SDRM.py:326)
//   x_t     = sqrt(ab[t]) * mu + (1 - ab[t]) * noise       (train_SDRM.py:203 -- NOT sqrt on the noise term)
//   x_p     = mu + mu_coef * noise                          (train_SDRM.py:194)
//   in_k    = input_k * keep_k * 2                          (F.dropout p=.5 always on, train_SDRM.py:100)
// Streams, keyed by the GLOBAL flat element index i = (row_offset + b) * L + f (identical for any row sharding):
//   normals: Philox(c0|c1 = i / 4, c2 = 0, c3 = STREAM_TRAIN_NOISE) -> Box-Muller pairs -> elements 4 (i/4) .. + 3
//   masks  : element i = 512 blk + 4 (32 j + l) + e;  Philox(c0|c1 = 32 blk + l, c2 = 0, c3 = STREAM_TRAIN_MASK),
//            keep bit of the k-th denoiser input = bit (4 j + e) of output word k            (oracle/philox_ref.py)
__global__ void __launch_bounds__(256) noise_inputs_kernel(
    const float* __restrict__ mu, const long long* __restrict__ t, const float* __restrict__ ab, long long B, int L,
    float nd, float mu_coef, unsigned long long seed, long long row_offset, const float* __restrict__ inj_noise,
    const uint8_t* __restrict__ inj_masks, float* __restrict__ noise_out, float* __restrict__ in_pert,
    float* __restrict__ in_clean, float* __restrict__ in_shift, uint8_t* __restrict__ masks_out) {
  const long long total = B * L;                       // local elements
  const unsigned long long g0 = static_cast<unsigned long long>(row_offset) * static_cast<unsigned long long>(L);  // global index of local 0
  // local element 0 may sit anywhere inside a global 512-block / quad: iterate over GLOBAL blocks covering the local range
  const unsigned long long first_blk = g0 >> 9, last_blk = (g0 + static_cast<unsigned long long>(total) + 511) >> 9;
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long n_warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const PhiloxKeys K = philox_make_keys(seed);
  const bool aligned = ((g0 & 3) == 0) && ((reinterpret_cast<uintptr_t>(mu) & 15) == 0) &&
                       ((reinterpret_cast<uintptr_t>(in_pert) & 15) == 0) && ((reinterpret_cast<uintptr_t>(in_clean) & 15) == 0) &&
                       ((reinterpret_cast<uintptr_t>(in_shift) & 15) == 0) && (!noise_out || (reinterpret_cast<uintptr_t>(noise_out) & 15) == 0);
  const bool fast_ok = aligned && !inj_masks && !inj_noise && !masks_out && L >= 4 && total <= 0x7fffffffLL;
  for (unsigned long long blk = first_blk + warp; blk < last_blk; blk += n_warps) {
    // Interior blocks (all 512 elements inside the local range, 16-byte aligned, in-kernel streams): the same arithmetic as the
    // general path below without its per-element range / alignment / injection branches (2/3 of its issued instructions)
    if (fast_ok && blk * 512ull >= g0 && blk * 512ull + 512ull <= g0 + static_cast<unsigned long long>(total)) {
      const unsigned long long mc = blk * 32ull + lane;
      const u32x4 m4 = philox4x32_10_keys(static_cast<uint32_t>(mc), static_cast<uint32_t>(mc >> 32), 0u, STREAM_TRAIN_MASK, K);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned long long gq = blk * 128ull + static_cast<unsigned long long>(j * 32 + lane);
        const uint32_t i0 = static_cast<uint32_t>(gq * 4ull - g0);
        const float4 v = *reinterpret_cast<const float4*>(mu + i0);
        const u32x4 r4 = philox4x32_10_keys(static_cast<uint32_t>(gq), static_cast<uint32_t>(gq >> 32), 0u, STREAM_TRAIN_NOISE, K);
        float nz[4];
        box_muller_fast(r4.x, r4.y, nz[0], nz[1]);
        box_muller_fast(r4.z, r4.w, nz[2], nz[3]);
        const uint32_t b0 = i0 / static_cast<uint32_t>(L);
        const int f_first = static_cast<int>(i0 - b0 * static_cast<uint32_t>(L));
        const float abt0 = __ldg(ab + __ldg(t + b0));
        float sa0 = sqrtf(abt0), om0 = 1.0f - abt0, sa1 = sa0, om1 = om0;
        if (f_first + 3 >= L && static_cast<long long>(b0) + 1 < B) {
          const float abt1 = __ldg(ab + __ldg(t + b0 + 1));
          sa1 = sqrtf(abt1); om1 = 1.0f - abt1;
        }
        const float m[4] = {v.x, v.y, v.z, v.w};
        float xp[4], xc[4], xs[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          nz[e] *= nd;
          const bool second = f_first + e >= L;
          const float sa = second ? sa1 : sa0, om = second ? om1 : om0;
          const int bit = 4 * j + e;
          const float xt = sa * m[e] + om * nz[e];
          const float xq = m[e] + mu_coef * nz[e];
          xp[e] = ((m4.x >> bit) & 1u) ? 2.0f * xt : 0.0f;
          xc[e] = ((m4.y >> bit) & 1u) ? 2.0f * m[e] : 0.0f;
          xs[e] = ((m4.z >> bit) & 1u) ? 2.0f * xq : 0.0f;
        }
        if (noise_out) __stcs(reinterpret_cast<float4*>(noise_out + i0), make_float4(nz[0], nz[1], nz[2], nz[3]));
        __stcs(reinterpret_cast<float4*>(in_pert + i0), make_float4(xp[0], xp[1], xp[2], xp[3]));
        __stcs(reinterpret_cast<float4*>(in_clean + i0), make_float4(xc[0], xc[1], xc[2], xc[3]));
        __stcs(reinterpret_cast<float4*>(in_shift + i0), make_float4(xs[0], xs[1], xs[2], xs[3]));
      }
      continue;
    }
    uint32_t keep[3] = {0u, 0u, 0u};
    if (!inj_masks) {
      const unsigned long long mc = blk * 32ull + lane;
      const u32x4 m4 = philox4x32_10_keys(static_cast<uint32_t>(mc), static_cast<uint32_t>(mc >> 32), 0u, STREAM_TRAIN_MASK, K);
      keep[0] = m4.x; keep[1] = m4.y; keep[2] = m4.z;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const unsigned long long gq = blk * 128ull + static_cast<unsigned long long>(j * 32 + lane);   // global quad index
      const long long i0 = static_cast<long long>(gq * 4ull - g0);                                    // local index of the quad
      if (i0 + 3 < 0 || i0 >= total) continue;
      const bool full = aligned && i0 >= 0 && i0 + 3 < total;
      float m[4] = {0.f, 0.f, 0.f, 0.f}, nz[4] = {0.f, 0.f, 0.f, 0.f};
      bool ok[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) ok[e] = (i0 + e >= 0) && (i0 + e < total);
      if (full) {
        const float4 v = *reinterpret_cast<const float4*>(mu + i0);
        m[0] = v.x; m[1] = v.y; m[2] = v.z; m[3] = v.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) if (ok[e]) m[e] = mu[i0 + e];
      }
      if (inj_noise) {
#pragma unroll
        for (int e = 0; e < 4; ++e) if (ok[e]) nz[e] = inj_noise[i0 + e];
      } else {
        const u32x4 r4 = philox4x32_10_keys(static_cast<uint32_t>(gq), static_cast<uint32_t>(gq >> 32), 0u, STREAM_TRAIN_NOISE, K);
        box_muller_fast(r4.x, r4.y, nz[0], nz[1]);
        box_muller_fast(r4.z, r4.w, nz[2], nz[3]);
#pragma unroll
        for (int e = 0; e < 4; ++e) nz[e] *= nd;
      }
      // rows of the four elements (a quad straddles two rows when L % 4 != 0)
      const long long ic = i0 < 0 ? 0 : i0;
      long long b0;
      int f_first;
      if (total <= 0x7fffffffLL) {   // 32-bit division: the 64-bit one costs more than the quad's Philox call
        const uint32_t q32 = static_cast<uint32_t>(ic) / static_cast<uint32_t>(L);
        b0 = q32;
        f_first = static_cast<int>(static_cast<uint32_t>(ic) - q32 * static_cast<uint32_t>(L));
      } else {
        b0 = ic / L;
        f_first = static_cast<int>(ic - b0 * L);
      }
      // schedule coefficients of the (at most two, for L >= 4) rows the quad touches: looked up once per row, not per element
      float sa0, om0, sa1, om1;
      {
        const float abt0 = __ldg(ab + __ldg(t + b0));
        sa0 = sqrtf(abt0); om0 = 1.0f - abt0;
        sa1 = sa0; om1 = om0;
        if (L >= 4 && f_first + 3 >= L && b0 + 1 < B) {
          const float abt1 = __ldg(ab + __ldg(t + b0 + 1));
          sa1 = sqrtf(abt1); om1 = 1.0f - abt1;
        }
      }
      float xp[4], xc[4], xs[4];
      uint32_t kb[3] = {0u, 0u, 0u};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (!ok[e]) { xp[e] = xc[e] = xs[e] = 0.f; continue; }
        const long long ie = i0 + e;
        float sa, om;
        if (L >= 4) {
          const bool second = (f_first + static_cast<int>(ie - ic)) >= L;
          sa = second ? sa1 : sa0; om = second ? om1 : om0;
        } else {
          const float abt = __ldg(ab + __ldg(t + ie / L));
          sa = sqrtf(abt); om = 1.0f - abt;
        }
        const int bit = 4 * j + e;
        if (inj_masks) {
#pragma unroll
          for (int k = 0; k < 3; ++k) kb[k] |= (inj_masks[static_cast<size_t>(k) * total + ie] ? 1u : 0u) << e;
        } else {
#pragma unroll
          for (int k = 0; k < 3; ++k) kb[k] |= ((keep[k] >> bit) & 1u) << e;
        }
        const float xt = sa * m[e] + om * nz[e];
        const float xq = m[e] + mu_coef * nz[e];
        xp[e] = ((kb[0] >> e) & 1u) ? 2.0f * xt : 0.0f;
        xc[e] = ((kb[1] >> e) & 1u) ? 2.0f * m[e] : 0.0f;
        xs[e] = ((kb[2] >> e) & 1u) ? 2.0f * xq : 0.0f;
      }
      if (full) {
        if (noise_out) __stcs(reinterpret_cast<float4*>(noise_out + i0), make_float4(nz[0], nz[1], nz[2], nz[3]));
        __stcs(reinterpret_cast<float4*>(in_pert + i0), make_float4(xp[0], xp[1], xp[2], xp[3]));
        __stcs(reinterpret_cast<float4*>(in_clean + i0), make_float4(xc[0], xc[1], xc[2], xc[3]));
        __stcs(reinterpret_cast<float4*>(in_shift + i0), make_float4(xs[0], xs[1], xs[2], xs[3]));
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (!ok[e]) continue;
          if (noise_out) noise_out[i0 + e] = nz[e];
          in_pert[i0 + e] = xp[e];
          in_clean[i0 + e] = xc[e];
          in_shift[i0 + e] = xs[e];
        }
      }
      if (masks_out) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (ok[e])
            for (int k = 0; k < 3; ++k) masks_out[static_cast<size_t>(k) * total + i0 + e] = static_cast<uint8_t>((kb[k] >> e) & 1u);
      }
    }
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// stats += {sum r, sum r^2, sum (sd-r)^2, sum (r-sx)^2, count};  r = pred - mu, sd = (psx - sx)/mu_coef^2
// The four terms of a quad are summed in fp32 and promoted to fp64 once per quad: B200 runs FP64 at a fraction of the fp32
// rate, and one DADD per element and statistic made this kernel ALU-bound.  Quads are read as float4 when all four arrays are
// 16-byte aligned and as four scalars otherwise (ScoreMatchingLoss passes sx and psx as row slices of one [3B, L] buffer, so
// B*L % 4 != 0 misaligns them): both give the same fp32 partials, in the same threads.
// r is accumulated about a shift K = r[0] and turned back into sum r and sum r^2 in fp64 once per thread: the fp32 partials
// then hold (r - K)^2 ~ var(r) instead of r^2, so the variance (sum r^2 - N mean^2) / (N - 1) that loss_seeds_kernel forms
// keeps its precision when the mean of r is large next to its spread (mean 3, std 0.05: 3600 x N var in sum r^2).
__global__ void __launch_bounds__(256) loss_stats_kernel(const float* __restrict__ pred, const float* __restrict__ sx,
                                                         const float* __restrict__ psx, const float* __restrict__ mu,
                                                         long long count, float mu2, double* __restrict__ stats) {
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  long long n = 0;                                     // elements this thread summed
  const long long tid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long nth = static_cast<long long>(gridDim.x) * blockDim.x;
  const bool vec = (((reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(sx) | reinterpret_cast<uintptr_t>(psx) |
                      reinterpret_cast<uintptr_t>(mu)) & 15) == 0);
  const long long n4 = count >> 2;
  const float K = __ldg(pred) - __ldg(mu);
  auto term = [&](float p, float s, float q, float m, float& a0, float& a1, float& a2, float& a3) {
    const float r = p - m, rk = r - K;
    const float sd = (q - s) / mu2;
    const float d1 = sd - r, d2 = r - s;
    a0 += rk; a1 = fmaf(rk, rk, a1); a2 = fmaf(d1, d1, a2); a3 = fmaf(d2, d2, a3);
  };
  for (long long i = tid; i < n4; i += nth) {
    float4 p, s, q, m;
    if (vec) {
      p = __ldcs(reinterpret_cast<const float4*>(pred) + i); s = __ldcs(reinterpret_cast<const float4*>(sx) + i);
      q = __ldcs(reinterpret_cast<const float4*>(psx) + i); m = __ldcs(reinterpret_cast<const float4*>(mu) + i);
    } else {
      const long long e = i << 2;
      p = make_float4(pred[e], pred[e + 1], pred[e + 2], pred[e + 3]); s = make_float4(sx[e], sx[e + 1], sx[e + 2], sx[e + 3]);
      q = make_float4(psx[e], psx[e + 1], psx[e + 2], psx[e + 3]); m = make_float4(mu[e], mu[e + 1], mu[e + 2], mu[e + 3]);
    }
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    term(p.x, s.x, q.x, m.x, a0, a1, a2, a3); term(p.y, s.y, q.y, m.y, a0, a1, a2, a3);
    term(p.z, s.z, q.z, m.z, a0, a1, a2, a3); term(p.w, s.w, q.w, m.w, a0, a1, a2, a3);
    s0 += a0; s1 += a1; s2 += a2; s3 += a3;
    n += 4;
  }
  for (long long i = (n4 << 2) + tid; i < count; i += nth) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    term(pred[i], sx[i], psx[i], mu[i], a0, a1, a2, a3);
    s0 += a0; s1 += a1; s2 += a2; s3 += a3;
    ++n;
  }
  {  // sums about K -> sums of r and r^2
    const double k = K, nd = static_cast<double>(n);
    s1 += k * (2.0 * s0 + nd * k);
    s0 += nd * k;
  }
  __shared__ double sh[4][8];
  s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2); s3 = warp_sum(s3);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sh[0][w] = s0; sh[1][w] = s1; sh[2][w] = s2; sh[3][w] = s3; }
  __syncthreads();
  if (threadIdx.x < 4) {
    double a = 0;
    for (int i = 0; i < 8; ++i) a += sh[threadIdx.x][i];
    atomicAdd(stats + threadIdx.x, a);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(stats + 4, static_cast<double>(count));
}

// Analytic seeds of d loss / d {pred, sx, psx} (SURVEY.md §8a9) from the GLOBAL statistics.
__global__ void __launch_bounds__(256) loss_seeds_kernel(const float* __restrict__ pred, const float* __restrict__ sx,
                                                         const float* __restrict__ psx, const float* __restrict__ mu,
                                                         long long count, float mu2, const double* __restrict__ stats,
                                                         float* __restrict__ g_pred, float* __restrict__ g_sx,
                                                         float* __restrict__ g_psx, float* __restrict__ loss_out) {
  const double N = stats[4];
  const double mean_r = stats[0] / N;
  const double V = (stats[1] - N * mean_r * mean_r) / (N - 1.0);
  const double A = stats[2] / N, Bm = stats[3] / N;
  const double den = 1e-8 + V;
  const double c = 0.5 / den;
  const double kvar = -0.5 * (A + Bm) / (den * den) * 2.0 / (N - 1.0);
  const float two_c_over_N = static_cast<float>(2.0 * c / N);
  const float kv = static_cast<float>(kvar), mr = static_cast<float>(mean_r);
  if (blockIdx.x == 0 && threadIdx.x == 0 && loss_out) loss_out[0] = static_cast<float>(0.5 * (A + Bm) / den);
  auto seed = [&](float p, float s, float q, float m, float& gp, float& gs, float& gq) {
    const float r = p - m;
    const float sd = (q - s) / mu2;
    const float d1 = sd - r, d2 = r - s;
    const float gsd = two_c_over_N * d1;
    gq = gsd / mu2;
    gs = -two_c_over_N * d2 - gsd / mu2;
    gp = two_c_over_N * (d2 - d1) + kv * (r - mr);
  };
  const long long tid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long nth = static_cast<long long>(gridDim.x) * blockDim.x;
  const bool vec = g_pred && g_sx && g_psx &&
                   (((reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(sx) | reinterpret_cast<uintptr_t>(psx) |
                      reinterpret_cast<uintptr_t>(mu) | reinterpret_cast<uintptr_t>(g_pred) | reinterpret_cast<uintptr_t>(g_sx) |
                      reinterpret_cast<uintptr_t>(g_psx)) & 15) == 0);
  const long long n4 = vec ? (count >> 2) : 0;
  for (long long i = tid; i < n4; i += nth) {
    const float4 p = __ldcs(reinterpret_cast<const float4*>(pred) + i), s = __ldcs(reinterpret_cast<const float4*>(sx) + i);
    const float4 q = __ldcs(reinterpret_cast<const float4*>(psx) + i), m = __ldcs(reinterpret_cast<const float4*>(mu) + i);
    float4 gp, gs, gq;
    seed(p.x, s.x, q.x, m.x, gp.x, gs.x, gq.x); seed(p.y, s.y, q.y, m.y, gp.y, gs.y, gq.y);
    seed(p.z, s.z, q.z, m.z, gp.z, gs.z, gq.z); seed(p.w, s.w, q.w, m.w, gp.w, gs.w, gq.w);
    __stcs(reinterpret_cast<float4*>(g_pred) + i, gp);
    __stcs(reinterpret_cast<float4*>(g_sx) + i, gs);
    __stcs(reinterpret_cast<float4*>(g_psx) + i, gq);
  }
  for (long long i = (n4 << 2) + tid; i < count; i += nth) {
    float gp, gs, gq;
    seed(pred[i], sx[i], psx[i], mu[i], gp, gs, gq);
    if (g_psx) g_psx[i] = gq;
    if (g_sx) g_sx[i] = gs;
    if (g_pred) g_pred[i] = gp;
  }
}


// ------------------------------------------------------------------------------------------------
// First encoder layer of the frozen VAE on CSR rows (SURVEY.md §8f-4; reference: VAE.encode in eval,
// train_SDRM.py:241-250, fed by `x.to_dense()` at train_SDRM.py:323):
//   hidden[r] = tanh( W_e1 (x_r / max(||x_r||_2, 1e-12)) + b_e1 )
// For a sparse interaction row this is a gather-sum of nnz(r) rows of W_e1^T (an embedding bag); the dense [B, I]
// batch of the reference (29 MB per step at adm, 80 GB for the scale-up shape) is never materialised.
// One CTA per row; thread t owns hidden columns t, t + 256, ...; every gathered weight row is read coalesced.
// ------------------------------------------------------------------------------------------------
constexpr int ENC_THREADS = 256;
constexpr int ENC_MAX_PER_THREAD = 8;   // H <= 2048
__global__ void __launch_bounds__(ENC_THREADS) encode_csr_kernel(const long long* __restrict__ indptr, const long long* __restrict__ indices,
                                                                 const float* __restrict__ values, int n_items,
                                                                 const float* __restrict__ W1T, const float* __restrict__ b1, int H,
                                                                 float* __restrict__ hidden) {
  const long long r = blockIdx.x;
  const long long lo = indptr[r], hi = indptr[r + 1];
  float acc[ENC_MAX_PER_THREAD];
#pragma unroll
  for (int u = 0; u < ENC_MAX_PER_THREAD; ++u) acc[u] = 0.0f;
  float ss = 0.0f;
  for (long long p = lo; p < hi; ++p) {
    const long long j = __ldg(indices + p);
    const float v = __ldg(values + p);
    ss = fmaf(v, v, ss);
    if (j < 0 || j >= n_items) continue;   // malformed index: ignored rather than read out of bounds
    const float* w = W1T + j * H;
#pragma unroll
    for (int u = 0; u < ENC_MAX_PER_THREAD; ++u) {
      const int h = threadIdx.x + u * ENC_THREADS;
      if (h < H) acc[u] = fmaf(v, __ldg(w + h), acc[u]);
    }
  }
  const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);   // F.normalize(x, p=2, dim=1)
#pragma unroll
  for (int u = 0; u < ENC_MAX_PER_THREAD; ++u) {
    const int h = threadIdx.x + u * ENC_THREADS;
    if (h < H) hidden[r * H + h] = tanhf(fmaf(acc[u], inv, b1[h]));
  }
}


// ------------------------------------------------------------------------------------------------
// Multinomial negative log-likelihood of the MultiVAE++ training step (SURVEY.md §8f-3; reference
// train_SDRM.py:143: neg_ll = -mean_r( sum_j log_softmax(output)[r, j] * X[r, j] )).
// Forward: ONE pass over the logits and the interaction rows (8 bytes per entry) with an online softmax gives, per row,
//   lse = log sum_j exp(o_j),  sx = sum_j X_j,  dot = sum_j X_j o_j      (loss_r = -(dot - sx * lse))
// Backward: one pass writes d loss / d o_j = scale * (softmax_j * sx - X_j)  (12 bytes per entry), scale = grad / rows.
// One CTA per row, float4 loads when the rows are 16-byte aligned.
// ------------------------------------------------------------------------------------------------
constexpr int NLL_THREADS = 256;

__device__ __forceinline__ void online_add(float& m, float& s, float v) {
  if (v > m) { s = s * __expf(m - v) + 1.0f; m = v; }
  else s += __expf(v - m);
}
__device__ __forceinline__ void online_merge(float& m, float& s, float m2, float s2) {
  const float mm = fmaxf(m, m2);
  s = (m == -INFINITY ? 0.0f : s * __expf(m - mm)) + (m2 == -INFINITY ? 0.0f : s2 * __expf(m2 - mm));
  m = mm;
}

__global__ void __launch_bounds__(NLL_THREADS) nll_fwd_kernel(const float* __restrict__ logits, const float* __restrict__ X, int n_items,
                                                              long long ld_o, long long ld_x, float* __restrict__ row_lse,
                                                              float* __restrict__ row_sx, float* __restrict__ row_dot) {
  const long long r = blockIdx.x;
  const float* o = logits + r * ld_o;
  const float* x = X + r * ld_x;
  float m = -INFINITY, s = 0.0f, sx = 0.0f, dot = 0.0f;
  const bool vec = ((ld_o & 3) == 0) && ((ld_x & 3) == 0) && ((reinterpret_cast<uintptr_t>(logits) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
  int j0 = 0;
  if (vec) {
    const int n4 = n_items >> 2;
    for (int j = threadIdx.x; j < n4; j += NLL_THREADS) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(o) + j);
      const float4 b = __ldg(reinterpret_cast<const float4*>(x) + j);
      online_add(m, s, a.x); online_add(m, s, a.y); online_add(m, s, a.z); online_add(m, s, a.w);
      sx += (b.x + b.y) + (b.z + b.w);
      dot = fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, fmaf(a.w, b.w, dot))));
    }
    j0 = n4 << 2;
  }
  for (int j = j0 + threadIdx.x; j < n_items; j += NLL_THREADS) {
    const float a = __ldg(o + j), b = __ldg(x + j);
    online_add(m, s, a);
    sx += b;
    dot = fmaf(a, b, dot);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    online_merge(m, s, __shfl_xor_sync(0xffffffffu, m, off), __shfl_xor_sync(0xffffffffu, s, off));
    sx += __shfl_xor_sync(0xffffffffu, sx, off);
    dot += __shfl_xor_sync(0xffffffffu, dot, off);
  }
  __shared__ float sh[4][NLL_THREADS / 32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = m; sh[1][w] = s; sh[2][w] = sx; sh[3][w] = dot; }
  __syncthreads();
  if (w == 0) {
    m = l < NLL_THREADS / 32 ? sh[0][l] : -INFINITY;
    s = l < NLL_THREADS / 32 ? sh[1][l] : 0.0f;
    sx = l < NLL_THREADS / 32 ? sh[2][l] : 0.0f;
    dot = l < NLL_THREADS / 32 ? sh[3][l] : 0.0f;
#pragma unroll
    for (int off = 4; off > 0; off >>= 1) {
      online_merge(m, s, __shfl_xor_sync(0xffffffffu, m, off), __shfl_xor_sync(0xffffffffu, s, off));
      sx += __shfl_xor_sync(0xffffffffu, sx, off);
      dot += __shfl_xor_sync(0xffffffffu, dot, off);
    }
    if (l == 0) { row_lse[r] = m + logf(s); row_sx[r] = sx; row_dot[r] = dot; }
  }
}

__global__ void __launch_bounds__(NLL_THREADS) nll_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ X, int n_items,
                                                              long long ld_o, long long ld_x, const float* __restrict__ row_lse,
                                                              const float* __restrict__ row_sx, const float* __restrict__ scale_ptr,
                                                              float scale_mul, float* __restrict__ grad, long long ld_g) {
  const long long r = blockIdx.x;
  const float* o = logits + r * ld_o;
  const float* x = X + r * ld_x;
  float* g = grad + r * ld_g;
  const float lse = row_lse[r], sx = row_sx[r];
  const float scale = (scale_ptr ? __ldg(scale_ptr) : 1.0f) * scale_mul;
  const bool vec = ((ld_o & 3) == 0) && ((ld_x & 3) == 0) && ((ld_g & 3) == 0) && ((reinterpret_cast<uintptr_t>(logits) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && ((reinterpret_cast<uintptr_t>(grad) & 15) == 0);
  int j0 = 0;
  if (vec) {
    const int n4 = n_items >> 2;
    for (int j = threadIdx.x; j < n4; j += NLL_THREADS) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(o) + j);
      const float4 b = __ldg(reinterpret_cast<const float4*>(x) + j);
      float4 d;
      d.x = scale * fmaf(__expf(a.x - lse), sx, -b.x);
      d.y = scale * fmaf(__expf(a.y - lse), sx, -b.y);
      d.z = scale * fmaf(__expf(a.z - lse), sx, -b.z);
      d.w = scale * fmaf(__expf(a.w - lse), sx, -b.w);
      reinterpret_cast<float4*>(g)[j] = d;
    }
    j0 = n4 << 2;
  }
  for (int j = j0 + threadIdx.x; j < n_items; j += NLL_THREADS)
    g[j] = scale * fmaf(__expf(__ldg(o + j) - lse), sx, -__ldg(x + j));
}

}  // namespace sdrm

using namespace sdrm;

static int grid_for(long long work, int sms_mult = 8) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  long long blocks = (work + 255) / 256;
  long long cap = static_cast<long long>(sms) * sms_mult;  // multiple of the SM count
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

extern "C" {

int sdrm_noise_inputs(const float* d_mu, const int64_t* d_t, const float* d_ab, int64_t B, int L, float noise_divider,
                      double mu_coef, uint64_t seed, int64_t row_offset, const float* d_inj_noise,
                      const uint8_t* d_inj_masks, float* d_noise_out, float* d_in_pert, float* d_in_clean,
                      float* d_in_shift, uint8_t* d_masks_out, void* stream) {
  if (!d_mu || !d_t || !d_ab || !d_in_pert || !d_in_clean || !d_in_shift)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_noise_inputs: null pointer");
  if (B <= 0 || L <= 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_noise_inputs: bad shape");
  const long long total = (B * L + 15) / 16;   // one thread per 16 elements (a warp per 512)
  noise_inputs_kernel<<<grid_for(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_mu, reinterpret_cast<const long long*>(d_t), d_ab, B, L, noise_divider, static_cast<float>(mu_coef), seed, row_offset, d_inj_noise,
      d_inj_masks, d_noise_out, d_in_pert, d_in_clean, d_in_shift, d_masks_out);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_loss_stats(const float* d_pred, const float* d_sx, const float* d_psx, const float* d_mu, int64_t count,
                    double mu_coef, double* d_stats, void* stream) {
  if (!d_pred || !d_sx || !d_psx || !d_mu || !d_stats) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_loss_stats: null pointer");
  if (count <= 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_loss_stats: count <= 0");
  loss_stats_kernel<<<grid_for(count, 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_pred, d_sx, d_psx, d_mu, count, static_cast<float>(mu_coef * mu_coef), d_stats);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_loss_grad_seeds(const float* d_pred, const float* d_sx, const float* d_psx, const float* d_mu, int64_t count,
                         double mu_coef, const double* d_stats, float* d_g_pred, float* d_g_sx, float* d_g_psx,
                         float* d_loss_out, void* stream) {
  if (!d_pred || !d_sx || !d_psx || !d_mu || !d_stats) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_loss_grad_seeds: null pointer");
  if (count <= 0) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_loss_grad_seeds: count <= 0");
  loss_seeds_kernel<<<grid_for(count), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_pred, d_sx, d_psx, d_mu, count, static_cast<float>(mu_coef * mu_coef), d_stats, d_g_pred, d_g_sx, d_g_psx, d_loss_out);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}


int sdrm_encode_csr(const int64_t* d_indptr, const int64_t* d_indices, const float* d_values, int64_t rows, int n_items,
                    const float* d_W1T, const float* d_b1, int H, float* d_hidden, void* stream) {
  if (!d_indptr || !d_W1T || !d_b1 || !d_hidden) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_encode_csr: null pointer");
  if (rows < 0 || n_items < 1 || H < 1) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_encode_csr: bad shape");
  if (H > ENC_THREADS * ENC_MAX_PER_THREAD) return sdrm_fail(SDRM_ERR_UNSUPPORTED, "sdrm_encode_csr: hidden width above 2048");
  if (rows == 0) return SDRM_OK;
  encode_csr_kernel<<<static_cast<unsigned>(rows), ENC_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const long long*>(d_indptr), reinterpret_cast<const long long*>(d_indices), d_values, n_items, d_W1T, d_b1, H,
      d_hidden);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}


int sdrm_multinomial_nll_fwd(const float* d_logits, const float* d_x, int64_t rows, int n_items, int64_t ld_logits, int64_t ld_x,
                             float* d_row_lse, float* d_row_sx, float* d_row_dot, void* stream) {
  if (!d_logits || !d_x || !d_row_lse || !d_row_sx || !d_row_dot) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_multinomial_nll_fwd: null pointer");
  if (rows < 0 || n_items < 1 || ld_logits < n_items || ld_x < n_items) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_multinomial_nll_fwd: bad shape");
  if (rows == 0) return SDRM_OK;
  nll_fwd_kernel<<<static_cast<unsigned>(rows), NLL_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(d_logits, d_x, n_items, ld_logits, ld_x,
                                                                                                   d_row_lse, d_row_sx, d_row_dot);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_multinomial_nll_bwd(const float* d_logits, const float* d_x, int64_t rows, int n_items, int64_t ld_logits, int64_t ld_x,
                             const float* d_row_lse, const float* d_row_sx, const float* d_grad_loss, float scale,
                             float* d_grad_logits, int64_t ld_grad, void* stream) {
  if (!d_logits || !d_x || !d_row_lse || !d_row_sx || !d_grad_logits) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_multinomial_nll_bwd: null pointer");
  if (rows < 0 || n_items < 1 || ld_logits < n_items || ld_x < n_items || ld_grad < n_items)
    return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_multinomial_nll_bwd: bad shape");
  if (rows == 0) return SDRM_OK;
  nll_bwd_kernel<<<static_cast<unsigned>(rows), NLL_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      d_logits, d_x, n_items, ld_logits, ld_x, d_row_lse, d_row_sx, d_grad_loss, scale, d_grad_logits, ld_grad);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

}  // extern "C"
