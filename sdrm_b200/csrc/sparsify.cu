// K4 — equal-sparsity thresholding of the synthetic score matrix on the device
// (reference: main.py:177-185, 259-262 and hyperparameter_search.py:162-166:
//   threshold = np.quantile(S.flatten(), SPARSITY);  S_bin = (S >= threshold).astype(int)
//   lower tail for the NeuMF negatives: S <= np.quantile(S.flatten(), 1 - SPARSITY)).
//
// The reference sorts/partitions the whole [n, I] float32 matrix on the host (80 GB at the scale-up shape).
// Here the two order statistics np.quantile interpolates between are found EXACTLY by a radix select over
// order-preserving 32-bit keys: three histogram passes (11 + 11 + 10 bits) that each read the matrix once
// (HBM-bound: 4 bytes per score), with the 2048-bin histograms summed across GPUs between passes when the rows
// are sharded.  A last pass compares against the threshold and emits 1 bit per score (32x less D2H / gather
// traffic than the fp32 matrix) plus the number of ones.
//
// bfloat16 score matrices (sdrm_*_bf16) use the 32-bit key of the score widened to float32, whose low 16 bits are fixed by its
// sign (0 for a positive score, 0xFFFF for a negative one): an 11-bit and a 5-bit digit (bits 31..21, 20..16) pin the score
// exactly, so the select reads the matrix twice at 2 bytes per score, and the pack pass once more.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/sdrm_b200.h"
#include "host_util.h"

namespace sdrm {

constexpr int HIST_BINS = 2048;
constexpr int HIST_THREADS = 256;   // 8 warp-private histograms = 64 KB per block, 3 blocks per SM
constexpr int HIST_WARPS = HIST_THREADS / 32;

// float -> uint32 whose unsigned order is the float order (-inf < ... < -0 < +0 < ... < +inf < NaN)
__device__ __forceinline__ uint32_t score_key(float x) {
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Device-resident state of one quantile selection (sdrm_select_*): the radix select walks its histograms on the DEVICE, so the
// three passes, the threshold and the bit-packing are enqueued back to back without a host round trip in between.
struct SelectState {
  unsigned long long rem[2];   // rank of the two order statistics np.quantile interpolates between, inside the current prefix
  unsigned long long nan_count;
  uint32_t prefix;             // key bits fixed so far (both statistics share them, else `fallback`)
  uint32_t fallback;           // 1 = the two statistics part ways before the last digit (or the upper one lies outside the
                               //     last digit's prefix): the caller must take the host-walk path (rare)
  uint32_t two;                // 1 = two distinct ranks, 0 = a single order statistic
  uint32_t pad;
  double threshold;            // the interpolated quantile (NaN if the matrix holds a NaN, like np.quantile)
  float v0, v1;                // the two order statistics
};
static_assert(sizeof(SelectState) == 56, "SelectState layout (mirrored by sdrm_b200/sparsify.py)");

// T = float, or uint16_t for bfloat16 bits
template <typename T>
struct MatViewT {
  const T* x;
  long long rows, ld;
  int n_cols;
};
using MatView = MatViewT<float>;
using MatViewBf16 = MatViewT<uint16_t>;

__device__ __forceinline__ float bf16_bits_float(uint32_t b) { return __uint_as_float(b << 16); }

// Calls f(value) for every score of the view; float4 loads when the layout allows, grid-stride over the matrix.
template <typename F>
__device__ __forceinline__ void for_each_score(const MatView& m, F&& f) {
  const long long tid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long nth = static_cast<long long>(gridDim.x) * blockDim.x;
  const bool vec = ((m.n_cols & 3) == 0) && ((m.ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(m.x) & 15) == 0);
  if (vec) {
    const long long c4 = m.n_cols >> 2;
    const long long total = m.rows * c4;
    if (m.ld == m.n_cols) {   // contiguous: plain 1-D sweep, four independent 16-byte loads in flight per thread
      const float4* p = reinterpret_cast<const float4*>(m.x);
      long long i = tid;
      for (; i + 3 * nth < total; i += 4 * nth) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldcs(p + i + u * nth);
#pragma unroll
        for (int u = 0; u < 4; ++u) { f(v[u].x); f(v[u].y); f(v[u].z); f(v[u].w); }
      }
      for (; i < total; i += nth) {
        const float4 v = __ldcs(p + i);
        f(v.x); f(v.y); f(v.z); f(v.w);
      }
    } else {
      for (long long i = tid; i < total; i += nth) {
        const long long r = i / c4, c = i - r * c4;
        const float4 v = __ldcs(reinterpret_cast<const float4*>(m.x + r * m.ld) + c);
        f(v.x); f(v.y); f(v.z); f(v.w);
      }
    }
  } else {
    const long long total = m.rows * m.n_cols;
    for (long long i = tid; i < total; i += nth) {
      const long long r = i / m.n_cols, c = i - r * m.n_cols;
      f(__ldcs(m.x + r * m.ld + c));
    }
  }
}

// bfloat16 scores: f(value widened to float32); 16-byte loads of 8 scores when the layout allows
template <typename F>
__device__ __forceinline__ void for_each_score(const MatViewBf16& m, F&& f) {
  const long long tid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long nth = static_cast<long long>(gridDim.x) * blockDim.x;
  const bool vec = ((m.n_cols & 7) == 0) && ((m.ld & 7) == 0) && ((reinterpret_cast<uintptr_t>(m.x) & 15) == 0);
  auto f8 = [&](const uint4& v) {
    f(bf16_bits_float(v.x & 0xFFFFu)); f(bf16_bits_float(v.x >> 16));
    f(bf16_bits_float(v.y & 0xFFFFu)); f(bf16_bits_float(v.y >> 16));
    f(bf16_bits_float(v.z & 0xFFFFu)); f(bf16_bits_float(v.z >> 16));
    f(bf16_bits_float(v.w & 0xFFFFu)); f(bf16_bits_float(v.w >> 16));
  };
  if (vec) {
    const long long c8 = m.n_cols >> 3;
    const long long total = m.rows * c8;
    if (m.ld == m.n_cols) {   // contiguous: plain 1-D sweep, four independent 16-byte loads in flight per thread
      const uint4* p = reinterpret_cast<const uint4*>(m.x);
      long long i = tid;
      for (; i + 3 * nth < total; i += 4 * nth) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldcs(p + i + u * nth);
#pragma unroll
        for (int u = 0; u < 4; ++u) f8(v[u]);
      }
      for (; i < total; i += nth) f8(__ldcs(p + i));
    } else {
      for (long long i = tid; i < total; i += nth) {
        const long long r = i / c8, c = i - r * c8;
        f8(__ldcs(reinterpret_cast<const uint4*>(m.x + r * m.ld) + c));
      }
    }
  } else {
    const long long total = m.rows * m.n_cols;
    for (long long i = tid; i < total; i += nth) {
      const long long r = i / m.n_cols, c = i - r * m.n_cols;
      f(bf16_bits_float(__ldcs(m.x + r * m.ld + c)));
    }
  }
}

// One radix-select pass: histogram of the `bits`-wide digit at `shift` over the keys whose top `prefix_bits` bits equal
// `prefix`; each warp keeps a private shared-memory histogram (no inter-warp conflicts), merged into global memory once.
template <typename T>
__global__ void __launch_bounds__(HIST_THREADS) key_hist_kernel(MatViewT<T> m, uint32_t prefix, int prefix_bits, int shift, int bits,
                                                               unsigned long long* __restrict__ hist, SelectState* __restrict__ st) {
  extern __shared__ uint32_t sh[];   // [HIST_WARPS][HIST_BINS]
  for (int i = threadIdx.x; i < HIST_WARPS * HIST_BINS; i += HIST_THREADS) sh[i] = 0;
  __syncthreads();
  if (st) prefix = st->prefix;       // device-side selection: the prefix was written by select_walk_kernel
  unsigned int nans = 0;
  const bool count_nan = st != nullptr && prefix_bits == 0;
  uint32_t* mine = sh + (threadIdx.x >> 5) * HIST_BINS;
  const uint32_t mask = (1u << bits) - 1u;
  const int pshift = 32 - prefix_bits;
  auto add = [&](float v) {
    const uint32_t k = score_key(v);
    // Plain shared-memory atomics on the warp-private histogram.  Even for the first digit, whose distribution is extremely
    // skewed (a handful of exponent values), the hardware's in-warp conflict serialisation is 4.7x faster than merging
    // equal bins with match.any first (measured on B200: 2.08 ms vs 9.69 ms for 10 GB).
    if (prefix_bits == 0 || (k >> pshift) == prefix) atomicAdd(mine + ((k >> shift) & mask), 1u);
    if (count_nan && v != v) ++nans;   // np.quantile returns NaN as soon as one score is NaN
  };
  for_each_score(m, add);
  __syncthreads();
  for (int b = threadIdx.x; b < HIST_BINS; b += HIST_THREADS) {
    unsigned long long s = 0;
#pragma unroll
    for (int w = 0; w < HIST_WARPS; ++w) s += sh[w * HIST_BINS + b];
    if (s) atomicAdd(hist + b, s);
  }
  if (count_nan) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nans += __shfl_xor_sync(0xffffffffu, nans, o);
    if ((threadIdx.x & 31) == 0 && nans) atomicAdd(&st->nan_count, static_cast<unsigned long long>(nans));
  }
}

__global__ void select_init_kernel(SelectState* st, unsigned long long r0, unsigned long long r1) {
  st->rem[0] = r0; st->rem[1] = r1; st->nan_count = 0; st->prefix = 0; st->fallback = 0; st->two = (r1 != r0) ? 1u : 0u; st->pad = 0;
  st->threshold = 0.0; st->v0 = st->v1 = 0.0f;
}

__device__ __forceinline__ float key_float(uint32_t key) {
  const uint32_t u = (key & 0x80000000u) ? (key ^ 0x80000000u) : ~key;
  return __uint_as_float(u);
}

// One block walks one (all-reduced) histogram: finds the digit of the lower order statistic, checks that the upper one (rank
// + 1) shares it, narrows the prefix; behind the LAST digit it rebuilds the two floats and interpolates with NumPy's rule
// (numpy/lib/_function_base_impl.py _lerp; since NumPy 2.0 gamma is float32 for float32 data, before it was float64).
// low_bits: key bits below the last digit (16 for bfloat16 scores: their value follows from the sign bit, see the top).
__global__ void __launch_bounds__(1024) select_walk_kernel(const unsigned long long* __restrict__ hist, SelectState* st, int bits, int last,
                                                           double gamma, int gamma_f32, int low_bits) {
  __shared__ unsigned long long cum[HIST_BINS];
  __shared__ unsigned long long part[32];
  const int n = 1 << bits;
  const int t = threadIdx.x;
  // inclusive scan of up to 2048 bins with 1024 threads (two bins per thread)
  const unsigned long long a = (2 * t < n) ? hist[2 * t] : 0ull, b = (2 * t + 1 < n) ? hist[2 * t + 1] : 0ull;
  unsigned long long v = a + b;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long u = __shfl_up_sync(0xffffffffu, v, o);
    if ((t & 31) >= o) v += u;
  }
  if ((t & 31) == 31) part[t >> 5] = v;
  __syncthreads();
  if (t < 32) {
    unsigned long long p = part[t];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long u = __shfl_up_sync(0xffffffffu, p, o);
      if (t >= o) p += u;
    }
    part[t] = p;
  }
  __syncthreads();
  const unsigned long long base = (t >= 32) ? part[(t >> 5) - 1] : 0ull;
  if (2 * t < n) cum[2 * t] = base + v - b;
  if (2 * t + 1 < n) cum[2 * t + 1] = base + v;
  __syncthreads();
  if (t == 0) {
    const unsigned long long r0 = st->rem[0];
    // first bin whose inclusive count exceeds r0 (binary search)
    int lo = 0, hi = n - 1;
    if (r0 >= cum[n - 1]) { st->fallback = 1; return; }   // rank beyond the number of scores: let the host path raise
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (cum[mid] > r0) hi = mid; else lo = mid + 1; }
    const int b0 = lo;
    const unsigned long long before = b0 ? cum[b0 - 1] : 0ull;
    int b1 = b0;
    if (st->two && r0 + 1 >= cum[b0]) {
      // the upper statistic is the first score of a later bin
      b1 = b0 + 1;
      while (b1 < n && cum[b1] == cum[b0]) ++b1;
      if (!last || b1 >= n) st->fallback = 1;
    }
    const uint32_t p0 = (st->prefix << bits) | static_cast<uint32_t>(b0);
    if (!last) {
      st->prefix = p0;
      st->rem[0] = r0 - before;
    } else {
      const uint32_t p1 = (st->prefix << bits) | static_cast<uint32_t>(b1 < n ? b1 : b0);
      auto full_key = [&](uint32_t p) {
        if (low_bits == 0) return p;
        const uint32_t positive = (p >> (31 - low_bits)) & 1u;
        return (p << low_bits) | (positive ? 0u : (1u << low_bits) - 1u);
      };
      const float x0 = key_float(full_key(p0)), x1 = st->two ? key_float(full_key(p1)) : x0;
      st->v0 = x0; st->v1 = x1;
      double thr;
      if (gamma_f32) {   // float32 arithmetic without contraction, exactly _lerp on np.float32 scalars
        const float g = static_cast<float>(gamma);
        const float diff = __fsub_rn(x1, x0);
        float o = __fadd_rn(x0, __fmul_rn(diff, g));
        if (g >= 0.5f) o = __fsub_rn(x1, __fmul_rn(diff, __fsub_rn(1.0f, g)));
        thr = static_cast<double>(o);
      } else {           // NumPy < 2.0: gamma is float64, the float32 difference is promoted
        const double diff = static_cast<double>(__fsub_rn(x1, x0));
        double o = __dadd_rn(static_cast<double>(x0), __dmul_rn(diff, gamma));
        if (gamma >= 0.5) o = __dsub_rn(static_cast<double>(x1), __dmul_rn(diff, __dsub_rn(1.0, gamma)));
        thr = o;
      }
      if (st->nan_count) thr = __longlong_as_double(0x7ff8000000000000ll);
      st->threshold = thr;
    }
  }
}

// bits[row][w] bit j = (score[row][32 w + j] >= thr)  (mode 0)  or  <= thr (mode 1).  A warp walks whole rows: every lane
// loads 4 consecutive scores (a 512-byte coalesced warp load, two in flight), forms its 4-bit nibble and three xor-shuffles
// assemble the four 32-bit words of the 128 columns.
template <int MODE>
__device__ __forceinline__ float device_threshold(float thr, const SelectState* __restrict__ st) {
  if (st) {   // threshold selected on the device: same double -> float32 predicate conversion as the host entry
    const double td = st->threshold;
    thr = static_cast<float>(td);
    if (MODE == 0 && static_cast<double>(thr) < td) thr = nextafterf(thr, INFINITY);
    if (MODE == 1 && static_cast<double>(thr) > td) thr = nextafterf(thr, -INFINITY);
  }
  return thr;
}

template <int MODE>
__global__ void __launch_bounds__(256) threshold_pack_kernel(MatView m, float thr, uint32_t* __restrict__ bits,
                                                             long long words_per_row, unsigned long long* __restrict__ count,
                                                             const SelectState* __restrict__ st) {
  const int lane = threadIdx.x & 31;
  thr = device_threshold<MODE>(thr, st);
  const long long warp = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long n_warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const bool vec = ((m.ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(m.x) & 15) == 0);
  const int n_cols = m.n_cols;
  unsigned long long ones = 0;
  auto hit = [&](float v) { return MODE == 0 ? (v >= thr) : (v <= thr); };
  for (long long r = warp; r < m.rows; r += n_warps) {
    const float* x = m.x + r * m.ld;
    uint32_t* out = bits + r * words_per_row;
    int c0 = 0;
    // interior: whole 512-column spans of 16-byte aligned rows, four loads in flight per lane, no per-element range checks
    if (vec) {
      for (; c0 + 512 <= n_cols; c0 += 512) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldcs(reinterpret_cast<const float4*>(x + c0 + u * 128 + lane * 4));
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint32_t w = ((hit(v[u].x) ? 1u : 0u) | (hit(v[u].y) ? 2u : 0u) | (hit(v[u].z) ? 4u : 0u) | (hit(v[u].w) ? 8u : 0u)) << (4 * (lane & 7));
          w |= __shfl_xor_sync(0xffffffffu, w, 1);
          w |= __shfl_xor_sync(0xffffffffu, w, 2);
          w |= __shfl_xor_sync(0xffffffffu, w, 4);
          if ((lane & 7) == 0) {
            out[(c0 + u * 128) / 32 + (lane >> 3)] = w;
            ones += __popc(w);
          }
        }
      }
    }
    for (; c0 < n_cols; c0 += 256) {
      uint32_t nib[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int c = c0 + u * 128 + lane * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        bool ok[4] = {c < n_cols, c + 1 < n_cols, c + 2 < n_cols, c + 3 < n_cols};
        if (vec && ok[3]) {
          v = __ldcs(reinterpret_cast<const float4*>(x + c));
        } else {
          if (ok[0]) v.x = __ldcs(x + c);
          if (ok[1]) v.y = __ldcs(x + c + 1);
          if (ok[2]) v.z = __ldcs(x + c + 2);
          if (ok[3]) v.w = __ldcs(x + c + 3);
        }
        nib[u] = (ok[0] && hit(v.x) ? 1u : 0u) | (ok[1] && hit(v.y) ? 2u : 0u) | (ok[2] && hit(v.z) ? 4u : 0u) | (ok[3] && hit(v.w) ? 8u : 0u);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        // lane l holds columns 4l..4l+3 of this 128-column block: word l/8, bits 4 (l%8) ..
        uint32_t w = nib[u] << (4 * (lane & 7));
        w |= __shfl_xor_sync(0xffffffffu, w, 1);
        w |= __shfl_xor_sync(0xffffffffu, w, 2);
        w |= __shfl_xor_sync(0xffffffffu, w, 4);
        const int word = (c0 + u * 128) / 32 + (lane >> 3);
        if ((lane & 7) == 0 && word * 32 < n_cols) {
          out[word] = w;
          ones += __popc(w);
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ones += __shfl_xor_sync(0xffffffffu, ones, o);
  if (count && lane == 0 && ones) atomicAdd(count, ones);
}

// The same on bfloat16 scores (compared widened to float32: exact).  A lane loads 8 consecutive scores (one 16-byte load, a
// 512-byte warp load of 256 columns) and forms their byte; two xor-shuffles assemble the eight 32-bit words.
template <int MODE>
__global__ void __launch_bounds__(256) threshold_pack_bf16_kernel(MatViewBf16 m, float thr, uint32_t* __restrict__ bits,
                                                                  long long words_per_row, unsigned long long* __restrict__ count,
                                                                  const SelectState* __restrict__ st) {
  const int lane = threadIdx.x & 31;
  thr = device_threshold<MODE>(thr, st);
  const long long warp = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long n_warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const bool vec = ((m.ld & 7) == 0) && ((reinterpret_cast<uintptr_t>(m.x) & 15) == 0);
  const int n_cols = m.n_cols;
  unsigned long long ones = 0;
  auto hit = [&](uint32_t b) { const float v = bf16_bits_float(b); return MODE == 0 ? (v >= thr) : (v <= thr); };
  auto byte_of = [&](const uint4& v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t r = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) r |= (hit(w[k] & 0xFFFFu) ? 1u : 0u) << (2 * k) | (hit(w[k] >> 16) ? 1u : 0u) << (2 * k + 1);
    return r;
  };
  // lane l holds columns 8l..8l+7 of a 256-column block: word l/4, bits 8 (l%4) ..
  auto emit = [&](uint32_t byte, uint32_t* out, int c_block) {
    uint32_t w = byte << (8 * (lane & 3));
    w |= __shfl_xor_sync(0xffffffffu, w, 1);
    w |= __shfl_xor_sync(0xffffffffu, w, 2);
    const int word = c_block / 32 + (lane >> 2);
    if ((lane & 3) == 0 && word * 32 < n_cols) {
      out[word] = w;
      ones += __popc(w);
    }
  };
  for (long long r = warp; r < m.rows; r += n_warps) {
    const uint16_t* x = m.x + r * m.ld;
    uint32_t* out = bits + r * words_per_row;
    int c0 = 0;
    // interior: whole 1024-column spans of 16-byte aligned rows, four loads in flight per lane, no per-element range checks
    if (vec) {
      for (; c0 + 1024 <= n_cols; c0 += 1024) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldcs(reinterpret_cast<const uint4*>(x + c0 + u * 256 + lane * 8));
#pragma unroll
        for (int u = 0; u < 4; ++u) emit(byte_of(v[u]), out, c0 + u * 256);
      }
    }
    for (; c0 < n_cols; c0 += 256) {
      const int c = c0 + lane * 8;
      uint32_t byte = 0;
      if (vec && c + 8 <= n_cols) {
        byte = byte_of(__ldcs(reinterpret_cast<const uint4*>(x + c)));
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (c + k < n_cols && hit(__ldcs(x + c + k))) byte |= 1u << k;
      }
      emit(byte, out, c0);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ones += __shfl_xor_sync(0xffffffffu, ones, o);
  if (count && lane == 0 && ones) atomicAdd(count, ones);
}

static int grid_for(long long work_items, int threads, int per_thread, int blocks_per_sm) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  long long blocks = (work_items + static_cast<long long>(threads) * per_thread - 1) / (static_cast<long long>(threads) * per_thread);
  const long long cap = static_cast<long long>(sms) * blocks_per_sm;   // one resident wave: a multiple of the SM count
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace sdrm

using namespace sdrm;

// ---- host side, shared by the float32 and the bfloat16 entries (T = float / uint16_t) -----------------------------------------
template <typename T>
static int launch_key_hist(const T* d_scores, int64_t rows, int n_cols, int64_t ld, uint32_t prefix, int prefix_bits,
                           int shift, int bits, unsigned long long* d_hist, SelectState* st, void* stream) {
  static bool attr_done = false;
  const int smem = HIST_WARPS * HIST_BINS * static_cast<int>(sizeof(uint32_t));   // 64 KB
  if (!attr_done) {
    SDRM_CUDA(cudaFuncSetAttribute(key_hist_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_done = true;
  }
  MatViewT<T> m{d_scores, rows, ld, n_cols};
  const int grid = grid_for(rows * static_cast<long long>(n_cols), HIST_THREADS, 64, 3);
  key_hist_kernel<T><<<grid, HIST_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(m, prefix, prefix_bits, shift, bits, d_hist, st);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

template <typename T>
static int key_histogram(const char* what, const T* d_scores, int64_t rows, int n_cols, int64_t ld, uint32_t prefix, int prefix_bits,
                         int shift, int bits, unsigned long long* d_hist, void* stream) {
  char msg[160];
  if (!d_scores || !d_hist) { snprintf(msg, sizeof msg, "%s: null pointer", what); return sdrm_fail(SDRM_ERR_BAD_ARG, msg); }
  if (rows < 0 || n_cols <= 0 || ld < n_cols) { snprintf(msg, sizeof msg, "%s: bad shape", what); return sdrm_fail(SDRM_ERR_BAD_ARG, msg); }
  if (bits < 1 || bits > 11 || shift < 0 || shift + bits > 32 || prefix_bits < 0 || prefix_bits > 31 || prefix_bits + bits + shift != 32) {
    snprintf(msg, sizeof msg, "%s: digit layout (prefix_bits + bits + shift must be 32, bits <= 11)", what);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  if (rows == 0) return SDRM_OK;
  return launch_key_hist<T>(d_scores, rows, n_cols, ld, prefix, prefix_bits, shift, bits, d_hist, nullptr, stream);
}

// Digits of the device-side select: float32 keys 11 + 11 + 10 bits, bfloat16 keys 11 + 5 (the low 16 key bits follow from the sign)
static const int kDigitBits[3] = {11, 11, 10}, kDigitShift[3] = {21, 10, 0};
static const int kDigitBitsBf16[2] = {11, 5}, kDigitShiftBf16[2] = {21, 16};

template <typename T>
static int select_histogram(const char* what, const T* d_scores, int64_t rows, int n_cols, int64_t ld, void* d_state, int digit,
                            unsigned long long* d_hist, void* stream) {
  constexpr bool BF16 = std::is_same<T, uint16_t>::value;
  const int n_digits = BF16 ? 2 : 3;
  char msg[160];
  if (!d_scores || !d_hist || !d_state) { snprintf(msg, sizeof msg, "%s: null pointer", what); return sdrm_fail(SDRM_ERR_BAD_ARG, msg); }
  if (rows < 0 || n_cols <= 0 || ld < n_cols || digit < 0 || digit >= n_digits) {
    snprintf(msg, sizeof msg, "%s: bad shape / digit", what);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  if (rows == 0) return SDRM_OK;
  const int bits = BF16 ? kDigitBitsBf16[digit] : kDigitBits[digit], shift = BF16 ? kDigitShiftBf16[digit] : kDigitShift[digit];
  return launch_key_hist<T>(d_scores, rows, n_cols, ld, 0u, 32 - bits - shift, shift, bits, d_hist, static_cast<SelectState*>(d_state),
                            stream);
}

template <typename T>
static int threshold_pack(const char* what, const T* d_scores, int64_t rows, int n_cols, int64_t ld, float tf, const void* d_state, int mode,
                          uint32_t* d_bits, int64_t words_per_row, unsigned long long* d_count, void* stream) {
  char msg[160];
  if (!d_scores || !d_bits) { snprintf(msg, sizeof msg, "%s: null pointer", what); return sdrm_fail(SDRM_ERR_BAD_ARG, msg); }
  if (rows < 0 || n_cols <= 0 || ld < n_cols || words_per_row < (n_cols + 31) / 32 || (mode != 0 && mode != 1)) {
    snprintf(msg, sizeof msg, "%s: bad shape / mode", what);
    return sdrm_fail(SDRM_ERR_BAD_ARG, msg);
  }
  if (rows == 0) return SDRM_OK;
  MatViewT<T> m{d_scores, rows, ld, n_cols};
  const int grid = grid_for(rows * 32, 256, 1, 8);   // one warp per row until the wave is full
  const SelectState* st = static_cast<const SelectState*>(d_state);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if constexpr (std::is_same<T, uint16_t>::value) {
    if (mode == 0) threshold_pack_bf16_kernel<0><<<grid, 256, 0, s>>>(m, tf, d_bits, words_per_row, d_count, st);
    else threshold_pack_bf16_kernel<1><<<grid, 256, 0, s>>>(m, tf, d_bits, words_per_row, d_count, st);
  } else {
    if (mode == 0) threshold_pack_kernel<0><<<grid, 256, 0, s>>>(m, tf, d_bits, words_per_row, d_count, st);
    else threshold_pack_kernel<1><<<grid, 256, 0, s>>>(m, tf, d_bits, words_per_row, d_count, st);
  }
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

// The scores are float32 (or bfloat16, exact in float32): x >= t (double) is the same predicate as x >= the smallest float32 not
// below t (and x <= t the same as x <= the largest float32 not above t), so the device compares in fp32 (B200 runs FP64 at a
// fraction of the rate).
static float predicate_threshold(double threshold, int mode) {
  float tf = static_cast<float>(threshold);
  if (mode == 0 && static_cast<double>(tf) < threshold) tf = nextafterf(tf, INFINITY);
  if (mode == 1 && static_cast<double>(tf) > threshold) tf = nextafterf(tf, -INFINITY);
  return tf;
}

extern "C" {

int sdrm_key_histogram(const float* d_scores, int64_t rows, int n_cols, int64_t ld, uint32_t prefix, int prefix_bits,
                       int shift, int bits, unsigned long long* d_hist, void* stream) {
  return key_histogram("sdrm_key_histogram", d_scores, rows, n_cols, ld, prefix, prefix_bits, shift, bits, d_hist, stream);
}

int sdrm_key_histogram_bf16(const uint16_t* d_scores, int64_t rows, int n_cols, int64_t ld, uint32_t prefix, int prefix_bits,
                            int shift, int bits, unsigned long long* d_hist, void* stream) {
  return key_histogram("sdrm_key_histogram_bf16", d_scores, rows, n_cols, ld, prefix, prefix_bits, shift, bits, d_hist, stream);
}

size_t sdrm_select_state_bytes(void) { return sizeof(SelectState); }

int sdrm_select_begin(void* d_state, uint64_t rank_lo, uint64_t rank_hi, void* stream) {
  if (!d_state || rank_hi < rank_lo || rank_hi > rank_lo + 1) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_select_begin: state / ranks (rank_hi must be rank_lo or rank_lo + 1)");
  select_init_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<SelectState*>(d_state), rank_lo, rank_hi);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_select_histogram(const float* d_scores, int64_t rows, int n_cols, int64_t ld, void* d_state, int digit,
                          unsigned long long* d_hist, void* stream) {
  return select_histogram("sdrm_select_histogram", d_scores, rows, n_cols, ld, d_state, digit, d_hist, stream);
}

int sdrm_select_histogram_bf16(const uint16_t* d_scores, int64_t rows, int n_cols, int64_t ld, void* d_state, int digit,
                               unsigned long long* d_hist, void* stream) {
  return select_histogram("sdrm_select_histogram_bf16", d_scores, rows, n_cols, ld, d_state, digit, d_hist, stream);
}

int sdrm_select_walk(const unsigned long long* d_hist, void* d_state, int digit, double gamma, int gamma_is_f32, void* stream) {
  if (!d_hist || !d_state || digit < 0 || digit > 2) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_select_walk: bad argument");
  select_walk_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(d_hist, static_cast<SelectState*>(d_state), kDigitBits[digit], digit == 2, gamma,
                                                                        gamma_is_f32, 0);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_select_walk_bf16(const unsigned long long* d_hist, void* d_state, int digit, double gamma, int gamma_is_f32, void* stream) {
  if (!d_hist || !d_state || digit < 0 || digit > 1) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_select_walk_bf16: bad argument");
  select_walk_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(d_hist, static_cast<SelectState*>(d_state), kDigitBitsBf16[digit], digit == 1,
                                                                        gamma, gamma_is_f32, 16);
  SDRM_CUDA(cudaGetLastError());
  return SDRM_OK;
}

int sdrm_select_threshold_pack(const float* d_scores, int64_t rows, int n_cols, int64_t ld, const void* d_state, int mode,
                               uint32_t* d_bits, int64_t words_per_row, unsigned long long* d_count, void* stream) {
  if (!d_state) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_select_threshold_pack: null pointer");
  return threshold_pack("sdrm_select_threshold_pack", d_scores, rows, n_cols, ld, 0.0f, d_state, mode, d_bits, words_per_row, d_count, stream);
}

int sdrm_select_threshold_pack_bf16(const uint16_t* d_scores, int64_t rows, int n_cols, int64_t ld, const void* d_state, int mode,
                                    uint32_t* d_bits, int64_t words_per_row, unsigned long long* d_count, void* stream) {
  if (!d_state) return sdrm_fail(SDRM_ERR_BAD_ARG, "sdrm_select_threshold_pack_bf16: null pointer");
  return threshold_pack("sdrm_select_threshold_pack_bf16", d_scores, rows, n_cols, ld, 0.0f, d_state, mode, d_bits, words_per_row, d_count,
                        stream);
}

int sdrm_threshold_pack(const float* d_scores, int64_t rows, int n_cols, int64_t ld, double threshold, int mode,
                        uint32_t* d_bits, int64_t words_per_row, unsigned long long* d_count, void* stream) {
  return threshold_pack("sdrm_threshold_pack", d_scores, rows, n_cols, ld, predicate_threshold(threshold, mode), nullptr, mode, d_bits,
                        words_per_row, d_count, stream);
}

int sdrm_threshold_pack_bf16(const uint16_t* d_scores, int64_t rows, int n_cols, int64_t ld, double threshold, int mode,
                             uint32_t* d_bits, int64_t words_per_row, unsigned long long* d_count, void* stream) {
  return threshold_pack("sdrm_threshold_pack_bf16", d_scores, rows, n_cols, ld, predicate_threshold(threshold, mode), nullptr, mode, d_bits,
                        words_per_row, d_count, stream);
}

}  // extern "C"
