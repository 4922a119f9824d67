// K1 — streaming tcgen05 layer engine for the SDRM reverse-diffusion chain and VAE decode.
//
// Replaces the reference's per-step eager op chain (sample_ddpm, train_SDRM.py:50-61; SDRM.forward
// 97-103; denoise_add_noise 20-25; VAE.decode 252-254) with ONE persistent kernel:
//   * a CTA owns a 128-row tile of users for the whole T-step chain and the decode;
//   * every dense layer is a tcgen05 (UMMA) GEMM: A = bf16 activations, B = bf16 weights.  Weights are stored in global
//     memory as pre-swizzled "tile images" that a bulk / tensor-map copy drops straight into the 128B-swizzled shared-memory
//     operand layout; activation images are LINEAR rows in global memory (written by TMA tensor stores from the epilogue
//     warps' shared-memory slots) and swizzled by the TMA tensor load; accumulators live in TMEM
//     (2 x 256 columns, double-buffered so the epilogue of chunk c overlaps the UMMAs of chunk c+1);
//   * the epilogue warps fuse bias (hoisted time embedding), PReLU / tanh, the DDPM posterior update
//     with in-kernel Philox Gaussian noise, the always-on dropout of the next step's input and the
//     bf16 (or bf16 hi/lo) re-quantisation, and write the next layer's A images (L2-resident scratch);
//   * warps 0-11 = epilogue, 12-15 = noise, 16 = weight TMA producer, 17 = UMMA issuer, 18 = activation TMA producer;
//     the epilogue
//     warps also pre-compute the Gaussian half of each step's posterior update while the tensor core is busy.
// Rows are independent, so the streaming / resident flows need no synchronisation between row tiles (a tcgen05 pair shares its
// barriers, and on multi-resolution launches its two tiles' start steps).  The column-split instantiation (SPLITK, below) is the
// exception by design: a cluster of CTAs shares ONE row tile and hands the layer outputs around through cluster-wide chunk barriers.
#pragma once
#include "layer_engine.cuh"
#include "philox.cuh"
#include "ptx_sm100.cuh"

#include <type_traits>

// Event-timeline tracing (tools/trace_timeline.py) and the perf-experiment switches cost instructions in the hottest
// loops of a kernel that is bound by issue slots: both are compiled in only on request (-DSDRM_TRACE / -DSDRM_PERF_DEBUG).
#ifdef SDRM_TRACE
#define SDRM_TR(role, code) TR(role, code)
#define SDRM_TR_SEQ() (++trace_seq)
#define SDRM_TR_EPI(code) do { if (warp == 0 && lane == 0) TR(2, code); } while (0)
#else
#define SDRM_TR(role, code) do { } while (0)
#define SDRM_TR_SEQ() do { } while (0)
#define SDRM_TR_EPI(code) do { } while (0)
#endif
#ifndef SDRM_NSTG_PAIR
#define SDRM_NSTG_PAIR 6   // pair-mode pipeline depth (32 KB stages); 7 (with 31 KB stages, MAX_NC = 240) measured no faster
#endif
#ifndef SDRM_POSTERIOR_MUFU_TANH
#define SDRM_POSTERIOR_MUFU_TANH 1   // eps = tanh.approx.f32 (1 MUFU instead of ex2 + rcp + 3 FP ops) in the posterior update
#endif
#ifndef SDRM_OUT_SLOTS
#define SDRM_OUT_SLOTS 1      // shared-memory boxes per epilogue warp for the TMA activation stores; 2 = the store of a box is issued one group later
                              // (measured r02: 278.7 / 277.4 vs 275.1 / 273.7 ms per cfg-5 shard on one box: the epilogue is not the critical path there)
#endif
#ifndef SDRM_SPLIT_RELAY
#define SDRM_SPLIT_RELAY 0    // column-split mode: 1 = chunk publications go through the relay warp with a cluster-scope release (see the kernel);
                              // 0 = the epilogue warps arrive on the peers' chunk barriers themselves (default: 2.70 -> 2.54 ms at cfg 1 for dropping
                              // the release alone)
#endif
#ifndef SDRM_RES_CLUSTER_SCOPE
#define SDRM_RES_CLUSTER_SCOPE 0   // resident flow: 1 = the peer's "tile written" signal is a cluster-scope release and the UMMA issuer fences at
                                   // cluster scope behind its wait (~1.6 us per layer, see profiles/k1_split_r02.txt).  Not needed: the peer's half of
                                   // the M = 256 operand is written by the peer's threads into the PEER's shared memory (fence.proxy.async there) and
                                   // read by the peer SM's own tensor core; the leader's thread only orders its instruction issue behind the barrier.
#endif
#ifndef SDRM_STATE_CS
#define SDRM_STATE_CS 1       // fp32 state accesses carry the streaming (.cs, evict-first) hint
#endif
#if SDRM_STATE_CS
#define SDRM_ST_HINT ".cs"
#else
#define SDRM_ST_HINT ""
#endif
#ifdef SDRM_PERF_DEBUG
#define SDRM_DEBUG_SKIP_ACT_STORES (P.debug_flags & 1)
#define SDRM_DEBUG_SKIP_NOISE (P.debug_flags & 4)
#define SDRM_DEBUG_NOISE_NO_RNG (P.debug_flags & 16)       // state pass without Philox / Box-Muller (z = 0)
#define SDRM_DEBUG_NOISE_NO_STATE (P.debug_flags & 32)     // Philox / Box-Muller without the state load / store
#define SDRM_DEBUG_ACT_STORE_FIXED (P.debug_flags & 64)    // every activation box goes to row 0 of the CTA's scratch (no new dirty lines)
#define SDRM_DEBUG_NO_STORE_WAIT (P.debug_flags & 128)     // publish chunks without waiting for the TMA stores to complete
#define SDRM_DEBUG_SKIP_A_LOADS (P.debug_flags & 256)      // single-CTA / split mode: no activation loads (the stage's arrival only)
#define SDRM_DEBUG_SKIP_W_LOADS (P.debug_flags & 512)      // single-CTA / split mode: no weight loads
#else
#define SDRM_DEBUG_SKIP_ACT_STORES 0
#define SDRM_DEBUG_SKIP_NOISE 0
#define SDRM_DEBUG_NOISE_NO_RNG 0
#define SDRM_DEBUG_NOISE_NO_STATE 0
#define SDRM_DEBUG_ACT_STORE_FIXED 0
#define SDRM_DEBUG_NO_STORE_WAIT 0
#define SDRM_DEBUG_SKIP_A_LOADS 0
#define SDRM_DEBUG_SKIP_W_LOADS 0
#endif

namespace sdrm {

namespace {


__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory"); }

// fp32 state layout inside a tile: [16-col group][half 0..1][row 0..127][8 floats]; a thread moves its 16 columns with two
// 256-bit streaming accesses (evict-first: the state must not push the activation images out of L2), a warp touches
// 1 KB contiguous per access
__device__ __forceinline__ float* xstate_ptr8(float* xs, int g16, int half, int r) {
  return xs + ((static_cast<size_t>(g16) * 2 + half) * TILE_M + r) * 8;
}
__device__ __forceinline__ void xs_load16(float* xs, int g16, int r, float (&x)[16]) {
#pragma unroll
  for (int hf = 0; hf < 2; ++hf)
    asm volatile("ld.global" SDRM_ST_HINT ".v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(x[8 * hf + 0]), "=f"(x[8 * hf + 1]), "=f"(x[8 * hf + 2]), "=f"(x[8 * hf + 3]), "=f"(x[8 * hf + 4]),
                   "=f"(x[8 * hf + 5]), "=f"(x[8 * hf + 6]), "=f"(x[8 * hf + 7])
                 : "l"(xstate_ptr8(xs, g16, hf, r))
                 : "memory");
}
__device__ __forceinline__ void xs_store16(float* xs, int g16, int r, const float (&x)[16]) {
#pragma unroll
  for (int hf = 0; hf < 2; ++hf)
    asm volatile("st.global" SDRM_ST_HINT ".v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"l"(xstate_ptr8(xs, g16, hf, r)), "f"(x[8 * hf + 0]), "f"(x[8 * hf + 1]), "f"(x[8 * hf + 2]), "f"(x[8 * hf + 3]),
                   "f"(x[8 * hf + 4]), "f"(x[8 * hf + 5]), "f"(x[8 * hf + 6]), "f"(x[8 * hf + 7])
                 : "memory");
}

}  // namespace

// PAIR = false: one CTA per row tile, tcgen05 cta_group::1, 4 stages of (A 16 KB + W 32 KB).
// PAIR = true : two CTAs (a thread-block cluster of 2 = one TPC) work as a tcgen05 cta_group::2 pair on TWO row tiles
//               (UMMA M = 256): each CTA stages its own A tile and only HALF of every weight k-block, so a stage is
//               32 KB and 7 of them fit -> 75 % more k-blocks in flight per SM, and half the weight bytes per SM.
//               The L2 round trip under load (~1.5 us) times the bytes per k-block is what bounds this kernel
//               (Little's law on 192 KB of staging), which is why the pair mode is the fast path.
//               (r01 / r02 also carried CS = 4 / 8: clusters of 2 / 4 pairs in lock step that shared one TMA-multicast weight
//               stream.  They never won: only 132 of the 148 SMs can hold clusters of 4, and a CS = 4 launch on those plus a
//               CS = 2 launch on the other 16 SMs measured 4.04 row tiles per ms against 4.02 for CS = 2 everywhere
//               (profiles/k1_bound_r02.txt): the kernel is bound by board power, not by L2 -> SM bytes.  Pruned.)
// RESK: the resident-mode instantiation (see below).  A template parameter, not a run-time flag: the streaming instantiation must not
// carry the mode's branches in the single-thread UMMA issue loop and in the epilogue group loops (measured: +1.2 % per cfg-5 shard).
// SPLITK: the column-split instantiation (see below): single-CTA tcgen05, a CLUSTER of 2 / 4 / 8 CTAs shares one row tile.
// BF16OUT: the logits are stored as bfloat16 (round to nearest even of the fp32 value the fp32 instantiation writes; P.logits
// points to uint16_t bits, ld_logits counts elements).  Only the decoder's last epilogue differs; the fp32 instantiations carry
// none of it.
template <int CS, bool RESK = false, bool SPLITK = false, bool BF16OUT = false>
__global__ void __launch_bounds__(ENGINE_THREADS, 1) sdrm_layer_engine_kernel(const __grid_constant__ ChainParams P) {
  static_assert(!RESK || CS == 2, "resident mode runs on CTA pairs");
  static_assert(!SPLITK || CS == 1, "column-split clusters are built from single-CTA (cta_group::1) tiles");
  static_assert(CS == 1 || CS == 2, "single CTAs or one tcgen05 pair per cluster");
  constexpr bool PAIR = CS == 2;
  constexpr int NSTG = PAIR ? SDRM_NSTG_PAIR : 4;
  constexpr uint32_t W_STAGE_BYTES = PAIR ? static_cast<uint32_t>(MAX_NC / 2 * 128) : static_cast<uint32_t>(MAX_NC * 128);
  static_assert((A_TILE_BYTES + W_STAGE_BYTES) % 1024 == 0, "stages stay 1024-byte aligned (SWIZZLE_128B operand atoms)");
  constexpr uint32_t STG_BYTES = A_TILE_BYTES + W_STAGE_BYTES;
  constexpr int NCTA = CS;
  constexpr int BIAS_SLOTS = (16 + EPI_SUB - 1) / EPI_SUB;            // column groups of one chunk a warp can own
  constexpr uint32_t BIAS_SLICE_BYTES = BIAS_SLOTS * 16 * 4;         // per epilogue warp: the bias of its column groups of one chunk
  constexpr int NBAR = 3 * NSTG + 5 + MAX_SUB * (MAX_ACT_CHUNKS + 6) + 6;   // mbarriers of a CTA (map below)
  constexpr uint32_t OUT_SLOT_BYTES = 32 * 32;        // one 16-column group of a warp's 32 rows, dense bf16 (TMA store box)
  constexpr uint32_t OUT_SLOTS_PER_WARP = SDRM_OUT_SLOTS;
  static_assert(NSTG * STG_BYTES + 8 * NBAR + 256 + EPI_WARPS * (BIAS_SLICE_BYTES + OUT_SLOTS_PER_WARP * OUT_SLOT_BYTES) + 128 + 1023 <= ENGINE_SMEM_BYTES, "smem budget");

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base_addr = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base_addr - raw_addr);
  const uint32_t bar_base = base_addr + NSTG * STG_BYTES;
  // barrier map (8 bytes each): full[NSTG] | empty[NSTG] | (unused NSTG) | acc_full[2] | acc_empty[2] | tile_ready |
  //                             act_chunk[MAX_SUB][MAX_ACT_CHUNKS] | state_ready[MAX_SUB] | noise_ready[MAX_SUB] |
  //                             layer_consumed[MAX_SUB][2] | discard_done[MAX_SUB][2]
  // column-split mode: the stage size follows the launch's widest chunk (A 16 KB + NC x 128 B of weights), so that up to 6 stages
  // fit the same 192 KB ring.  (Measured at cfg 1: 6 stages of 32 KB run like 4 of 48 KB -- neither the ring depth nor the bytes
  // bound a split layer, its single-warp control loops did: profiles/k1_split_r02.txt.)
  constexpr int NSTG_B = SPLITK ? 6 : NSTG;   // barrier slots per array (2 x 6 fit the 3 x 4 slots of the single-CTA map)
  static_assert(2 * NSTG_B <= 3 * NSTG, "full / empty barrier slots");
  const uint32_t stg_bytes = SPLITK ? P.split_stage_bytes : STG_BYTES;
  auto stage_a = [&](uint32_t s) { return base_addr + s * stg_bytes; };
  auto stage_w = [&](uint32_t s) { return base_addr + s * stg_bytes + A_TILE_BYTES; };
  auto bar_full = [&](uint32_t s) { return bar_base + 8u * s; };
  auto bar_empty = [&](uint32_t s) { return bar_base + 8u * (NSTG_B + s); };
  auto bar_acc_full = [&](uint32_t b) { return bar_base + 8u * (3 * NSTG + b); };
  auto bar_acc_empty = [&](uint32_t b) { return bar_base + 8u * (3 * NSTG + 2 + b); };
  const uint32_t bar_tile_ready = bar_base + 8u * (3 * NSTG + 4);
  // one barrier per chunk INDEX: chunk c of layer l+1 cannot finish before the A producer consumed chunk c of layer l,
  // so a waiter never lags more than one phase (a single barrier would be lapped by fast chunk epilogues)
  // (one set per interleaved row tile s, see "sub-tiles" below)
  auto bar_act_chunk = [&](uint32_t s, uint32_t c) { return bar_base + 8u * (3 * NSTG + 5 + s * MAX_ACT_CHUNKS + c); };
  auto bar_state_ready = [&](uint32_t s) { return bar_base + 8u * (3 * NSTG + 5 + MAX_SUB * MAX_ACT_CHUNKS + s); };            // epilogue -> noise warps
  auto bar_noise_ready = [&](uint32_t s) { return bar_base + 8u * (3 * NSTG + 5 + MAX_SUB * MAX_ACT_CHUNKS + MAX_SUB + s); };  // noise warps -> epilogue
  // dead-buffer discard (pair mode): the UMMA issuer commits `layer_consumed` behind a chain layer's last UMMA (its input image
  // has been read for the last time), the discard warp drops those lines from the L2 and signals `discard_done`, which the
  // epilogue warps check before the NEXT layer's first store into that buffer
  // Both are rings of TWO barriers per sub-tile, indexed by the low bit of the sub-tile's layer count k (parity = bit 1 of k):
  // with interleaved sub-tiles the UMMAs of a two-chunk layer can retire a whole layer ahead of the epilogue, so up to two
  // phases of a sub-tile are outstanding and a single barrier would be lapped (parity aliasing = deadlock).
  auto bar_layer_consumed = [&](uint32_t s, uint32_t k) { return bar_base + 8u * (3 * NSTG + 5 + MAX_SUB * MAX_ACT_CHUNKS + 2 * MAX_SUB + 2 * s + (k & 1u)); };
  auto bar_discard_done = [&](uint32_t s, uint32_t k) { return bar_base + 8u * (3 * NSTG + 5 + MAX_SUB * MAX_ACT_CHUNKS + 4 * MAX_SUB + 2 * s + (k & 1u)); };
  // resident mode: a_ready = this CTA's epilogue warps have written the whole input tile of the next chain layer into shared
  // memory; peer_ready (leader's copy) = the same for the peer CTA, relayed by the peer's otherwise idle UMMA warp
  const uint32_t bar_a_ready = bar_base + 8u * (3 * NSTG + 5 + MAX_SUB * (MAX_ACT_CHUNKS + 6));
  const uint32_t bar_peer_ready = bar_a_ready + 8u;
  // resident mode, two-chunk layers: the second chunk's UMMAs have read the k-blocks that the FIRST chunk's output overwrites
  const uint32_t bar_half_read = bar_a_ready + 16u;
  // column-split mode: epilogue warps -> relay warp ("this CTA's chunk of the layer's output is in the L2"), a ring of two
  auto bar_relay = [&](uint32_t k) { return bar_a_ready + 24u + 8u * (k & 1u); };
  // multi-resolution chains on a CTA pair: the peer's tile start step has arrived (one phase per tile iteration)
  const uint32_t bar_pair_T = bar_a_ready + 40u;
  // per-role layer counters: two bits per sub-tile (k mod 4 is all the ring index and the parity need)
  auto cnt_get = [](uint32_t cnt, int s) -> uint32_t { return (cnt >> (2 * s)) & 3u; };
  auto cnt_inc = [](uint32_t cnt, int s) -> uint32_t { return (cnt & ~(3u << (2 * s))) | ((((cnt >> (2 * s)) + 1u) & 3u) << (2 * s)); };
  uint8_t* misc = smem + NSTG * STG_BYTES + 8 * NBAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(misc);       // 4 B
  volatile int* peer_T = reinterpret_cast<volatile int*>(misc + 4);                // 1 int: the peer CTA's start step of the current tile (written by the peer)
  volatile int* tile_T = reinterpret_cast<volatile int*>(misc + 8);                // 2 ints
  volatile int* warp_max = reinterpret_cast<volatile int*>(misc + 16);             // 2 x EPI_WARPS ints
  uint8_t* bias_slices = smem + ((NSTG * STG_BYTES + 8 * NBAR + 16 + 8 * EPI_WARPS + 15) & ~15);   // EPI_WARPS x BIAS_SLICE_BYTES, 16-byte aligned
  const uint32_t out_slots = (smem_u32(bias_slices) + EPI_WARPS * BIAS_SLICE_BYTES + 127u) & ~127u;   // EPI_WARPS x OUT_SLOT_BYTES, 128-byte aligned

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const uint32_t leader_rank = cta_rank & ~1u;   // CTA of this tcgen05 pair that issues the UMMAs and owns the barriers
  // Column-split mode (SPLIT): the latency regime -- launches of a handful of row tiles, the reference's own dataset-sized calls
  // (the ml-100k configuration has 7 tiles of 830 columns).  One SM per tile spends a layer's whole N x K on ONE tensor core while
  // 140 SMs idle (and at 830 columns the resident flow does not fit: tile > shared memory, N > 512 TMEM columns).  Here a cluster
  // of S = 2 / 4 / 8 CTAs owns
  // ONE row tile: CTA j computes the N chunks c = j (mod S) of every layer over the full K -- it streams the whole activation image
  // and only its own chunks' weights -- and owns the same columns of the fp32 state, the keep bits and the noise.  Activations
  // still travel through the tile's scratch in the L2 (TMA store -> TMA load), but the chunk barriers now span the cluster: once
  // a warp's TMA stores of a chunk have completed, its lanes 0 .. S-1 arrive on the S peers' copies of the chunk barrier (see
  // relay_chunk; -DSDRM_SPLIT_RELAY=1: through a local barrier and the otherwise idle fourth control warp, which forwards ONE
  // cluster-scope release arrival per chunk -- an epilogue thread's own cluster-scope release would first drain its outstanding
  // fp32 state stores).  The chunk barriers are a ring of two per chunk index (layer parity): a CTA can finish layer l + 1 before a
  // slow peer has consumed layer l's phases, but not layer l + 2 (that needs the peer's chunk of layer l + 1).  The host launches
  // ONE tile per cluster (a second tile's x_T pass would overwrite buffers a slower peer is still decoding from); full- and
  // multi-resolution chains (every CTA of the cluster derives the same start step from the tile's rows).  The last layer of a
  // tile must publish nothing (the decoder's logits layer: sdrm_sample always ends with it).
  constexpr bool SPLIT = SPLITK;
  const uint32_t split_n = SPLIT ? cluster_nctarank() : 1u;
  const uint32_t split_rank = SPLIT ? cluster_ctarank() : 0u;
  // this CTA's chunks of a layer: c = c_first, c_first + c_step, ...  (macros over the special registers, NOT variables: the
  // epilogue's group loops have no register to spare for two more loop invariants; 0 and 1 at compile time without the split)
#define c_first (SPLIT ? static_cast<int>(cluster_ctarank()) : 0)
#define c_step (SPLIT ? static_cast<int>(cluster_nctarank()) : 1)

  if (warp == W_WARP && lane == 0) {
    for (int s = 0; s < NSTG_B; ++s) {
      mbar_init(bar_full(s), 2);     // weight producer + activation producer each arm their own byte count
      mbar_init(bar_empty(s), 1);    // one tcgen05.commit per consumed stage
    }
    mbar_init(bar_acc_full(0), 1);
    mbar_init(bar_acc_full(1), 1);
    mbar_init(bar_acc_empty(0), EPI_WARPS * (PAIR ? 2 : 1));   // the leader's UMMA issuer waits for the epilogue warps of both CTAs
    mbar_init(bar_acc_empty(1), EPI_WARPS * (PAIR ? 2 : 1));
    for (int s = 0; s < MAX_SUB; ++s) {
      for (int c = 0; c < MAX_ACT_CHUNKS; ++c) mbar_init(bar_act_chunk(s, c), (SPLIT && SDRM_SPLIT_RELAY) ? 1 : EPI_WARPS);   // (relayed split publications: one arrival)
      mbar_init(bar_state_ready(s), EPI_WARPS);
      mbar_init(bar_noise_ready(s), NOISE_WARPS);
      for (uint32_t k = 0; k < 2; ++k) {
        mbar_init(bar_layer_consumed(s, k), 1);
        mbar_init(bar_discard_done(s, k), 1);
      }
    }
    mbar_init(bar_tile_ready, EPI_WARPS);
    mbar_init(bar_a_ready, EPI_WARPS);
    mbar_init(bar_peer_ready, 1);
    mbar_init(bar_half_read, 1);
    mbar_init(bar_relay(0), EPI_WARPS);
    mbar_init(bar_relay(1), EPI_WARPS);
    mbar_init(bar_pair_T, 1);
    fence_mbar_init();
  }
  if (warp == M_WARP) {
    if (PAIR) { tmem_alloc_pair(smem_u32(const_cast<uint32_t*>(tmem_slot)), 512); tmem_relinquish_pair(); }
    else { tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 512); tmem_relinquish(); }
  }
  if constexpr (SPLIT) {
    // the tile's activation buffers are shared by the cluster: every CTA zeroes its slice (K-padding columns must read as exact
    // zeros) before ANY CTA may store into them -- the cluster barrier below orders it
    uint4* z = reinterpret_cast<uint4*>(P.scratch + static_cast<size_t>(blockIdx.x / split_n) * P.scratch_stride);
    const size_t n16 = NUM_ACT_BUFS * P.act_buf_bytes / 16;
    for (size_t i = static_cast<size_t>(split_rank) * ENGINE_THREADS + threadIdx.x; i < n16; i += static_cast<size_t>(split_n) * ENGINE_THREADS)
      z[i] = make_uint4(0, 0, 0, 0);
    __threadfence();
    fence_proxy_async();   // read by TMA loads, partly overwritten by TMA stores
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR || SPLIT) cluster_sync_all();   // the peer's barriers exist before anyone commits / arrives remotely
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Resident mode (pair mode, every CTA owns ONE row tile: the dataset-sized configurations, where a layer's latency and not
  // the tensor throughput is what counts).  The chain's activation tile [128 rows x K] never leaves the SM: it lives in the
  // part of the stage ring the weight stream does not use (res_nstg stages stay), as KB k-block images in the UMMA operand
  // layout.  A chain layer accumulates ALL its N <= 512 columns in TMEM (chunk c in accumulator c), and once the layer's last
  // UMMA has retired the epilogue warps overwrite the tile in place with the layer's output (bias / PReLU / posterior update /
  // dropout / bf16) -- no TMA store, no L2 round trip, no chunk barriers: the hand-off is one proxy fence and one mbarrier
  // (the peer CTA's half of the M = 256 operand is signalled through its idle UMMA warp with a cluster-scope release).  The
  // weights still stream from the L2; x_0 goes to the scratch as bf16 hi / lo and the decoder runs as in streaming mode.
  constexpr bool RES = RESK;
  const uint32_t nstg = (RES || SPLIT) ? static_cast<uint32_t>(P.res_nstg) : static_cast<uint32_t>(NSTG);   // (split: stages of split_stage_bytes)
  const uint32_t res_a = base_addr + nstg * STG_BYTES;

  const long long n_tiles = (P.n_rows + TILE_M - 1) / TILE_M;
  const long long n_clusters = SPLIT ? gridDim.x / split_n : gridDim.x / NCTA;
  const long long my_cluster = SPLIT ? blockIdx.x / split_n : blockIdx.x / NCTA;
  // both CTAs of a pair run the same number of tile iterations (a ghost tile past n_tiles has no valid row)
  const int n_local = SPLIT ? static_cast<int>((n_tiles + n_clusters - 1) / n_clusters)
                            : static_cast<int>((n_tiles + gridDim.x - 1) / gridDim.x);   // row tiles of this CTA (split: of this cluster)
  // Sub-tiles: an iteration works on NSUB = P.n_sub (1 or 2) row tiles at once and INTERLEAVES them layer by layer
  // (step i: layer 0 of tile 0, layer 0 of tile 1, layer 1 of tile 0, ...).  A layer's first chunk needs the last chunk
  // of the previous layer of the SAME tile out of its epilogue (stores + proxy fence + TMA round trip: the tensor pipe
  // idled ~3 us of every 21 us layer, 8 us at a step boundary, and through the slow posterior epilogue); with a second,
  // independent tile in between that dependency is a whole layer old when it is needed.  Each sub-tile has its own
  // scratch slot (activation buffers, fp32 state, keep bits) and its own chunk / state / noise barriers; the UMMA
  // issuer and the accumulator hand-off just see a longer chunk sequence.  An odd last tile runs alone (nsub = 1).
  const int NSUB = P.n_sub;
  const int n_iters = (n_local + NSUB - 1) / NSUB;
  auto nsub_of = [&](int it) -> int { return min(NSUB, n_local - it * NSUB); };
  auto tile_of = [&](int it, int s) -> long long {
    return (static_cast<long long>(it * NSUB + s) * n_clusters + my_cluster) * NCTA + cta_rank;
  };
  int* err = P.err_word;
#ifdef SDRM_TRACE
  int trace_n = 0;
  const bool tracing = (P.trace != nullptr) && (blockIdx.x == static_cast<unsigned>(P.debug_flags >> 16)) && (lane == 0 || warp < W_WARP);   // (traced CTA: bits 16+ of the debug flags)
  unsigned long long trace_seq = 0;  // k-block sequence number of the role (for matching producer / consumer events)
  const bool trace_kb = (P.debug_flags & 8) != 0;   // per-k-block events perturb the pipeline; off by default
  auto TR = [&](int role, unsigned long long code) {
    if (tracing && trace_n < TRACE_CAP && (trace_kb || !((role == 0 && (code == 4 || code == 5)) || (role == 1 && code >= 5))))
      P.trace[role * TRACE_CAP + trace_n++] = (code << 56) | ((trace_seq & 0xFFFFull) << 40) | (globaltimer_ns() & 0xFFFFFFFFFFull);
  };
#endif

  auto scratch_of = [&](long long tile, int s) -> uint8_t* {
    const long long idx = P.preloaded_input ? tile : SPLIT ? my_cluster : static_cast<long long>(blockIdx.x) * NSUB + s;
    return P.scratch + static_cast<size_t>(idx) * P.scratch_stride;
  };

  // setmaxnreg sits at the top of each role's own branch: ptxas budgets every program point with the smallest register
  // count that can reach it, so a shared prologue would cap all roles at the control warps' budget
  if (warp == W_WARP || warp == A_WARP) {
    setmaxnreg_dec<REGS_CTRL>();
    // ============================ TMA producers: warp 0 streams weights, warp 2 streams activations =========
    // The whole warp runs the loops CONVERGED and one elected lane issues the copies: single-lane (divergent) code makes
    // the compiler wrap every uniform-datapath instruction (UBLKCP / UTMALDG / UTCHMMA) in an elect loop and costs
    // ~0.5 us per k-block.  The weight stream does not depend on the previous layer's epilogue and runs ahead.
    const bool is_w = (warp == W_WARP);
#ifdef SDRM_TRACE
    const bool tr_me = is_w == ((P.debug_flags & 4096) != 0);   // the traced producer: activations, or (flag 4096) weights
#else
    constexpr bool tr_me = false;
#endif
    const uint64_t pol_keep = l2_policy_evict_last();
    uint32_t stage = 0, sphase = 0, act_par = 0;   // act_par: one parity bit per chunk-index barrier (sub-tile s: bits 8s..8s+7)
    static_assert(MAX_SUB * MAX_ACT_CHUNKS <= 32, "act_par bits");
    for (int it = 0; it < n_iters; ++it) {
      const int ns = nsub_of(it);
      if (!PAIR && tile_of(it, 0) >= n_tiles) break;
      int T_tile = P.T;
      if (!is_w || !PAIR || P.t_start != nullptr) {   // (single mode and multi-resolution pairs: T_tile is per tile / per pair)
        mbar_wait(bar_tile_ready, it & 1, err, WD_PRODUCER_TILE);
        T_tile = tile_T[it & 1];
      }
      // Readiness of a layer's input is tracked per CHUNK of the producing layer (one barrier per chunk index): k-block
      // kb only needs the chunks covering features < 64 (kb + 1), so a layer starts while the previous layer's last
      // chunk is still in its epilogue.
      int prev_nch = 0, prev_nc = 1;
      uint32_t lk = 0;   // layers of this tile so far (split mode: the chunk-barrier ring is indexed by its low bit)
      if (SPLIT) {       // x_T and the first input image are published like a layer's output, in the posterior layer's chunk geometry
        prev_nch = P.step[P.n_step - 1].NCH;
        prev_nc = P.step[P.n_step - 1].NC;
      }
      auto run = [&](const LayerDesc& ldref, const CUtensorMap* tm_w, int in_hi_buf, int in_lo_buf, int s, bool res_layer) {
        const int KB = ldref.KB, NCH = ldref.NCH, NC = ldref.NC, passes = ldref.passes;
        if (res_layer && !is_w) {
          // the activation producer sits a resident chain layer out: it only keeps its ring position in step (it meets the ring
          // again at the decoder's first k-block, after the x_0 pass -- by then every chain UMMA has retired, so its parity
          // cannot alias an older phase)
          const uint32_t pos = stage + static_cast<uint32_t>(NCH * passes * ((KB + 1) >> 1));   // (two weight k-blocks per stage)
          sphase ^= (pos / nstg) & 1u;
          stage = pos % nstg;
          return;
        }
        const uint8_t* w_img = ldref.w_img;
        const uint8_t* sc = scratch_of(tile_of(it, s), s);
        const int a_row_base = static_cast<int>((static_cast<size_t>(sc - P.scratch)) >> 7);
        const uint32_t bset = SPLIT ? (lk & 1u) : static_cast<uint32_t>(s);   // chunk-barrier set: sub-tile, or layer parity (split mode)
        const uint32_t par_shift = bset * MAX_ACT_CHUNKS;
        // The k-block loop of this warp is a serial instruction chain that a split layer's tensor work (0.24 us per k-block) does
        // not hide: no division, no special-register reads in it (the chunk need is tracked as covered features; measured with
        // loads AND UMMAs switched off the loop ran at 0.4 us per k-block with an integer division and an S2R per iteration).
        int ready = 0, covered = 0;   // chunks of the input image waited for so far, and the features they cover
        bool gate = !is_w;            // the first (chunk, pass) this warp streams waits for the input image chunk by chunk
        auto wait_chunks = [&](int lim) {
          while (ready < prev_nch && covered < lim) {
            covered += prev_nc;
            // (split mode: the chunk was written by another CTA's TMA stores, whose completion that CTA has observed (bulk wait_group)
            // before it arrived here: the bytes are in the L2, and the only reader is this warp's TMA load, which reads
            // the L2 directly -- no cache of this SM is involved.  A cluster-scope acquire costs ~1 us per wait, as a fence behind the
            // wait (fence.acq_rel.cluster) and as a qualifier on it (try_wait.acquire.cluster) alike: 8 of them were 60 % of a layer.)
#ifdef SDRM_SPLIT_ACQUIRE_CLUSTER
            mbar_wait<SPLIT>(bar_act_chunk(bset, ready), (act_par >> (par_shift + ready)) & 1u, err, WD_PRODUCER_ACT);
#else
            mbar_wait(bar_act_chunk(bset, ready), (act_par >> (par_shift + ready)) & 1u, err, WD_PRODUCER_ACT);
#endif
            act_par ^= (1u << (par_shift + ready));
            ++ready;
            if (SPLIT) SDRM_TR(0, 6);
          }
        };
        if (tr_me) SDRM_TR(0, 1);
        const uint32_t w_bytes = static_cast<uint32_t>(NC) * 128u;          // one whole weight k-block image
        const int half_rows = NC >> 1;
        for (int c = c_first; c < NCH; c += c_step) {   // (split mode: this CTA's chunks; otherwise all)
          for (int p = 0; p < passes; ++p) {
            const int which = (p == 1) ? 1 : 0;
            const int a_buf = (p == 2) ? in_lo_buf : in_hi_buf;
            const uint8_t* a_src = sc + static_cast<size_t>(a_buf) * P.act_buf_bytes;
            const uint8_t* w_src = w_img + (static_cast<size_t>(which) * NCH + c) * KB * w_bytes;
            int w_row = ((which * NCH + c) * KB) * NC + static_cast<int>(cta_rank & 1u) * half_rows;
            int a_row = a_row_base + static_cast<int>((static_cast<size_t>(a_buf) * P.act_buf_bytes) >> 7);
            // resident chain layers: a stage has no activation half to fill, so it carries TWO weight k-blocks (the second in the
            // activation half): twice the weight bytes in flight -- this mode is bound by the L2 latency of the weight stream
            const int kstep = res_layer ? 2 : 1;
            for (int kb = 0; kb < KB; kb += kstep) {
              if (gate) {
                int lim = (kb == KB - 1) ? 0x7fffffff : (kb + 1) * KBLK;   // k-block kb needs the chunks covering features < 64 (kb + 1)
#ifdef SDRM_PERF_DEBUG
                if (P.debug_flags & 1024) lim = 0x7fffffff;   // (experiment: wait for the whole input image before the first k-block)
#endif
                wait_chunks(lim);
                if (kb == 0) SDRM_TR(0, 2);
              }
              mbar_wait(bar_empty(stage), sphase ^ 1, err, WD_PRODUCER_EMPTY);
              const uint32_t fb = bar_full(stage);
              if (elect_one()) {
                if (PAIR) {
                  // both CTAs load into their own stage but complete on the LEADER's full barrier; the leader's two
                  // producers arm it with the bytes of both CTAs
                  const uint32_t fb0 = mapa_cluster(fb, leader_rank);
                  if (is_w) {
                    const bool two = res_layer && kb + 1 < KB;
                    if (cta_rank == leader_rank) {
                      mbar_arrive_expect_tx(fb, two ? 2u * w_bytes : w_bytes);
                      if (res_layer) mbar_arrive(fb);   // resident chain layer: no activation load takes the stage's second arrival
                    }
                    if (res_layer) {
                      tma_load_2d_pair_hint(mapa_cluster(stage_a(stage), cta_rank), tm_w, 0, w_row, fb0, pol_keep);
                      if (two) tma_load_2d_pair_hint(mapa_cluster(stage_w(stage), cta_rank), tm_w, 0, w_row + NC, fb0, pol_keep);
                    } else {
                      tma_load_2d_pair_hint(mapa_cluster(stage_w(stage), cta_rank), tm_w, 0, w_row, fb0, pol_keep);
                    }
                  } else {
                    if (cta_rank == leader_rank) mbar_arrive_expect_tx(fb, 2 * A_TILE_BYTES);
                    tma_load_2d_pair_hint(mapa_cluster(stage_a(stage), cta_rank), &P.tm_act, 0, a_row, fb0, pol_keep);
                  }
                } else if (is_w) {
                  if (SDRM_DEBUG_SKIP_W_LOADS) mbar_arrive(fb);
                  else {
                    mbar_arrive_expect_tx(fb, w_bytes);
                    bulk_g2s_hint(stage_w(stage), w_src, w_bytes, fb, pol_keep);
                  }
                } else {
                  if (SDRM_DEBUG_SKIP_A_LOADS) mbar_arrive(fb);
                  else {
                    mbar_arrive_expect_tx(fb, A_TILE_BYTES);
                    tma_load_2d_hint(stage_a(stage), &P.tm_act, 0, a_row, fb, pol_keep);
                  }
                }
              }
              __syncwarp();
              w_row += NC * kstep;
              a_row += A_TILE_BYTES >> 7;
              w_src += w_bytes;
              a_src += A_TILE_BYTES;
              if (tr_me) { SDRM_TR(0, 5); SDRM_TR_SEQ(); }
              if (++stage == nstg) { stage = 0; sphase ^= 1; }
            }
            gate = false;
          }
          if (tr_me) SDRM_TR(0, 3);
        }
        if (SPLIT && !is_w) wait_chunks(0x7fffffff);   // a CTA without a chunk in this layer still consumes the phases
      };
      // the layer whose output the NEXT layer of the same tile reads (all sub-tiles go through the same layer sequence)
      auto done = [&](const LayerDesc& ldref) {
        prev_nch = (ldref.kind == EPI_LINEAR_OUT) ? 0 : ldref.NCH;
        prev_nc = ldref.NC;
        ++lk;
      };
      // chain layers ping-pong between activation buffers 0 and 1 (in = parity of the layer count so far); only two
      // hot buffers per tile keep the scratch L2-resident.  The decoder reads x0 hi from the chain's last buffer.
      int cur = 0;
      for (int i = T_tile; i >= 1; --i)
        for (int l = 0; l < P.n_step; ++l) {
          for (int s = 0; s < ns; ++s) run(P.step[l], &P.tm_step_w[l], cur, cur, s, RES);
          done(P.step[l]);
          cur ^= 1;
        }
      for (int l = 0; l < P.n_dec; ++l) {
        for (int s = 0; s < ns; ++s) run(P.dec[l], &P.tm_dec_w[l], P.dec[l].in_hi == 0 ? cur : cur ^ 1, P.dec[l].in_lo, s, false);
        done(P.dec[l]);
      }
    }
  } else if (warp == M_WARP) {
    setmaxnreg_dec<REGS_CTRL>();
    if (PAIR && cta_rank != leader_rank) {
      // peer CTA of a pair: the leader issues every UMMA; the peer's TMA loads complete on the leader's barriers
      if (RES) {
        // resident mode: relay "this CTA's half of the next layer's input tile is written" to the leader.  The epilogue warps
        // arrive on the local barrier (CTA-scope release behind their proxy fence); this thread has no memory operation of its
        // own in flight, so its cluster-scope release costs nothing (an epilogue thread's would wait for its state stores).
        const uint32_t remote = mapa_cluster(bar_peer_ready, leader_rank);
        const int n_layers = n_iters * P.T * P.n_step;   // (both CTAs of a pair run the same number of tile iterations)
        for (int k = 0; k < n_layers; ++k) {
          mbar_wait(bar_a_ready, static_cast<uint32_t>(k) & 1u, err, WD_RELAY);
#if SDRM_RES_CLUSTER_SCOPE
          if (elect_one()) mbar_arrive_cluster_release(remote);
#else
          if (elect_one()) mbar_arrive_cluster(remote);
#endif
          __syncwarp();
        }
      }
    } else {
      // ======================================= UMMA issuer ========================================
      // whole warp converged, one elected lane issues (see the producer comment)
      uint32_t stage = 0, sphase = 0, cc = 0, lc_cnt = 0, a_par = 0;
      for (int it = 0; it < n_iters; ++it) {
        if (!PAIR && tile_of(it, 0) >= n_tiles) break;
        const int ns = nsub_of(it);
        int T_tile = P.T;   // (multi-resolution pairs: both row tiles run the longer of their two chains, see the epilogue warps)
        if (!PAIR || P.t_start != nullptr) {
          mbar_wait(bar_tile_ready, it & 1, err, WD_MMA_TILE);
          T_tile = tile_T[it & 1];
        }
        auto run = [&](const LayerDesc& ldref, int s, bool chain) {
          const int KB = ldref.KB, NCH = ldref.NCH, passes = ldref.passes, kmma_last = ldref.kmma_last;
          const uint32_t idesc = umma_idesc_bf16(PAIR ? 256 : 128, ldref.NC);
          const bool res_layer = RES && chain;
          const int half_kb = (ldref.NC - 1) >> 6;   // last k-block under the first chunk's output columns
          if (res_layer) {
            // both halves of the M = 256 input tile are in place (and the previous layer's accumulators have been read)
            mbar_wait(bar_a_ready, a_par, err, WD_MMA_AREADY);
            mbar_wait(bar_peer_ready, a_par, err, WD_MMA_PEER);
            a_par ^= 1u;
#if SDRM_RES_CLUSTER_SCOPE
            fence_acq_rel_cluster();
#endif
            tc_fence_after();
            SDRM_TR(1, 7);
          }
          for (int c = c_first; c < NCH; c += c_step) {
            const uint32_t buf = cc & 1u;
            SDRM_TR(1, 1);
            mbar_wait(bar_acc_empty(buf), ((cc >> 1) & 1u) ^ 1u, err, WD_MMA_ACC);
            tc_fence_after();
            SDRM_TR(1, 2);
            const uint32_t d_tmem = tmem_base + buf * 256u;
            uint32_t acc = 0;
            for (int p = 0; p < passes; ++p) {
              for (int kb = 0; kb < KB; kb += (res_layer ? 2 : 1)) {
                mbar_wait(bar_full(stage), sphase, err, WD_MMA_FULL);
                tc_fence_after();
                SDRM_TR(1, kb == 0 && p == 0 ? 3 : 5);
                const uint64_t a_desc = umma_desc_sw128(res_layer ? res_a + static_cast<uint32_t>(kb) * A_TILE_BYTES : stage_a(stage));
                const uint64_t b_desc = umma_desc_sw128(res_layer ? stage_a(stage) : stage_w(stage));
                const int nk = (kb == KB - 1) ? kmma_last : 4;
                if (elect_one()) {
                  // +32 B (16 bf16) along K inside the swizzle row = +2 in the 16-byte address field
                  if (PAIR && res_layer && kb + 1 < KB) {
                    // resident chain layer: the stage holds two weight k-blocks (see the producer)
                    const uint64_t a2 = umma_desc_sw128(res_a + static_cast<uint32_t>(kb + 1) * A_TILE_BYTES);
                    const uint64_t b2 = umma_desc_sw128(stage_w(stage));
                    const int nk2 = (kb + 1 == KB - 1) ? kmma_last : 4;
                    umma_bf16_ss_pair(d_tmem, a_desc, b_desc, idesc, acc);
                    umma_bf16_ss_pair(d_tmem, a_desc + 2u, b_desc + 2u, idesc, 1u);
                    umma_bf16_ss_pair(d_tmem, a_desc + 4u, b_desc + 4u, idesc, 1u);
                    umma_bf16_ss_pair(d_tmem, a_desc + 6u, b_desc + 6u, idesc, 1u);
                    umma_bf16_ss_pair(d_tmem, a2, b2, idesc, 1u);
                    if (nk2 > 1) umma_bf16_ss_pair(d_tmem, a2 + 2u, b2 + 2u, idesc, 1u);
                    if (nk2 > 2) umma_bf16_ss_pair(d_tmem, a2 + 4u, b2 + 4u, idesc, 1u);
                    if (nk2 > 3) umma_bf16_ss_pair(d_tmem, a2 + 6u, b2 + 6u, idesc, 1u);
                    umma_commit_pair(bar_empty(stage), static_cast<uint16_t>((1u << CS) - 1u));
                    // two-chunk layer, second chunk: once the k-blocks under the first chunk's output columns have been read
                    // (by BOTH chunks: a commit covers every earlier UMMA) the epilogue may overwrite them -- the first chunk's
                    // epilogue then runs in the shadow of the rest of this chunk
                    if (NCH == 2 && c == 1 && kb <= half_kb && half_kb <= kb + 1)
                      umma_commit_pair(bar_half_read, static_cast<uint16_t>(0x3u << leader_rank));
                  } else if (PAIR) {
                    umma_bf16_ss_pair(d_tmem, a_desc, b_desc, idesc, acc);
                    if (nk > 1) umma_bf16_ss_pair(d_tmem, a_desc + 2u, b_desc + 2u, idesc, 1u);
                    if (nk > 2) umma_bf16_ss_pair(d_tmem, a_desc + 4u, b_desc + 4u, idesc, 1u);
                    if (nk > 3) umma_bf16_ss_pair(d_tmem, a_desc + 6u, b_desc + 6u, idesc, 1u);
                    umma_commit_pair(bar_empty(stage), static_cast<uint16_t>((1u << CS) - 1u));   // every CTA of the cluster
                  } else {
#ifdef SDRM_PERF_DEBUG
                    if (!(P.debug_flags & 2048))   // (experiment: no UMMAs, only the commits -- the pace of the barrier machinery alone)
#endif
                    {
                    umma_bf16_ss(d_tmem, a_desc, b_desc, idesc, acc);
                    if (nk > 1) umma_bf16_ss(d_tmem, a_desc + 2u, b_desc + 2u, idesc, 1u);
                    if (nk > 2) umma_bf16_ss(d_tmem, a_desc + 4u, b_desc + 4u, idesc, 1u);
                    if (nk > 3) umma_bf16_ss(d_tmem, a_desc + 6u, b_desc + 6u, idesc, 1u);
                    }
                    umma_commit(bar_empty(stage));
                  }
                }
                __syncwarp();
                acc = 1;
                SDRM_TR(1, 6);
                SDRM_TR_SEQ();
                if (++stage == nstg) { stage = 0; sphase ^= 1; }
              }
            }
            if (elect_one()) {
              if (PAIR) umma_commit_pair(bar_acc_full(buf), static_cast<uint16_t>(0x3u << leader_rank));
              else umma_commit(bar_acc_full(buf));
            }
            __syncwarp();
            SDRM_TR(1, 4);
            ++cc;
          }
          if (PAIR && chain && P.discard_kb > 0) {
            // every UMMA of this layer has retired when this arrives: the layer's input image is dead
            if (elect_one()) umma_commit_pair(bar_layer_consumed(s, cnt_get(lc_cnt, s)), static_cast<uint16_t>(0x3u << leader_rank));
            __syncwarp();
            lc_cnt = cnt_inc(lc_cnt, s);
          }
        };
        for (int i = T_tile; i >= 1; --i)
          for (int l = 0; l < P.n_step; ++l)
            for (int s = 0; s < ns; ++s) run(P.step[l], s, true);
        for (int l = 0; l < P.n_dec; ++l)
          for (int s = 0; s < ns; ++s) run(P.dec[l], s, false);
      }
    }
  } else if (warp > A_WARP) {
    setmaxnreg_dec<REGS_CTRL>();
    // ======================================= discard warp (fourth control warp) =================================
    // A chain layer's input image is dead once the layer's last UMMA has read it, but its lines are DIRTY in the L2 and, with
    // 148 x 0.98 MB of scratch against ~60 MB of effective L2, they are written back to HBM before the layer after next
    // overwrites them: 1.47 MB of DRAM writes per CTA and step for data nobody will read (ncu: 93 % of all bytes the kernel
    // writes reach DRAM).  discard.global.L2 drops such lines without a write-back (tools/ubench_discard.cu: 15.4 GB -> 0.5 GB of
    // DRAM writes).  Only whole k-blocks that the next writer rewrites completely are discarded (discard_kb), so the zero
    // padding columns written once at kernel start survive.
    if constexpr (SPLIT && SDRM_SPLIT_RELAY) {
      // ===================================== relay warp (column-split mode, -DSDRM_SPLIT_RELAY=1) ================
      // forwards "chunk c of the layer's output is complete in the L2" from this CTA's epilogue warps to the chunk barrier of
      // every CTA of the cluster, lane j -> CTA j, with a cluster-scope release (this warp has no memory operation in flight)
      uint32_t rk = 0;
      auto forward = [&](uint32_t bset, int c) {
        mbar_wait(bar_relay(rk), (rk >> 1) & 1u, err, WD_RELAY);
        ++rk;
        if (lane < static_cast<int>(split_n)) mbar_arrive_cluster_release(mapa_cluster(bar_act_chunk(bset, static_cast<uint32_t>(c)), static_cast<uint32_t>(lane)));
        __syncwarp();
      };
      for (int it = 0; it < n_iters; ++it) {
        if (tile_of(it, 0) >= n_tiles) break;
        uint32_t lk = 0;
        const LayerDesc& lo = P.step[P.n_step - 1];
        for (int c = c_first; c < lo.NCH; c += c_step) forward(0u, c);   // x_T and the first input image
        for (int i = P.T; i >= 1; --i)
          for (int l = 0; l < P.n_step; ++l) {
            ++lk;
            for (int c = c_first; c < P.step[l].NCH; c += c_step) forward(lk & 1u, c);
          }
        for (int l = 0; l < P.n_dec; ++l) {
          ++lk;
          if (P.dec[l].kind != EPI_LINEAR_OUT && l != P.n_dec - 1)
            for (int c = c_first; c < P.dec[l].NCH; c += c_step) forward(lk & 1u, c);
        }
      }
    }
    if (PAIR && P.discard_kb > 0) {
      uint32_t dcnt = 0;   // layer counters of the sub-tiles
      const int n_lines = P.discard_kb * (A_TILE_BYTES / 128);
      for (int it = 0; it < n_iters; ++it) {
        const int ns = nsub_of(it);
        int cur = 0;
        for (int i = P.T; i >= 1; --i)
          for (int l = 0; l < P.n_step; ++l) {
            for (int s = 0; s < ns; ++s) {
              const uint32_t k = cnt_get(dcnt, s);
              dcnt = cnt_inc(dcnt, s);
              mbar_wait(bar_layer_consumed(s, k), (k >> 1) & 1u, err, WD_DISCARD);
              if (!(i == 1 && l == P.n_step - 1)) {   // (the last chain layer's neighbours are the decoder's buffers: left alone)
                uint8_t* dead = scratch_of(tile_of(it, s), s) + static_cast<size_t>(cur) * P.act_buf_bytes;
#ifndef SDRM_DISCARD_DRY   // (debug builds: the barrier protocol without the discards)
                for (int j = lane; j < n_lines; j += 32)
                  asm volatile("discard.global.L2 [%0], 128;" ::"l"(dead + static_cast<size_t>(j) * 128) : "memory");
#endif
#ifndef SDRM_DISCARD_NOFENCE   // (perf experiment)
                fence_proxy_async();   // the next writes to these lines are TMA stores (async proxy)
#endif
              }
              __syncwarp();
              if (lane == 0) mbar_arrive(bar_discard_done(s, k));
            }
            cur ^= 1;
          }
      }
    }
  } else if (warp < EPI_WARPS) {
    // ======================================= epilogue warps =====================================
    // 16 warps: warp (q, sub) reads TMEM lane quarter q (rows 32q..32q+31) and owns the 16-column groups
    // g = sub (mod 4).  One thread always touches the same (row, columns) of the fp32 state, so the state
    // needs no synchronisation at all.  The SM's issue slots, not the tensor pipe, bound this kernel (ncu: ~150 k warp
    // instructions per step and SM sub-partition against 173 k cycles of UMMA time), so the per-group code is specialised
    // per layer kind, runs on packed f32x2 arithmetic and keeps every loop-invariant out of the loop.
    setmaxnreg_inc<REGS_EPI>();
    const uint64_t pol_keep = l2_policy_evict_last();
    const int q = warp & 3;
    int sub = warp >> 2;
    const int r = q * 32 + lane;
    uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    uint32_t lane0 = (lane == 0) ? 1u : 0u;
    pin_reg(lane0); pin_reg(lane_addr);
    const uint32_t row_off = static_cast<uint32_t>(r) * 128u;
    float* bias_s = reinterpret_cast<float*>(bias_slices + warp * BIAS_SLICE_BYTES);   // this warp's private bias slice
    uint32_t cc = 0;
    int it = 0;

    // Write 16 consecutive bf16 features [f0, f0+16) of the warp's 32 rows into a k-block image: the lanes drop their 32 bytes
    // into the warp's dense shared-memory slot and lane 0 hands the 32 x 32-byte box to the TMA (tensor-map store into the
    // linear activation image; the TMA LOAD swizzles it into the UMMA operand layout).  Against 256-bit global stores
    // scattered over 32 rows this frees the source registers at once (the next iteration's loads waited for the LSU to dequeue
    // the store: 27 % of the PReLU loop's samples), needs no swizzle shuffles, and the writes stay in the async proxy, so
    // publishing a chunk is a bulk-group wait of one lane instead of a membar.gpu + proxy fence of every thread.
    // Two slots per warp, and the TMA store of a slot is issued one call LATER (right before the other slot is filled): by then
    // the slot's st.shared are long complete, so the proxy fence does not wait for them, and the slot about to be overwritten
    // was handed to the TMA a whole group iteration ago, so waiting for its read costs nothing either.  (r01f profile, PReLU
    // group loop: 12.9 % of its samples waited for the previous box to be read, 13.2 % on the fence behind the stores.)
    const uint32_t out_slot = out_slots + static_cast<uint32_t>(warp) * (OUT_SLOTS_PER_WARP * OUT_SLOT_BYTES);
    const uint32_t out_lane = out_slot + static_cast<uint32_t>(lane) * 32u;
    uint32_t slot_sel = 0;     // slot written last
    int pend_x = -1, pend_y = 0;   // tensor coordinates of the box waiting in slot `slot_sel` (pend_x < 0: none)
    auto flush_pending = [&]() {
      if (pend_x >= 0) {   // warp-uniform
        fence_proxy_async_smem();
        __syncwarp();
        // (elect.sync with a full mask always names the same lane; converged single-lane issue keeps ptxas from wrapping the
        // uniform-datapath TMA instruction in an elect loop)
        if (elect_one()) {
          tma_store_2d_hint(&P.tm_act_st, pend_x, pend_y, out_slot + slot_sel * OUT_SLOT_BYTES, pol_keep);
          bulk_commit_group();
        }
        pend_x = -1;
      }
    };
    auto store_act = [&](uint8_t* buf_row, int f0, const uint32_t (&pk)[8]) {
      flush_pending();
      if (OUT_SLOTS_PER_WARP == 1) {
        if (elect_one()) bulk_wait_group_read<0>();   // the box has been read out of the slot
      } else {
        if (elect_one()) bulk_wait_group_read<1>();   // every box but the one just issued has been read: the other slot is free
        slot_sel ^= 1u;
      }
      __syncwarp();
      const uint32_t dst = out_lane + slot_sel * OUT_SLOT_BYTES;
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + 16u), "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7]) : "memory");
      // first row of the box = row 32 q of the tile (lane 0's buf_row)
      pend_y = __shfl_sync(0xffffffffu, static_cast<int>((buf_row - P.scratch) >> 7), 0) + (f0 >> 6) * TILE_M;
      if (SDRM_DEBUG_ACT_STORE_FIXED) pend_y = static_cast<int>((static_cast<size_t>(blockIdx.x) * P.scratch_stride) >> 7) + 32 * q;
      pend_x = (f0 & 63) * 2;
      if (OUT_SLOTS_PER_WARP == 1) flush_pending();
    };
    // resident mode: the same 16 features go straight into the shared-memory operand tile (k-block f0 / 64, row r, the two
    // 16-byte chunks of the 128-byte row XOR-swizzled with r % 8 exactly as a SWIZZLE_128B tensor load would place them)
    const uint32_t res_row = res_a + static_cast<uint32_t>(r) * 128u;
    const uint32_t res_xor = static_cast<uint32_t>(r & 7);
    auto store_res = [&](int f0, const uint32_t (&pk)[8]) {
      const uint32_t blk = res_row + static_cast<uint32_t>(f0 >> 6) * A_TILE_BYTES;
      const uint32_t j = static_cast<uint32_t>(f0 & 63) >> 3;
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(blk + ((j ^ res_xor) << 4)), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(blk + (((j + 1u) ^ res_xor) << 4)), "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7]) : "memory");
    };
    // this warp's part of the resident tile is written: visible to the tensor core (async proxy), then one arrival per warp
    auto res_publish = [&]() {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane0) mbar_arrive(bar_a_ready);
    };
    // all TMA stores of this warp have been written (lane 0 issued them): what a chunk / tile publication waits for
    auto stores_done = [&]() {
      flush_pending();
      if (!SDRM_DEBUG_NO_STORE_WAIT) {
        if (elect_one()) bulk_wait_group<0>();
      }
      __syncwarp();
    };
    // dropout (F.dropout p = .5: kept values are doubled) + bf16 pack of 16 state values
    auto dropout_pack = [&](const float (&x)[16], uint32_t keep, uint32_t (&pk)[8]) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        // 2.0f = 0x40000000: the keep bit moved to bit 30 IS the scale factor (0 or 2)
        const float s0 = __uint_as_float((keep << (30 - 2 * e)) & 0x40000000u);
        const float s1 = __uint_as_float((keep << (29 - 2 * e)) & 0x40000000u);
        const float2 m = __fmul2_rn(make_float2(x[2 * e], x[2 * e + 1]), make_float2(s0, s1));
        pk[e] = pack_bf16x2(m.x, m.y);
      }
    };

    // zero the activation buffers once: K-padding columns must read as exact zeros (split mode: done by the whole cluster above)
    if (!SPLIT && !P.preloaded_input) {
      for (int s = 0; s < NSUB; ++s) {
        uint4* z = reinterpret_cast<uint4*>(scratch_of(0, s));
        const size_t n16 = NUM_ACT_BUFS * P.act_buf_bytes / 16;
        for (size_t i = threadIdx.x; i < n16; i += EPI_THREADS) z[i] = make_uint4(0, 0, 0, 0);
      }
      epi_bar_sync();
    }
    if constexpr (RES) {   // K-padding columns of the resident tile must read as exact zeros too
      const uint32_t n16 = (static_cast<uint32_t>(NSTG) - nstg) * STG_BYTES / 16u;
      for (uint32_t i = threadIdx.x; i < n16; i += EPI_THREADS)
        asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(res_a + i * 16u), "r"(0u) : "memory");
      epi_bar_sync();
    }
    // Lazy publication (two interleaved sub-tiles only): waiting for a chunk's TMA stores to complete right behind them costs the
    // epilogue warps ~1.5 us per chunk (the round trip of bulk_wait_group), as much as the chunk's arithmetic.  With a second tile
    // in between, the consumer of a chunk (the same tile's next layer) is a whole tile-layer away, so the chunk is only NOTED here
    // and published at the start of the next chunk epilogue, when its stores have long completed.  (With one tile the next
    // accumulator cannot become ready before the publication: prompt publication there.)
    uint32_t pub_pend = 0;    // bit 8 s + c: chunk c of sub-tile s has been stored but not published
    static_assert(MAX_SUB * MAX_ACT_CHUNKS <= 32 && MAX_ACT_CHUNKS == 8, "pub_pend bits");
    auto publish_pending = [&]() {
      if (pub_pend) {   // warp-uniform
        stores_done();
        if (lane0)
          for (uint32_t m = pub_pend; m; m &= m - 1u) {
            const uint32_t b = static_cast<uint32_t>(__ffs(m)) - 1u;
            mbar_arrive(bar_act_chunk(b >> 3, b & 7u));
          }
        pub_pend = 0;
      }
    };
    // Split mode: publish own chunk c of the layer's output to every CTA of the cluster.  This warp's TMA stores of the chunk have
    // completed (stores_done() first: lane 0 has waited for its bulk group, the __syncwarp behind it orders the other lanes), i.e. the
    // bytes are in the L2, and the only readers are the peers' TMA loads, which read the L2 directly -- so lane j arrives on CTA j's
    // chunk barrier with the default (CTA-scope) release, like every cross-CTA "slot is free" signal of a TMA pipeline.  The
    // cluster-scope release (through the relay warp, -DSDRM_SPLIT_RELAY=1) costs 0.5 us per layer and changes no result.
    uint32_t rk = 0;          // relay build: chunks handed to the relay warp so far; default: layers of this tile so far (chunk-barrier set)
    auto relay_chunk = [&](int c) {
      if (SDRM_SPLIT_RELAY) {
        if (lane0) mbar_arrive(bar_relay(rk));
        ++rk;
      } else {
        if (lane < static_cast<int>(cluster_nctarank()))
          mbar_arrive_cluster(mapa_cluster(bar_act_chunk(rk & 1u, static_cast<uint32_t>(c)), static_cast<uint32_t>(lane)));
      }
    };
    uint32_t half_par = 0;    // parity of bar_half_read (resident mode, two-chunk layers)
    uint32_t noise_par = 0;   // bit s: parity of sub-tile s's noise_ready barrier
    uint32_t dd_cnt = 0;      // discard_done phases consumed per sub-tile (two bits each)
    // context of the sub-tile a layer works on (set_ctx): scratch pointers are recomputed, the row facts are kept per sub-tile
    uint8_t* sc = nullptr;
    float* xs = nullptr;
    const uint16_t* mask_row = nullptr;
    bool valid = false;
    long long row = 0;
    int t_row = 0;
    for (; it < n_iters; ++it) {
      if (!PAIR && tile_of(it, 0) >= n_tiles) break;
      const int ns = nsub_of(it);
      if (SPLIT && !SDRM_SPLIT_RELAY) rk = 0;   // (the producers' layer count restarts with every tile)
      auto set_ctx = [&](int s) {
        sc = scratch_of(tile_of(it, s), s);
        xs = reinterpret_cast<float*>(sc + NUM_ACT_BUFS * P.act_buf_bytes);
        mask_row = reinterpret_cast<const uint16_t*>(sc + P.mask_off + static_cast<size_t>(r) * P.mask_pitch);
        // row facts are recomputed per layer (a handful of instructions, two cached loads in multi-resolution mode) rather
        // than kept per sub-tile: the group loops have no register to spare
        const long long prow = tile_of(it, s) * TILE_M + r;   // physical row of this launch
        valid = prow < P.n_rows;
        row = (valid && P.row_ids) ? static_cast<long long>(P.row_ids[prow]) : prow;  // logical row
        t_row = P.T;
        if (P.t_start) t_row = valid ? min(max(P.t_start[prow], 0), P.T) : 0;   // clamped: an out-of-range entry must not index bias0 / coef out of bounds
      };

      // ---- row facts of every sub-tile; tile start step = max over rows (and sub-tiles)
      int m = 0;
      for (int s = 0; s < ns; ++s) {
        set_ctx(s);
        m = max(m, t_row);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
      if (lane == 0) warp_max[(it & 1) * EPI_WARPS + warp] = m;
      epi_bar_sync();
      int T_tile = 0;
#pragma unroll
      for (int w = 0; w < EPI_WARPS; ++w) T_tile = max(T_tile, warp_max[(it & 1) * EPI_WARPS + w]);
      if (P.n_step == 0) T_tile = 0;
      if (PAIR && P.t_start != nullptr) {
        // Multi-resolution chains on a CTA pair: the UMMAs of the two row tiles are one instruction stream, so both tiles run
        // max(T_a, T_b) steps -- rows whose own chain is shorter stay inactive until their start step, exactly like the
        // shorter rows inside one tile (the public call sorts the rows by chain length, so neighbouring tiles differ little).
        // Once per tile: thread 0 drops its tile's start step into the peer's shared memory and arrives on the peer's barrier
        // with a cluster-scope release; everybody acquires the own barrier and takes the maximum.
        if (warp == 0 && lane == 0) {
          const uint32_t peer = cta_rank ^ 1u;
          asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(mapa_cluster(smem_u32(const_cast<int*>(peer_T)), peer)), "r"(T_tile) : "memory");
          mbar_arrive_cluster_release(mapa_cluster(bar_pair_T, peer));
        }
        mbar_wait<true>(bar_pair_T, static_cast<uint32_t>(it) & 1u, err, WD_EPI_LAYER);
        T_tile = max(T_tile, *peer_T);
      }

      // ---- x_T and the first denoiser input (train_SDRM.py:51 / 38).  Once per tile: not performance critical.
      if (P.n_step > 0) {
        const PhiloxKeys K = philox_make_keys(P.seed);
        for (int s = 0; s < ns; ++s) {
          set_ctx(s);
          const unsigned long long grow = static_cast<unsigned long long>(P.row_offset + row);
          uint8_t* in0_row = sc + row_off;   // the first chain layer reads activation buffer 0
          // (split mode: only the columns of this CTA's chunks of the posterior layer -- the state columns it owns for the whole chain)
          const int xg_per = SPLIT ? (P.step[P.n_step - 1].NC >> 4) : P.Lg16;
          const int xg_blocks = SPLIT ? P.step[P.n_step - 1].NCH : 1;
          for (int cb = c_first; cb < xg_blocks; cb += c_step)
          for (int gg = sub; gg < xg_per; gg += EPI_SUB) {
            const int g = cb * xg_per + gg;
            if (g >= P.Lg16) break;
            float x[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float z4[4];
              if (P.inj_xT) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int f = g * 16 + j * 4 + e;
                  z4[e] = (valid && f < P.L) ? P.inj_xT[static_cast<size_t>(row) * P.L + f] : 0.0f;
                }
              } else {
                philox_normal4_keys(K, STREAM_NORMAL, grow, 0u, static_cast<uint32_t>(g * 4 + j), z4);
              }
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int f = g * 16 + j * 4 + e;
                x[j * 4 + e] = (valid && f < P.L) ? z4[e] : 0.0f;   // padding columns / rows stay exactly 0 for the whole chain
              }
            }
            xs_store16(xs, g, r, x);
            if (T_tile == 0) {
              // no reverse step in this tile (every row starts at t = 0): x_0 = x_T.  What the x_0 pass of the last posterior
              // step would leave for the decoder: bf16 hi image in buffer 0 (the chain's last output when it ran no layer), lo
              // image in buffer 2, and x0_out.  (T_tile is uniform over the CTA: the warp-collective stores stay converged.)
              uint32_t ph[8], pl[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const float h0 = bf16_round(x[2 * e]), h1 = bf16_round(x[2 * e + 1]);
                ph[e] = pack_bf16x2(h0, h1);
                pl[e] = pack_bf16x2(x[2 * e] - h0, x[2 * e + 1] - h1);
              }
              store_act(in0_row, g * 16, ph);
              store_act(sc + 2 * P.act_buf_bytes + row_off, g * 16, pl);
              if (P.x0_out && valid) {
#pragma unroll
                for (int e = 0; e < 16; ++e)
                  if (g * 16 + e < P.L) P.x0_out[static_cast<size_t>(row) * P.L + g * 16 + e] = x[e];
              }
              continue;
            }
            // keep mask of the first step (the noise warps produce the masks of all later steps)
            uint32_t keep = 0;
            if (valid) {
              if (P.inj_mask) {
                const uint8_t* mp = P.inj_mask + (static_cast<size_t>(T_tile) * P.n_rows + row) * P.L;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                  const int f = g * 16 + e;
                  if (f < P.L && mp[f]) keep |= (1u << e);
                }
              } else {
                const u32x4 w4 = philox_mask128(K, STREAM_MASK, grow, static_cast<uint32_t>(T_tile), static_cast<uint32_t>(g >> 3));
                const uint32_t wsel = ((g >> 1) & 3) == 0 ? w4.x : ((g >> 1) & 3) == 1 ? w4.y : ((g >> 1) & 3) == 2 ? w4.z : w4.w;
                keep = (wsel >> (16 * (g & 1))) & 0xFFFFu;
              }
            }
            uint32_t pk[8];
            dropout_pack(x, keep, pk);
            if (RES) store_res(g * 16, pk);
            else store_act(in0_row, g * 16, pk);
          }
        }
      }
      if (warp == 0 && lane == 0) tile_T[it & 1] = T_tile;
      fence_proxy_async();   // the zero fill of the buffers (generic stores) is read by the TMA loads too
      stores_done();
      if (lane == 0) mbar_arrive(bar_tile_ready);
      if (SPLIT)
        for (int c = c_first; c < P.step[P.n_step - 1].NCH; c += c_step) relay_chunk(c);   // the first input image: "layer 0" of the chunk-barrier ring
      if (RES && P.n_step > 0) res_publish();   // the first chain layer's input tile

      // ---- layers: one instantiation per epilogue kind so that the group loop carries no dispatch
      auto run = [&](auto kind_c, const LayerDesc& ld, int step, bool last_of_tile, int out_hi_buf, int out_lo_buf, int s) {
        constexpr int KIND = decltype(kind_c)::value;
        // The LAST reverse step hands x_0 to the decoder as bf16 hi/lo images (and to x0_out).  That conversion runs as a
        // separate pass over the finished fp32 state after the layer (once per tile), NOT inside the group loop: with both
        // paths in the loop ptxas spilled loop invariants, and a spill reload issued behind the state loads of the next group
        // returns only after them (in-order L1 return): 60 % of the posterior loop's stall samples (r01b profile).
        const bool last_step = (KIND == EPI_POSTERIOR) && step == 1;
        uint8_t* out_hi_row = sc + static_cast<size_t>(out_hi_buf) * P.act_buf_bytes + row_off;
        uint8_t* out_lo_row = sc + static_cast<size_t>(out_lo_buf) * P.act_buf_bytes + row_off;
        const float* bias_row = ld.bias + static_cast<size_t>(step) * ld.bias_step_stride;
        const int NC = ld.NC, NCH = ld.NCH, ngroups = NC >> 4, n_valid = ld.n_valid;
        float slope = 0.0f, c12 = 0.0f;
        bool slope01 = true;
        if (KIND == EPI_PRELU) {
          slope = __ldg(ld.slope);
          slope01 = slope >= 0.0f && slope <= 1.0f;   // PReLU(h) = max(h, a h) for 0 <= a <= 1 (every trained SDRM slope; init 0.25)
        }
        if (KIND == EPI_POSTERIOR) {
          const float4 cf = __ldg(reinterpret_cast<const float4*>(P.coef) + step);
          c12 = (valid && step <= t_row) ? cf.x * cf.y : 0.0f;   // rows not started yet (multi-resolution) keep their state
          // the noise warps have turned the state into x_i / sqrt(a_i) + sqrt(b_i) nd z_i and written the keep masks of step i-1
          mbar_wait_sleepy(bar_noise_ready(s), (noise_par >> s) & 1u, err, WD_EPI_NOISE, 128);
          noise_par ^= 1u << s;
        }
        using OutT = std::conditional_t<BF16OUT, uint16_t, float>;
        constexpr long long VEC_ELEMS = 16 / sizeof(OutT);   // logits per 16-byte store
        const bool vec_out = ((P.ld_logits & (VEC_ELEMS - 1)) == 0) && ((reinterpret_cast<uintptr_t>(P.logits) & 15) == 0);
        const bool lin_rows = P.row_ids == nullptr;   // the warp's 32 rows are consecutive rows of the logits matrix (row = physical row)
        OutT* orow = (KIND == EPI_LINEAR_OUT) ? static_cast<OutT*>(P.logits) + static_cast<size_t>(row) * P.ld_logits : nullptr;
        const bool res_layer = RES && (KIND == EPI_PRELU || KIND == EPI_POSTERIOR);   // (chain layers; the decoder streams)
        const bool publishes = !last_of_tile && KIND != EPI_LINEAR_OUT && !last_step && !res_layer;
        const bool lazy = ns == 2;   // see publish_pending
        // The bias row is warp-uniform and read by every thread: an L1-thrashed LDG costs an L2 round trip per group.  Each
        // warp stages the 16 floats of each of its own groups of a chunk in a private shared-memory slice (lane l < 4 BIAS_SLOTS
        // holds elements 4l .. 4l+3: group slot l / 4, columns 4 (l % 4) ..) one chunk ahead, and the group loop reads them with LDS.128.
        const int slice_g = sub + EPI_SUB * (lane >> 2);            // group whose bias this lane fetches (lanes < 4 BIAS_SLOTS)
        const int slice_o = slice_g * 16 + 4 * (lane & 3);
        auto fetch_slice = [&](int c) -> float4 {
          return (lane < 4 * BIAS_SLOTS && slice_g < ngroups) ? *reinterpret_cast<const float4*>(bias_row + c * NC + slice_o) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        float4 bnext = (c_first < NCH) ? fetch_slice(c_first) : make_float4(0.f, 0.f, 0.f, 0.f);
        // Resident layer: the output overwrites the layer's own input tile.  One chunk: its accumulator is complete, so every UMMA
        // has retired.  Two chunks: the first chunk's epilogue starts as soon as ITS accumulator is complete and only waits, before
        // its first store, until the second chunk's UMMAs have read the k-blocks under its columns (bar_half_read) -- it runs in
        // the shadow of the rest of the second chunk.
        for (int c = c_first; c < NCH; c += c_step) {
          const uint32_t buf = cc & 1u;
          const uint32_t t_chunk = tmem_base + lane_addr + buf * 256u;
          const int fc = c * NC;
          __syncwarp();                                             // every lane is done with the previous chunk's slice
          if (lane < 4 * BIAS_SLOTS) *reinterpret_cast<float4*>(bias_s + 4 * lane) = bnext;
          __syncwarp();
          // Software pipeline over this warp's groups: the TMEM load (and, for the posterior update, the state columns and
          // keep bits) of group g+4 is requested as soon as group g has consumed its own, so its latency hides behind the
          // arithmetic and the store of group g.
          uint32_t v[16];
          float xn[16];
          uint32_t keep = 0;
          auto request_state = [&](int g) {
            const int g16 = (fc >> 4) + g;
            if (g16 < P.Lg16) {
              keep = mask_row[g16];   // first: loads return in order, and this one hits L1/L2 (stale at the last step: its
                                      // dropout output is overwritten by the x_0 pass)
              xs_load16(xs, g16, r, xn);
            }
          };
          // does not depend on the accumulator: ask before waiting (first chunk only: later chunks fence first, and a membar
          // would wait for these loads to return)
          if (KIND == EPI_POSTERIOR && c == c_first && sub < ngroups) request_state(sub);
          SDRM_TR_EPI(1);
          mbar_wait_sleepy(bar_acc_full(buf), (cc >> 1) & 1u, err, WD_EPI_ACC, 512);
          tc_fence_after();
          SDRM_TR_EPI(2);
          if (lazy) {
            publish_pending();
          } else if (!SPLIT && c > 0 && c == NCH - 2 && publishes) {
            // Deferred publication of ALL earlier chunks (0 .. NCH-3) with ONE proxy fence: their stores were issued at least
            // a whole accumulator wait ago, and only the next layer reads these activations -- it cannot issue its first UMMA
            // before this layer's last chunk is in the tensor pipe.  (A fence.proxy.async is a membar.gpu round trip of ~1.3 us
            // per warp whatever is outstanding -- r01c profile -- so the epilogue pays three per layer instead of four.)
            // (Issued before the TMEM load: with the accumulator registers live across the fence ptxas spills.)  The last two
            // chunks are published right behind their stores: the next layer's tail k-blocks wait for them.
            stores_done();
            if (lane0)
              for (int cp = 0; cp < c; ++cp) mbar_arrive(bar_act_chunk(s, cp));
            SDRM_TR_EPI(5);
          }
          if (c + c_step < NCH) bnext = fetch_slice(c + c_step);   // after the fence: a membar would wait for this load to return
          if (KIND == EPI_POSTERIOR && c != c_first && sub < ngroups) request_state(sub);
          if (res_layer && NCH == 2 && c == 0) {   // (before the TMEM load: with the accumulator registers live across a wait ptxas spills)
            mbar_wait(bar_half_read, half_par, err, WD_EPI_LAYER);
            half_par ^= 1u;
          }
          if (sub < ngroups) tmem_ld16(t_chunk + sub * 16u, v);
          const float4* bs = reinterpret_cast<const float4*>(bias_s);
#pragma unroll 1
          for (int g = sub; g < ngroups; g += EPI_SUB, bs += 4) {
            const int f0 = fc + g * 16;
            const int g16 = f0 >> 4;
            // bias first: the LDS latency (long while the UMMAs and the TMA keep shared memory busy) overlaps the TMEM wait
            // instead of following it (r01c profile: 27 % + 25 % of the PReLU loop's samples were these two waits back to back)
            float4 b4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) b4[j] = bs[j];
            tmem_ld_wait();
            float h[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b = b4[j];
              const float2 lo = __fadd2_rn(make_float2(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1])), make_float2(b.x, b.y));
              const float2 hi = __fadd2_rn(make_float2(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])), make_float2(b.z, b.w));
              h[4 * j] = lo.x; h[4 * j + 1] = lo.y; h[4 * j + 2] = hi.x; h[4 * j + 3] = hi.y;
            }
            // (posterior update: the next group's accumulator columns are requested at the END of the iteration instead: with
            // v[] live across the update the loop spilled its invariants, and a spill reload queued behind the state loads of
            // the next group returns only after them (in-order L1 return) -- 60 % of this loop's stall samples in the r01 profile)
            if (KIND != EPI_POSTERIOR && g + EPI_SUB < ngroups) tmem_ld16(t_chunk + (g + EPI_SUB) * 16u, v);
            if (KIND == EPI_PRELU) {
              uint32_t pk[8];
              if (slope01) {
                const float2 s2 = make_float2(slope, slope);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  const float2 t = __fmul2_rn(make_float2(h[2 * e], h[2 * e + 1]), s2);
                  pk[e] = pack_bf16x2(fmaxf(h[2 * e], t.x), fmaxf(h[2 * e + 1], t.y));
                }
              } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  const float a0 = h[2 * e] > 0.f ? h[2 * e] : slope * h[2 * e];
                  const float a1 = h[2 * e + 1] > 0.f ? h[2 * e + 1] : slope * h[2 * e + 1];
                  pk[e] = pack_bf16x2(a0, a1);
                }
              }
              if (res_layer) store_res(f0, pk);
              else if (!SDRM_DEBUG_SKIP_ACT_STORES) store_act(out_hi_row, f0, pk);
            } else if (KIND == EPI_POSTERIOR) {
              // x_{i-1} = (x_i - eps (1-a_i)/sqrt(1-ab_i)) / sqrt(a_i) + sqrt(b_i) nd z; the state already holds
              // x_i / sqrt(a_i) + sqrt(b_i) nd z (noise warps), so only the eps term is left.  Padding columns need no
              // masking: their weights and bias are 0, so eps = tanh(0) = 0 and the state stays exactly 0.
              if (g16 < P.Lg16) {
                const float2 nc = make_float2(-c12, -c12);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
#if SDRM_POSTERIOR_MUFU_TANH
                  const float2 nv = __ffma2_rn(nc, make_float2(mufu_tanh(h[2 * e]), mufu_tanh(h[2 * e + 1])), make_float2(xn[2 * e], xn[2 * e + 1]));
#else
                  const float2 nv = __ffma2_rn(nc, make_float2(fast_tanh(h[2 * e]), fast_tanh(h[2 * e + 1])), make_float2(xn[2 * e], xn[2 * e + 1]));
#endif
                  xn[2 * e] = nv.x; xn[2 * e + 1] = nv.y;
                }
                xs_store16(xs, g16, r, xn);
                {
                  uint32_t pk[8];
                  dropout_pack(xn, keep, pk);
                  if (res_layer) { if (!last_step) store_res(f0, pk); }
                  else store_act(out_hi_row, f0, pk);
                }
                if (g + EPI_SUB < ngroups) request_state(g + EPI_SUB);   // xn is dead: fetch the next group's state columns
              }
              if (g + EPI_SUB < ngroups) tmem_ld16(t_chunk + (g + EPI_SUB) * 16u, v);
            } else if (KIND == EPI_TANH_SPLIT) {
              uint32_t ph[8], pl[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const float t0 = fast_tanh(h[2 * e]), t1 = fast_tanh(h[2 * e + 1]);
                const float h0 = bf16_round(t0), h1 = bf16_round(t1);
                ph[e] = pack_bf16x2(h0, h1);
                pl[e] = pack_bf16x2(t0 - h0, t1 - h1);
              }
              store_act(out_hi_row, f0, ph);
              store_act(out_lo_row, f0, pl);
            } else if constexpr (BF16OUT) {  // EPI_LINEAR_OUT, bfloat16 logits: the same three store paths at half the bytes
              uint32_t pk[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) pk[e] = pack_bf16x2(h[2 * e], h[2 * e + 1]);
              if (vec_out && (f0 + 16 <= n_valid)) {
                if (valid) {
                  __stcs(reinterpret_cast<uint4*>(orow + f0), make_uint4(pk[0], pk[1], pk[2], pk[3]));
                  __stcs(reinterpret_cast<uint4*>(orow + f0) + 1, make_uint4(pk[4], pk[5], pk[6], pk[7]));
                }
              } else if (lin_rows) {
                // Unaligned rows (an item count that is no multiple of 8): the group's 16 columns x 32 rows of bf16 fill the warp's
                // slot in one pass and go out with lanes along the columns: one instruction = 2 rows x 32 contiguous bytes.
                if (elect_one()) bulk_wait_group_read<0>();
                __syncwarp();
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(out_lane), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(out_lane + 16u), "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7]) : "memory");
                __syncwarp();
                const int col = f0 + (lane & 15);
#pragma unroll
                for (int i2 = 0; i2 < 16; ++i2) {
                  const int rr = 2 * i2 + (lane >> 4);
                  unsigned short val;
                  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(val) : "r"(out_slot + static_cast<uint32_t>(rr * 32 + (lane & 15) * 2)) : "memory");
                  if (row - lane + rr < P.n_rows && col < n_valid) __stcs(orow + static_cast<long long>(rr - lane) * P.ld_logits + col, val);
                }
                __syncwarp();
              } else if (valid) {
#pragma unroll
                for (int e = 0; e < 16; ++e)
                  if (f0 + e < n_valid) orow[f0 + e] = static_cast<uint16_t>(pk[e >> 1] >> (16 * (e & 1)));
              }
            } else {  // EPI_LINEAR_OUT
              if (vec_out && (f0 + 16 <= n_valid)) {
                if (valid) {
#pragma unroll
                  for (int j = 0; j < 4; ++j)
                    __stcs(reinterpret_cast<float4*>(orow + f0) + j, make_float4(h[4 * j], h[4 * j + 1], h[4 * j + 2], h[4 * j + 3]));
                }
              } else if (lin_rows) {
                // Rows that are not 16-byte aligned (an item count that is no multiple of 4: ml-1m 3 125, ALB 729): 16 scalar stores
                // per thread are 16 warp instructions of 32 four-byte pieces in 32 different rows -- 512 partial-sector writes per
                // group, and the decoder epilogue, not its UMMAs, set the pace (timeline: 25 us per 256-column chunk against 6.5 us
                // of tensor work).  Instead the group goes through the warp's shared-memory slot 8 columns at a time and is written
                // with lanes along the columns: one instruction = 4 rows x 32 contiguous bytes.
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                  if (elect_one()) bulk_wait_group_read<0>();   // (a TMA store of the previous layer may still be reading the slot)
                  __syncwarp();
                  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(out_lane), "f"(h[8 * hf]), "f"(h[8 * hf + 1]), "f"(h[8 * hf + 2]), "f"(h[8 * hf + 3]) : "memory");
                  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(out_lane + 16u), "f"(h[8 * hf + 4]), "f"(h[8 * hf + 5]), "f"(h[8 * hf + 6]), "f"(h[8 * hf + 7]) : "memory");
                  __syncwarp();
                  const int col = f0 + 8 * hf + (lane & 7);
#pragma unroll
                  for (int i4 = 0; i4 < 8; ++i4) {
                    const int rr = 4 * i4 + (lane >> 3);
                    float val;
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(val) : "r"(out_slot + static_cast<uint32_t>(rr * 32 + (lane & 7) * 4)) : "memory");
                    if (row - lane + rr < P.n_rows && col < n_valid) __stcs(orow + static_cast<long long>(rr - lane) * P.ld_logits + col, val);
                  }
                  __syncwarp();
                }
              } else if (valid) {
#pragma unroll
                for (int e = 0; e < 16; ++e)
                  if (f0 + e < n_valid) orow[f0 + e] = h[e];
              }
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane0) {
            if (PAIR) mbar_arrive_cluster(mapa_cluster(bar_acc_empty(buf), leader_rank));   // the leader CTA issues the UMMAs
            else mbar_arrive(bar_acc_empty(buf));
          }
          SDRM_TR_EPI(3);
          ++cc;
          // publish the layer's LAST chunk to the TMA (async) proxy right away: the next layer's tail k-blocks wait for it
          // The last two chunks are published right away: the next layer's k-blocks wait for them.  For the second-to-last
          // chunk the fence sits in the slack before the last accumulator is ready; the last chunk's is the critical path.
          if (SPLIT) {
            if (publishes) {   // every own chunk right away, through the relay warp (cluster-wide chunk barriers)
              stores_done();
              relay_chunk(c);
              SDRM_TR_EPI(5);
            }
          } else if (publishes && lazy) {
            pub_pend |= 1u << (8 * s + c);
          } else if (publishes && c >= NCH - 2) {
            stores_done();
            if (lane0) mbar_arrive(bar_act_chunk(s, c));
            SDRM_TR_EPI(5);
          }
        }
        if (KIND == EPI_POSTERIOR && last_step) {
          // x_0 pass: every thread re-reads the state columns it wrote itself (same chunk / group ownership as above)
          for (int c = c_first; c < NCH; c += c_step)
            for (int g = sub; g < ngroups; g += EPI_SUB) {
              const int g16 = ((c * NC) >> 4) + g;
              if (g16 >= P.Lg16) continue;
              const int f0 = g16 * 16;
              float x0v[16];
              xs_load16(xs, g16, r, x0v);
              uint32_t ph[8], pl[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const float h0 = bf16_round(x0v[2 * e]), h1 = bf16_round(x0v[2 * e + 1]);
                ph[e] = pack_bf16x2(h0, h1);
                pl[e] = pack_bf16x2(x0v[2 * e] - h0, x0v[2 * e + 1] - h1);
              }
              store_act(out_hi_row, f0, ph);
              store_act(out_lo_row, f0, pl);
              if (P.x0_out && valid) {
#pragma unroll
                for (int e = 0; e < 16; ++e)
                  if (f0 + e < P.L) P.x0_out[static_cast<size_t>(row) * P.L + f0 + e] = x0v[e];
              }
            }
          if (SPLIT) {
            if (!last_of_tile) {
              stores_done();
              for (int c = c_first; c < NCH; c += c_step) relay_chunk(c);
            }
          } else if (!last_of_tile && lazy) {
            pub_pend |= ((1u << NCH) - 1u) << (8 * s);
          } else if (!last_of_tile) {
            stores_done();
            if (lane0)
              for (int c = 0; c < NCH; ++c) mbar_arrive(bar_act_chunk(s, c));
          }
        }
        if (res_layer && !last_step) { res_publish(); SDRM_TR_EPI(5); }   // the next chain layer's input tile is complete (this warp's part)
        if (KIND == EPI_POSTERIOR && !last_step) {
          __syncwarp();
          if (lane0) mbar_arrive(bar_state_ready(s));   // x_{i-1} is complete: the noise warps may prepare step i-1
        }
      };
      auto run_kind = [&](const LayerDesc& ld, int step, bool last_of_tile, int out_hi_buf, int out_lo_buf, int s) __attribute__((always_inline)) {
        set_ctx(s);
        if (SPLIT && !SDRM_SPLIT_RELAY) ++rk;   // this layer's output goes to chunk-barrier set rk & 1
        switch (ld.kind) {
          case EPI_PRELU: run(std::integral_constant<int, EPI_PRELU>{}, ld, step, last_of_tile, out_hi_buf, out_lo_buf, s); break;
          case EPI_POSTERIOR: run(std::integral_constant<int, EPI_POSTERIOR>{}, ld, step, last_of_tile, out_hi_buf, out_lo_buf, s); break;
          case EPI_TANH_SPLIT: run(std::integral_constant<int, EPI_TANH_SPLIT>{}, ld, step, last_of_tile, out_hi_buf, out_lo_buf, s); break;
          default: run(std::integral_constant<int, EPI_LINEAR_OUT>{}, ld, step, last_of_tile, out_hi_buf, out_lo_buf, s); break;
        }
      };
      // a layer writes into the buffer the PREVIOUS layer of the same sub-tile read: that layer's dead lines must have been
      // discarded first (long done by then: the discard follows the previous layer's last UMMA, this follows its last epilogue)
      const bool discarding = PAIR && P.discard_kb > 0;
      uint32_t dd_pending = 0;   // bit s: a chain layer of sub-tile s has run in this tile
      auto discard_gate = [&](int s) {
        if (discarding && ((dd_pending >> s) & 1u)) {
          const uint32_t k = cnt_get(dd_cnt, s);
          dd_cnt = cnt_inc(dd_cnt, s);
          mbar_wait(bar_discard_done(s, k), (k >> 1) & 1u, err, WD_EPI_DISCARD);
        }
      };
      int cur = 0;
      for (int i = T_tile; i >= 1; --i)
        for (int l = 0; l < P.n_step; ++l) {
          for (int s = 0; s < ns; ++s) {
            discard_gate(s);
            run_kind(P.step[l], i, (P.n_dec == 0) && (i == 1) && (l == P.n_step - 1), cur ^ 1, 2, s);   // x0 lo -> buffer 2
            dd_pending |= 1u << s;
          }
          cur ^= 1;
        }
      for (int s = 0; s < ns; ++s) discard_gate(s);   // the last chain layer's phase (keeps the parities in step across tiles)
      for (int l = 0; l < P.n_dec; ++l)
        for (int s = 0; s < ns; ++s) run_kind(P.dec[l], 0, l == P.n_dec - 1, P.dec[l].out_hi == 0 ? cur : cur ^ 1, P.dec[l].out_lo, s);
      publish_pending();   // (nothing is left pending behind a decoder: its last layer publishes nothing; probe / chain-only launches)
    }
    stores_done();   // no TMA store may still be reading this CTA's shared memory at exit
  } else {
    // ======================================= noise warps ========================================
    // Thread r owns tile row r.  For every step i it (1) writes the dropout keep bits of step i-1 (one Philox call per 128
    // columns; the OUT epilogue of step i applies them to x_{i-1}) and (2) turns the fp32 state x_i into
    // x_i / sqrt(a_i) + sqrt(b_i) nd z_i (the part of the DDPM posterior that does not depend on the network) while the
    // tensor core and the epilogue warps run the step's dense layers; z comes from the Philox stream keyed by
    // (global row, step, column).
    setmaxnreg_dec<REGS_NOISE>();
    const int r = (warp - NOISE_WARP0) * 32 + lane;
    const PhiloxKeys K = philox_make_keys(P.seed);
    uint32_t st_par = 0;                     // bit s: parity of sub-tile s's state_ready barrier
    const int L = P.L, Lg16 = P.Lg16;
    const int full_groups = L >> 4;          // groups without padding columns
    for (int it = 0; it < n_iters; ++it) {
      if (!PAIR && tile_of(it, 0) >= n_tiles) break;
      const int ns = nsub_of(it);
      mbar_wait_sleepy(bar_tile_ready, it & 1, err, WD_NOISE_TILE, 128);   // x_T is in place
      const int T_tile = (P.n_step == 0) ? 0 : tile_T[it & 1];
      for (int i = T_tile; i >= 1; --i)
      for (int s = 0; s < ns; ++s) {
        const long long tile = tile_of(it, s);
        uint8_t* sc = scratch_of(tile, s);
        float* xs = reinterpret_cast<float*>(sc + NUM_ACT_BUFS * P.act_buf_bytes);
        uint4* mask_row = reinterpret_cast<uint4*>(sc + P.mask_off + static_cast<size_t>(r) * P.mask_pitch);
        const long long prow = tile * TILE_M + r;
        const bool valid = prow < P.n_rows;
        const long long row = (valid && P.row_ids) ? static_cast<long long>(P.row_ids[prow]) : prow;
        const unsigned long long grow = static_cast<unsigned long long>(P.row_offset + row);
        int t_row = P.T;
        if (P.t_start) t_row = valid ? min(max(P.t_start[prow], 0), P.T) : 0;   // clamped: an out-of-range entry must not index bias0 / coef out of bounds
        if (i != T_tile) {
          mbar_wait_sleepy(bar_state_ready(s), (st_par >> s) & 1u, err, WD_NOISE_STATE, 128);
          st_par ^= 1u << s;
        }
        // ---- (1) keep masks of step i-1 (F.dropout p = .5 of the NEXT forward, train_SDRM.py:100)
        if (SPLIT && i > 1) {
          // split mode: only the 16-bit pieces of this CTA's own column groups -- a peer may already be a layer ahead and must
          // not have its bits of the same 128-column block overwritten with the next step's
          const LayerDesc& lo = P.step[P.n_step - 1];
          uint16_t* mask16 = reinterpret_cast<uint16_t*>(mask_row);
          for (int c = c_first; c < lo.NCH; c += c_step) {
            const int g_lo = c * (lo.NC >> 4), g_hi = min(g_lo + (lo.NC >> 4), Lg16);
            for (int b = g_lo >> 3; b <= ((g_hi - 1) >> 3) && g_lo < g_hi; ++b) {
              uint32_t ww[4] = {0, 0, 0, 0};
              if (valid) {
                if (P.inj_mask) {
                  const uint8_t* mp = P.inj_mask + (static_cast<size_t>(i - 1) * P.n_rows + row) * L;
                  for (int e = 0; e < 128; ++e) {
                    const int f = b * 128 + e;
                    if (f < L && mp[f]) ww[e >> 5] |= 1u << (e & 31);
                  }
                } else {
                  const u32x4 m4 = philox_mask128(K, STREAM_MASK, grow, static_cast<uint32_t>(i - 1), static_cast<uint32_t>(b));
                  ww[0] = m4.x; ww[1] = m4.y; ww[2] = m4.z; ww[3] = m4.w;
                }
              }
              for (int g = max(g_lo, 8 * b); g < min(g_hi, 8 * b + 8); ++g) {
                const int q8 = g & 7;
                const uint32_t wsel = (q8 >> 1) == 0 ? ww[0] : (q8 >> 1) == 1 ? ww[1] : (q8 >> 1) == 2 ? ww[2] : ww[3];
                mask16[g] = static_cast<uint16_t>((wsel >> (16 * (q8 & 1))) & 0xFFFFu);
              }
            }
          }
        } else if (i > 1) {
          const int nblk = (Lg16 + 7) >> 3;
          for (int b = 0; b < nblk; ++b) {
            uint4 w = make_uint4(0, 0, 0, 0);
            if (valid) {
              if (P.inj_mask) {
                const uint8_t* mp = P.inj_mask + (static_cast<size_t>(i - 1) * P.n_rows + row) * L;
                uint32_t ww[4] = {0, 0, 0, 0};
                for (int e = 0; e < 128; ++e) {
                  const int f = b * 128 + e;
                  if (f < L && mp[f]) ww[e >> 5] |= 1u << (e & 31);
                }
                w = make_uint4(ww[0], ww[1], ww[2], ww[3]);
              } else {
                const u32x4 m4 = philox_mask128(K, STREAM_MASK, grow, static_cast<uint32_t>(i - 1), static_cast<uint32_t>(b));
                w = make_uint4(m4.x, m4.y, m4.z, m4.w);
              }
            }
            mask_row[b] = w;
          }
        }
        // ---- (2) noise half of the posterior update, AHEAD of the eps GEMM of the same step:
        //      state := state / sqrt(a_i) + sqrt(b_i) nd z_i.  The OUT epilogue then only subtracts eps * c1 / sqrt(a_i).
        const float4 cf = __ldg(reinterpret_cast<const float4*>(P.coef) + i);
        const bool active = valid && (i <= t_row);   // inactive (multi-resolution) or padding rows keep their state
        if (active && !SDRM_DEBUG_SKIP_NOISE) {
          const float2 c2 = make_float2(cf.y, cf.y), sg = make_float2(cf.z, cf.z);
          const bool has_z = cf.z != 0.0f;
          // 8 columns (one 256-bit state access, two Philox calls) at a time keeps this role inside its small register budget
          auto half_group = [&](int g16, int hf, bool padded) {
            float xo[8];
            float* px = xstate_ptr8(xs, g16, hf, r);
            if (SDRM_DEBUG_NOISE_NO_STATE) {
#pragma unroll
              for (int e = 0; e < 8; ++e) xo[e] = 0.5f;
            } else
            asm volatile("ld.global" SDRM_ST_HINT ".v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                         : "=f"(xo[0]), "=f"(xo[1]), "=f"(xo[2]), "=f"(xo[3]), "=f"(xo[4]), "=f"(xo[5]), "=f"(xo[6]), "=f"(xo[7])
                         : "l"(px)
                         : "memory");
            float z[8];
            const int f0 = g16 * 16 + hf * 8;
            if (has_z && !SDRM_DEBUG_NOISE_NO_RNG) {
              if (P.inj_z) {
                const float* zp = P.inj_z + (static_cast<size_t>(i) * P.n_rows + row) * L;
#pragma unroll
                for (int e = 0; e < 8; ++e) z[e] = (f0 + e) < L ? zp[f0 + e] : 0.0f;
              } else {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                  float z4[4];
                  philox_normal4_keys(K, STREAM_NORMAL, grow, static_cast<uint32_t>(i), static_cast<uint32_t>(g16 * 4 + hf * 2 + j), z4);
                  z[4 * j] = z4[0]; z[4 * j + 1] = z4[1]; z[4 * j + 2] = z4[2]; z[4 * j + 3] = z4[3];
                }
              }
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e) z[e] = 0.0f;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 t = __fmul2_rn(make_float2(xo[2 * e], xo[2 * e + 1]), c2);
              const float2 n = __ffma2_rn(sg, make_float2(z[2 * e], z[2 * e + 1]), t);
              xo[2 * e] = n.x; xo[2 * e + 1] = n.y;
            }
            if (padded) {
#pragma unroll
              for (int e = 0; e < 8; ++e)
                if (f0 + e >= L) xo[e] = 0.0f;   // padding columns stay exactly 0
            }
            if (SDRM_DEBUG_NOISE_NO_STATE) {
              float acc = 0.f;
#pragma unroll
              for (int e = 0; e < 8; ++e) acc += xo[e];
              if (acc == 12345.678f) px[0] = acc;   // keeps the arithmetic alive
            } else
            asm volatile("st.global" SDRM_ST_HINT ".v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                         ::"l"(px), "f"(xo[0]), "f"(xo[1]), "f"(xo[2]), "f"(xo[3]), "f"(xo[4]), "f"(xo[5]), "f"(xo[6]), "f"(xo[7])
                         : "memory");
          };
          auto group = [&](int g16, bool padded) {
            half_group(g16, 0, padded);
            half_group(g16, 1, padded);
          };
          if (SPLIT) {   // the state columns this CTA owns (its chunks of the posterior layer)
            const LayerDesc& lo = P.step[P.n_step - 1];
            for (int c = c_first; c < lo.NCH; c += c_step) {
              const int g_lo = c * (lo.NC >> 4), g_hi = min(g_lo + (lo.NC >> 4), Lg16);
#pragma unroll 1
              for (int g = g_lo; g < g_hi; ++g) group(g, g >= full_groups);
            }
          } else {
#pragma unroll 1
            for (int g = 0; g < full_groups; ++g) group(g, false);
            if (full_groups < Lg16) group(full_groups, true);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_noise_ready(s));
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
#undef c_first
#undef c_step
  if (PAIR || SPLIT) cluster_sync_all();   // nobody exits while the peer may still signal its barriers / read its operands
  if (warp == M_WARP) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_pair(tmem_base, 512);
    else tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace sdrm
