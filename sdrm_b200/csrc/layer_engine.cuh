// Shared definitions of the streaming tcgen05 layer engine (kernel K1, SURVEY.md §8a3-a6).
#pragma once
#include <cuda.h>
#include <stdint.h>
#include <stddef.h>

namespace sdrm {

constexpr int TILE_M = 128;                        // rows of users per CTA tile (UMMA M)
constexpr int KBLK = 64;                           // bf16 elements per 128-byte swizzle row
constexpr int A_TILE_BYTES = TILE_M * 128;         // one activation k-block image: 128 rows x 128 B
#ifndef SDRM_MAX_NC
#define SDRM_MAX_NC 256   // widest UMMA N.  240 would shrink a pair-mode stage to 31 KB and fit 7 stages, but measured
#endif                    // slower (81.4 vs 79.8 ms for two waves at cfg 5): the decoder then needs 84 instead of 79 chunks
constexpr int MAX_NC = SDRM_MAX_NC;
constexpr int W_TILE_BYTES_MAX = MAX_NC * 128;     // one weight k-block image
constexpr int STAGE_BYTES = A_TILE_BYTES + W_TILE_BYTES_MAX;
constexpr int NUM_STAGES = 4;
constexpr int MAX_STEP_LAYERS = 8;                 // 2 + nh, nh <= 6
constexpr int NUM_ACT_BUFS = 4;
constexpr int MAX_ACT_CHUNKS = 8;                  // N chunks of an activation-producing layer (features <= 8 * MAX_NC)
constexpr int MAX_SUB = 2;                         // row tiles a CTA interleaves layer by layer (ChainParams::n_sub)
#ifndef SDRM_EPI_WARPS
#define SDRM_EPI_WARPS 12   // 12 warps x 128 registers beat 16 x 96 (264.5 vs 271.7 ms per cfg-5 shard, same box): no spills in the group loops
#endif
constexpr int EPI_WARPS = SDRM_EPI_WARPS;          // 3 (or 4) per TMEM lane quarter
constexpr int EPI_SUB = EPI_WARPS / 4;             // warps sharing a lane quarter split the column groups
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int CTRL_WARPS = 4;                      // weight producer, UMMA issuer, activation producer (+1 idle: setmaxnreg works on whole warpgroups)
constexpr int NOISE_WARPS = 4;                     // one thread per tile row: Gaussian half of the posterior update
constexpr int ENGINE_THREADS = CTRL_WARPS * 32 + EPI_THREADS + NOISE_WARPS * 32;
// warp roles: epilogue 0..EPI_WARPS-1, then 4 noise warps, then the control warps.  The control warps get the HIGHEST warp ids: the SM's warp
// arbiter favours higher ids, and the three single-issuer loops must never wait behind the busy ALU warps.
constexpr int NOISE_WARP0 = EPI_WARPS;
constexpr int W_WARP = EPI_WARPS + NOISE_WARPS;    // weight TMA producer
constexpr int M_WARP = W_WARP + 1;                 // UMMA issuer (also allocates TMEM)
constexpr int A_WARP = W_WARP + 2;                 // activation TMA producer
// Register budget (setmaxnreg, per warpgroup): 640 threads launch with 96 registers per thread; the control and the noise
// warpgroup drop to 48 so that the three epilogue warpgroups can grow to 128.  (16 epilogue warps x 96 registers made ptxas
// spill loop invariants into the group loops -- and a spill reload queued behind the state loads returns only after them;
// 12 x 128 compiles without spills and measured 264.5 vs 271.7 ms per cfg-5 shard on the same box.)
#ifndef SDRM_REGS_EPI
#define SDRM_REGS_CTRL 48
#define SDRM_REGS_NOISE 48
#define SDRM_REGS_EPI 128
#endif
constexpr int REGS_CTRL = SDRM_REGS_CTRL, REGS_NOISE = SDRM_REGS_NOISE, REGS_EPI = SDRM_REGS_EPI;
constexpr int LAUNCH_REGS = (65536 / ENGINE_THREADS) / 8 * 8;   // what __launch_bounds__(ENGINE_THREADS, 1) lets ptxas allocate per thread
static_assert(128 * (REGS_CTRL + REGS_NOISE) + EPI_THREADS * REGS_EPI <= LAUNCH_REGS * ENGINE_THREADS, "register pool");
constexpr int ENGINE_SMEM_BYTES = 232448;          // all 227 KB: pair mode stages 7 x 32 KB, single mode 4 x 48 KB

enum EpiKind : int { EPI_PRELU = 0, EPI_POSTERIOR = 1, EPI_TANH_SPLIT = 2, EPI_LINEAR_OUT = 3 };

// error codes the device watchdog writes (which wait timed out)
enum : int { WD_PRODUCER_EMPTY = 101, WD_PRODUCER_ACT = 102, WD_PRODUCER_TILE = 103, WD_MMA_FULL = 201,
             WD_MMA_ACC = 202, WD_MMA_TILE = 203, WD_EPI_ACC = 301, WD_EPI_NOISE = 302, WD_EPI_DISCARD = 303, WD_NOISE_STATE = 401, WD_NOISE_TILE = 402, WD_DISCARD = 601,
             WD_MMA_AREADY = 204, WD_MMA_PEER = 205, WD_RELAY = 701, WD_EPI_LAYER = 304 };

struct LayerDesc {
  const uint8_t* w_img;   // weight images [which: hi, lo][chunk][k block][NC rows x 128 B], 128B-swizzled
  const float* bias;      // [bias rows][Np]
  const float* slope;     // PReLU slope (device scalar) or nullptr
  int bias_step_stride;   // floats between the bias rows of consecutive diffusion steps (0: constant)
  int KB;                 // 64-wide k blocks per pass
  int kmma_last;          // UMMAs (K = 16 each) issued for the last k block, 1..4
  int passes;             // 1 = bf16, 3 = bf16x3 split (hi*hi + hi*lo + lo*hi)
  int NCH, NC;            // N chunks and chunk width (multiple of 16, <= 256)
  int kind;               // EpiKind
  int in_hi, in_lo;       // activation buffers read (lo only when passes == 3)
  int out_hi, out_lo;     // activation buffers written
  int n_valid;            // real output features
};

struct ChainParams {
  LayerDesc step[MAX_STEP_LAYERS];
  LayerDesc dec[2];
  int n_step, n_dec;
  int T, L, Lg16;         // Lg16 = ceil(L / 16) column groups of the fp32 state
  int preloaded_input;    // probe mode: activation images were packed per TILE by the host
  int n_sub;              // 1 or 2: row tiles per CTA iteration, interleaved layer by layer (scratch slot = CTA * n_sub + s)
  long long n_rows, row_offset;
  const float* coef;      // [T+1][4] = c1, c2, sigma*nd, 0   (denoise_add_noise, train_SDRM.py:20-25)
  const int32_t* t_start; // per-row start step or nullptr (indexed by physical row)
  const int32_t* row_ids; // physical -> logical row or nullptr
  float* x0_out;          // [n, L] or nullptr
  void* logits;           // [n, ld_logits] fp32, or bfloat16 bits in the BF16OUT instantiations (ld_logits in elements)
  long long ld_logits;
  const float* inj_xT;    // [n, L]
  const float* inj_z;     // [T+1, n, L]
  const uint8_t* inj_mask;// [T+1, n, L]
  unsigned long long seed;
  uint8_t* scratch;       // per-CTA (or per-tile in probe mode) scratch
  size_t scratch_stride;  // bytes per CTA
  size_t act_buf_bytes;   // bytes of one activation buffer (KBmax * A_TILE_BYTES)
  size_t mask_off;        // per-CTA scratch: offset of the dropout keep bits [128 rows][mask_pitch bytes] (bit c of a row = column c)
  int mask_pitch;         // bytes per row of keep bits: 16 * ceil(Lg16 / 8)
  int discard_kb;         // pair mode: k-blocks of a chain layer's dead input image the discard warp drops from the L2 (0 = off)
  int resident;           // pair mode, one row tile per CTA: the chain's activation tile lives in shared memory (see the kernel)
  int res_nstg;           // resident mode: pipeline stages left to the weight / decoder stream (the rest of the ring holds the tile)
                          // column-split mode: stages of split_stage_bytes in the 192 KB ring (4 .. 6)
  uint32_t split_stage_bytes;   // column-split mode: A_TILE_BYTES + the widest chunk's weight k-block, 1024-byte multiple
  int* err_word;
  // pair mode only: TMA tensor maps over the weight blobs (rows of 128 B, box = NC/2 rows) and over the whole
  // activation scratch (box = 128 rows); tensor-map loads may complete on the LEADER CTA's mbarrier (.cta_group::2)
  CUtensorMap tm_step_w[MAX_STEP_LAYERS];
  CUtensorMap tm_dec_w[2];
  CUtensorMap tm_act;       // loads: box 128 B x 128 rows, SWIZZLE_128B (linear global rows -> UMMA operand layout)
  CUtensorMap tm_act_st;    // epilogue stores: box 32 B x 32 rows, no swizzle
  int debug_flags;            // perf experiments only (-DSDRM_PERF_DEBUG builds): 1 = skip activation stores, 4 = skip noise; 8 = trace k-blocks
  unsigned long long* trace;  // debug: [3 roles][TRACE_CAP] (event code << 56 | globaltimer ns), CTA 0 only; or nullptr
};
constexpr int TRACE_CAP = 8192;

}  // namespace sdrm
