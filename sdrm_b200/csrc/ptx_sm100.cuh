// Thin inline-PTX wrappers for the sm_100a features the SDRM kernels use:
// mbarrier, cp.async.bulk (TMA bulk engine), tcgen05 (UMMA + TMEM), proxy fences.
// Hand-written; descriptor bit layouts follow the PTX ISA tcgen05 matrix / instruction
// descriptor tables.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "host_util.h"

namespace sdrm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// one lane of a converged warp (uniform-datapath instructions should be issued under this predicate)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
// warpgroup-wide register re-budgeting (all four warps of an aligned warpgroup execute it)
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Watchdog: a protocol bug must become an error code, never a hung GPU box.  The limit is a run-time value (per translation
// unit: apply_watchdog_env below copies it in; environment variable SDRM_WATCHDOG_MS, 0 = no limit), because the
// global timer keeps running while a context is preempted (time-sliced GPU, debugger, profiler replay) and a healthy run must
// not be killed there.
#ifndef SDRM_WATCHDOG_NS
#define SDRM_WATCHDOG_NS 4000000000ull
#endif
static __constant__ unsigned long long g_sdrm_watchdog_ns = SDRM_WATCHDOG_NS;
// Copies SDRM_WATCHDOG_MS into the calling translation unit's g_sdrm_watchdog_ns (static, so each unit's module has its own
// copy) on the current device, once per device: every device a process uses gets the limit.
static inline int apply_watchdog_env() {
  static bool done[64] = {false};
  int dev = 0;
  SDRM_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && done[dev]) return 0;
  if (dev < 64) done[dev] = true;
  const char* e = getenv("SDRM_WATCHDOG_MS");
  if (!e || !*e) return 0;
  const unsigned long long ns = strtoull(e, nullptr, 10) * 1000000ull;
  SDRM_CUDA(cudaMemcpyToSymbol(g_sdrm_watchdog_ns, &ns, sizeof ns));
  return 0;
}
// try_wait with a suspend-time hint: the waiting thread is parked by the hardware until the phase completes or the hint
// (ns) expires, so a waiter neither issues poll instructions nor wakes up late.  (The polling loops with __nanosleep were
// 45 % of all executed warp instructions of the engine kernel — ncu source page, r01 — and every epilogue warp woke up
// to half a microsecond after its accumulator was ready.)
#ifndef SDRM_WAIT_HINT_NS
#define SDRM_WAIT_HINT_NS 200000u
#endif
// CL: acquire at CLUSTER scope (the phase was completed by another CTA's release.cluster arrival: column-split chunk barriers)
template <bool CL = false>
__device__ __forceinline__ uint32_t mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t hint_ns) {
  uint32_t ok;
  if (CL)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(hint_ns)
        : "memory");
  else
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(hint_ns)
        : "memory");
  return ok;
}
// bounded wait: the timer is only read every 256 expired hints
template <bool CL = false>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err_word, int code) {
  if (mbar_try_wait_hint<CL>(bar, parity, SDRM_WAIT_HINT_NS)) return;
  uint32_t spins = 0;
  uint64_t t0 = 0;
  while (!mbar_try_wait_hint<CL>(bar, parity, SDRM_WAIT_HINT_NS)) {
    if ((++spins & 0xffu) == 0) {
      const uint64_t t = globaltimer_ns();
      if (t0 == 0) t0 = t;
      else if (g_sdrm_watchdog_ns != 0ull && t - t0 > g_sdrm_watchdog_ns) {
        // (may be mapped host memory: plain accesses.)  Word 0 = the first wait that timed out; word code / 100 (1 producers, 2 UMMA
        // issuer, 3 epilogue, 4 noise, 5 GEMM, 6 discard) = where that role is stuck -- the other roles time out moments later
        if (err_word) {
          volatile int* ew = reinterpret_cast<volatile int*>(err_word);
          if (ew[0] == 0) ew[0] = code;
          ew[(code / 100) & 7] = code;
          // give the other stuck roles the time to record themselves before the context dies
          const uint64_t t1 = globaltimer_ns();
          while (globaltimer_ns() - t1 < 200000000ull) { }
        }
        __threadfence_system();
        __trap();
      }
    }
  }
}
// (historical name: the waits of the epilogue / noise warps used to sleep between polls)
__device__ __forceinline__ void mbar_wait_sleepy(uint32_t bar, uint32_t parity, int* err_word, int code, uint32_t sleep_ns) {
#ifdef SDRM_WAIT_POLL   // the previous polling loop, kept for A/B measurements only
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(sleep_ns);
    if (++spins == (1u << 22)) {
      if (err_word && *reinterpret_cast<volatile int*>(err_word) == 0) *reinterpret_cast<volatile int*>(err_word) = code;
      __threadfence_system();
      __trap();
    }
  }
#else
  (void)sleep_ns;
  mbar_wait(bar, parity, err_word, code);
#endif
}

// ----------------------------------------------------------------------------------------------
// TMA bulk engine (1-D bulk copy global -> shared, completion on an mbarrier)
// ----------------------------------------------------------------------------------------------
// L2 eviction-priority policies: the activation images and weights are re-read within microseconds (evict_last), the
// fp32 state and the logits stream through (evict_first / .cs)
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
// 2-D tensor-map load whose destination is this CTA's shared memory but whose completion is signalled on the mbarrier of
// either CTA of the tcgen05 pair (both addresses are shared::cluster addresses, see mapa_cluster)
__device__ __forceinline__ void tma_load_2d_pair_hint(uint32_t dst_cluster, const void* tmap, int c0, int c1, uint32_t bar_cluster,
                                                      uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.cta_group::2.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
      ::"r"(dst_cluster), "l"(tmap), "r"(c0), "r"(c1), "r"(bar_cluster), "l"(pol)
      : "memory");
}
// 2-D tensor-map load into this CTA's shared memory, completion on a local mbarrier (single-CTA mode)
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst_smem, const void* tmap, int c0, int c1, uint32_t bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
      ::"r"(dst_smem), "l"(tmap), "r"(c0), "r"(c1), "r"(bar), "l"(pol)
      : "memory");
}
// 2-D tensor-map store shared -> global (bulk async-group completion: bulk_commit_group / bulk_wait_group[_read])
__device__ __forceinline__ void tma_store_2d_hint(const void* tmap, int c0, int c1, uint32_t src_smem, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;"
      ::"l"(tmap), "r"(c0), "r"(c1), "r"(src_smem), "l"(pol)
      : "memory");
}
// 1-D bulk copy global -> shared, completion on a local mbarrier (plain form: used by the microbenchmarks in tools/)
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(dst_smem), "l"(src_gmem), "r"(bytes), "r"(bar)
      : "memory");
}
// same with an L2 eviction-priority hint (single-CTA mode of the engine)
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(dst_smem), "l"(src_gmem), "r"(bytes), "r"(bar), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(dst_gmem), "r"(src_smem), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// generic-proxy writes -> visible to the async proxy (TMA / UMMA operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, UMMA issue, commit, TMEM loads
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// cta_group::2 variants: one warp of EACH CTA of the pair executes alloc / dealloc
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle, bf16:
//   rows are 128 B (64 bf16) apart inside an 8-row / 1024 B swizzle atom, atoms are SBO = 1024 B apart.
//   bits [0,14) addr>>4 | [16,30) LBO>>4 (unused for swizzled K-major, 1) | [32,46) SBO>>4 | [46,48) version=1
//   | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16: D=f32, A=B=bf16, both K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Instruction descriptor for kind::i8: D=s32, A=B=u8 (unsigned), both K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_u8(int M, int N) {
  return (2u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
// one K = 32 step (32 bytes of each K-major row): exact integer products, s32 accumulate
__device__ __forceinline__ void umma_u8_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued UMMAs of this thread arrive on `bar` when they retire
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// cta_group::2: issued by the leader CTA only; A rows 0-127 / 128-255 and the two N-halves of B come from the shared
// memory of CTA 0 / CTA 1 at the same CTA-relative offsets, D lands in each CTA's own TMEM (its 128 rows).
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (.release at CTA scope) like CUTLASS ClusterBarrier::arrive(cta_id): a cluster-scope release would
  // first drain every outstanding global store of the thread (measured: ~10 us per epilogue chunk)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// arrive with a CLUSTER-scope release: what the issuing thread observed / wrote before is visible to the CTA that owns the barrier
// (only for threads without outstanding global stores: see above)
__device__ __forceinline__ void mbar_arrive_cluster_release(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void fence_acq_rel_cluster() { asm volatile("fence.acq_rel.cluster;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// 32 lanes x 16 consecutive fp32 columns: thread t of the warp reads TMEM lane (base_lane + t)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// small math
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ float fast_tanh(float x) {
  // tanh(x) = 1 - 2 / (exp(2x) + 1) on two MUFU ops (ex2.approx, rcp.approx: no Newton step, no slow path), abs error ~3e-7,
  // saturates cleanly (e = inf -> r = 0 -> 1;  e = 0 -> r = 1 -> -1)
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));   // 2*log2(e)
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return fmaf(-2.0f, r, 1.0f);
}
// one MUFU op (tanh.approx.f32, max abs error 2^-10.99): only where the result is scaled by a small coefficient (the posterior
// update multiplies it by (1-a_i)/sqrt(1-ab_i)/sqrt(a_i): <= 0.02 for T >= 50, up to ~0.14 at T = 1, i.e. <= 7e-5 absolute per step)
__device__ __forceinline__ float mufu_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// keep a loop-invariant value in its register: without this ptxas re-derives thread-index based values with S2R
// (a ~20-cycle short-scoreboard stall) inside the hottest loops
__device__ __forceinline__ void pin_reg(uint32_t& v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ void pin_reg(int& v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bf16_round(float x) {
  uint32_t u = pack_bf16x2(x, 0.0f) & 0xFFFFu;
  return __uint_as_float(u << 16);
}

}  // namespace sdrm
