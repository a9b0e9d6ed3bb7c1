// Thin inline-PTX wrappers for the sm_100a features the TDNN kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and fences.
// sm_100a only — there is no fallback path.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>

namespace xvec {

// Device-side watchdog: when an mbarrier wait or a flag spin does not complete the kernel writes a code and traps, so a
// protocol bug shows up as a launch failure instead of hanging the GPU.  A trap destroys the context (and every device
// allocation with it), so the code goes to ONE word of mapped, pinned HOST memory shared by all translation units
// (capi.cu: watchdog_host_word()); each TU keeps the word's address in its own copy of this pointer, bound once per
// device by XVEC_DEFINE_WATCHDOG_BINDER's function before the TU's first launch.
static __device__ unsigned int* g_watchdog_ptr = nullptr;

static __device__ __noinline__ void watchdog_report(unsigned int code) {
  unsigned int* p = g_watchdog_ptr;
  if (p) {
    *reinterpret_cast<volatile unsigned int*>(p) = code;
    __threadfence_system();
  }
}
static __device__ __noinline__ void watchdog_trip(unsigned int code) {
  watchdog_report(code);
  __trap();
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One lane of a fully converged warp (warp-uniform control flow keeps addresses/descriptors in uniform registers; only the
// single-thread instructions — TMA, tcgen05.mma, tcgen05.commit — are predicated on the elected lane).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
// Non-blocking probe (try_wait may suspend the thread for a system-dependent time before it answers).
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, uint32_t code) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {  // seconds; a healthy wait is microseconds
      watchdog_trip(code);
    }
  }
}

// The same by 32-bit shared-memory address: the hot loops keep barrier / ring base addresses in registers — taking the address
// of a __shared__ object costs an S2UR + ULEA each time (the shared window of a CTA in a cluster), three times per K step.
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar_addr, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar_addr), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar_addr, uint32_t parity, uint32_t code) {
  uint32_t spins = 0;
  while (!mbar_try_wait_a(bar_addr, parity)) {
    if (++spins > (1u << 26)) watchdog_trip(code);
  }
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
}

// Arrive on the same-offset barrier of another CTA of the cluster (shared::cluster address from mapa).
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ----------------------------------------------------------------------------- cluster-scope hand-off of a 32-bit word
// The word travels as an ASYNC store that completes 4 bytes of transaction on the peer's barrier (st.async ...
// mbarrier::complete_tx::bytes), which the writer has armed with a remote arrive.expect_tx.  Observing the phase completion makes
// the word visible (the mbarrier's transaction mechanism, as for TMA loads), so the reader waits with an ordinary try_wait.  The
// plain form — st.shared::cluster, a release.cluster arrive, acquire.cluster waits — costs more: ptxas implements
// `mbarrier.arrive.release.cluster` as MEMBAR.ALL.GPU and every `try_wait.acquire.cluster` as CCTL.IVALL (an L1 invalidation),
// i.e. one GPU-scope barrier per work item in the scheduler warp and twelve L1 invalidations per work item in the peer CTA
// (tdnn_stack.cu on a B200: 267.0 vs 268.8 us per launch at 256 x 300 frames in bf16, 1 314 vs 1 338 us at 64 x 6000).
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t cluster_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void st_async_cluster_u32(uint32_t cluster_addr, uint32_t v, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.u32 [%0], %1, [%2];" ::"r"(cluster_addr), "r"(v), "r"(cluster_mbar) : "memory");
}

// ----------------------------------------------------------------------------- inter-CTA flags in global memory
__device__ __forceinline__ uint32_t ld_acquire_gpu_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu_add_u32(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Shared-memory counter with acquire + release at CTA scope: what the arriving threads did before is visible to the one that
// sees the last count.
__device__ __forceinline__ uint32_t atom_add_acq_rel_cta_shared_u32(uint32_t smem_addr, uint32_t v) {
  uint32_t old;
  asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_addr), "r"(v) : "memory");
  return old;
}
// Orders generic-proxy accesses (the flag acquire / release) against async-proxy accesses (TMA loads / stores) of this thread.
// The data behind the flags (activation tiles) lives in GLOBAL memory, so the fence is restricted to that state space: ptxas
// emits FENCE.VIEW.ASYNC.G for it, while the unrestricted `fence.proxy.async` is MEMBAR.ALL.GPU + FENCE.VIEW.ASYNC.S — a
// GPU-scope memory barrier of ~1 000 cycles that sat in the dependency warp's per-tile chain (scheduler -> flags -> fence ->
// producer may start) and in every publication of a stored tile (measured: 287 -> 281 us per launch in the debug build with
// the fences switched off; profiles/r02_experiments.txt).
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// ----------------------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ----------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled store shared -> global (bulk async group); rows / columns outside the tensor are clipped.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1, uint64_t l2_policy) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(l2_policy)
               : "memory");
}
// L2 eviction-priority descriptors for TMA cache hints (fixed encodings of createpolicy.fractional.L2::evict_*).
constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull;
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull;
constexpr uint64_t L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// All but the kPending most recent bulk groups of this thread are COMPLETE (written, not only read from smem).
template <int kPending>
__device__ __forceinline__ void tma_store_wait_done() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(kPending) : "memory");
}

// ----------------------------------------------------------------------------- tensor memory
// CTA-pair variants: the same warp index of BOTH CTAs of the pair issues them.
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(kCols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// Shared-memory operand descriptor: K-major tile, 128-byte swizzle, rows of 128 B, 8-row groups 1024 B apart.
// (bit layout: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | layout [61,64), 2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (static_cast<uint64_t>(1024 >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}

// Instruction descriptor for kind::f16 / kind::tf32, fp32 accumulate, both operands K-major.
// fmt: 0 = f16, 1 = bf16, 2 = tf32 (umma_format in gemm_tile.cuh).  (c_format [4,6) | a_format [7,10) | b_format [10,13) | N>>3 [17,23) | M>>4 [24,29))
__host__ __device__ constexpr uint32_t umma_idesc(uint32_t fmt, uint32_t m, uint32_t n) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// One K step of the CTA-pair mainloop as a single instruction group, issued by a converged warp:
//   - the elected lane issues the four tcgen05.mma of this 128-byte K chunk (32 bytes of K each) and the commits that
//     release the operand stages,
//   - every lane probes the barriers the NEXT step will need with test_wait (non-blocking) BEFORE the issue, so that the
//     ~100-150 cycles the probe takes to answer overlap the issue work instead of sitting between two steps of a single warp
//     (round 2: the MMA warp's own instruction stream, ~600-750 cycles per K step against 512 of tensor work, is what the
//     K = 512 tiles wait for).  try_wait is not usable there: it may suspend the thread until the phase completes or a time
//     limit expires, which in front of the issue delayed the MMAs of a stage that was ready until the following stage had
//     landed.  A probe that answers "not yet" leaves its bit clear; the caller then waits (try_wait loop) at the top of the
//     next step.
// Returns bit0 = next A barrier already complete, bit1 = next B barrier already complete.
// One producer step of the CTA-pair mainloop as a single instruction group (converged warp): the elected lane arms the
// leader's full barrier (leader only) and issues the two tensor loads of this stage, then the warp probes (try_wait, which may
// suspend) the empty barrier of the NEXT stage.  Returns 1 if the next stage was seen free.
__device__ __forceinline__ uint32_t tma_step_pair(uint32_t elected, uint32_t is_leader, uint32_t full_bar_local, uint32_t full_bar_leader,
                                                  uint32_t tx_bytes, uint32_t smem_a, const CUtensorMap* map_a, int32_t a0, int32_t a1,
                                                  uint64_t pol_a, uint32_t smem_b, const CUtensorMap* map_b, int32_t b0, int32_t b1,
                                                  uint64_t pol_b, uint32_t probe_bar, uint32_t probe_par) {
  uint32_t rdy;
  asm volatile(
      "{\n\t"
      ".reg .pred pe, pl, pw;\n\t"
      "setp.ne.b32 pe, %1, 0;\n\t"
      "setp.ne.b32 pl, %2, 0;\n\t"
      "and.pred pl, pl, pe;\n\t"
      "@pl mbarrier.arrive.expect_tx.shared::cta.b64 _, [%3], %5;\n\t"
      "@pe cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%6], [%7, {%8, %9}], [%4], %10;\n\t"
      "@pe cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%11], [%12, {%13, %14}], [%4], %17;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 pw, [%15], %16;\n\t"
      "selp.u32 %0, 1, 0, pw;\n\t"
      "}"
      : "=r"(rdy)
      : "r"(elected), "r"(is_leader), "r"(full_bar_local), "r"(full_bar_leader), "r"(tx_bytes), "r"(smem_a),
        "l"(reinterpret_cast<uint64_t>(map_a)), "r"(a0), "r"(a1), "l"(pol_a), "r"(smem_b), "l"(reinterpret_cast<uint64_t>(map_b)),
        "r"(b0), "r"(b1), "r"(probe_bar), "r"(probe_par), "l"(pol_b)
      : "memory");
  return rdy;
}

// One producer step for ONE operand (tdnn_stack.cu runs the activation slabs and the weight tiles on two producer warps): every
// lane probes (test_wait, non-blocking) the empty barrier of the slot this warp fills NEXT, then the elected lane arms the
// leader's full barrier (leader only; the bytes of both CTAs) and issues this CTA's tensor load.  Returns 1 if the next slot
// was seen free.  do_load = 0 arms / loads nothing (timing experiments).
__device__ __forceinline__ uint32_t tma_step_one(uint32_t elected, uint32_t is_leader, uint32_t do_load, uint32_t bar_local, uint32_t bar_leader,
                                                 uint32_t tx, uint32_t smem_dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint64_t pol,
                                                 uint32_t probe_bar, uint32_t probe_par) {
  uint32_t rdy;
  asm volatile(
      "{\n\t"
      ".reg .pred pe, pl, pw;\n\t"
      "setp.ne.b32 pe, %1, 0;\n\t"
      "setp.ne.b32 pl, %2, 0;\n\t"
      "and.pred pl, pl, pe;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 pw, [%11], %12;\n\t"
      "@pl mbarrier.arrive.expect_tx.shared::cta.b64 _, [%3], %5;\n\t"
      "@pe cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%6], [%7, {%8, %9}], [%4], %10;\n\t"
      "selp.u32 %0, 1, 0, pw;\n\t"
      "}"
      : "=r"(rdy)
      : "r"(elected & do_load), "r"(is_leader), "r"(bar_local), "r"(bar_leader), "r"(tx), "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)),
        "r"(c0), "r"(c1), "l"(pol), "r"(probe_bar), "r"(probe_par)
      : "memory");
  return rdy;
}

// A bare CTA-pair tensor load (no arming of the barrier): the bytes complete on the leader's barrier `bar_leader`, which the
// caller has armed for them.  Used by a timing experiment of the debug build only (tdnn_stack.cu, XVEC_STACK_DBG bit 32).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t bar_leader, uint32_t smem_dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar_leader), "l"(pol)
      : "memory");
}

enum { STEP_COMMIT_A = 1, STEP_COMMIT_B = 2, STEP_PROBE_A = 4, STEP_PROBE_B = 8 };
template <bool kTf32>
__device__ __forceinline__ uint32_t umma_step_pair(uint32_t elected, uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc,
                                                   uint32_t acc0, uint32_t flags, uint32_t commit_a_bar, uint32_t commit_b_bar,
                                                   uint32_t probe_a_bar, uint32_t probe_a_par, uint32_t probe_b_bar,
                                                   uint32_t probe_b_par) {
  uint32_t rdy;
#define XVEC_STEP_BODY(KIND)                                                                                      \
  asm volatile(                                                                                                   \
      "{\n\t"                                                                                                     \
      ".reg .pred pe, pacc, pt, pca, pcb, ppa, ppb, pwa, pwb;\n\t"                                                \
      ".reg .b64 a1, a2, a3, b1, b2, b3;\n\t"                                                                     \
      ".reg .b32 ra, rb, f;\n\t"                                                                                  \
      ".reg .b16 mk;\n\t"                                                                                         \
      "mov.b16 mk, 3;\n\t"                                                                                        \
      "setp.ne.b32 pe, %1, 0;\n\t"                                                                                \
      "setp.ne.b32 pacc, %6, 0;\n\t"                                                                              \
      "setp.eq.b32 pt, 0, 0;\n\t"                                                                                 \
      "and.b32 f, %7, 4;\n\tsetp.ne.b32 ppa, f, 0;\n\t"                                                          \
      "and.b32 f, %7, 8;\n\tsetp.ne.b32 ppb, f, 0;\n\t"                                                          \
      "setp.ne.b32 pwa, 0, 0;\n\t"                                                                                \
      "setp.ne.b32 pwb, 0, 0;\n\t"                                                                                \
      "@ppa mbarrier.test_wait.parity.shared::cta.b64 pwa, [%10], %11;\n\t"                                       \
      "@ppb mbarrier.test_wait.parity.shared::cta.b64 pwb, [%12], %13;\n\t"                                       \
      "add.u64 a1, %3, 2;\n\tadd.u64 a2, %3, 4;\n\tadd.u64 a3, %3, 6;\n\t"                                      \
      "add.u64 b1, %4, 2;\n\tadd.u64 b2, %4, 4;\n\tadd.u64 b3, %4, 6;\n\t"                                      \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%2], %3, %4, %5, pacc;\n\t"                                   \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%2], a1, b1, %5, pt;\n\t"                                     \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%2], a2, b2, %5, pt;\n\t"                                     \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%2], a3, b3, %5, pt;\n\t"                                     \
      "and.b32 f, %7, 2;\n\tsetp.ne.b32 pcb, f, 0;\n\tand.pred pcb, pcb, pe;\n\t"                               \
      "and.b32 f, %7, 1;\n\tsetp.ne.b32 pca, f, 0;\n\tand.pred pca, pca, pe;\n\t"                               \
      "@pcb tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%9], mk;\n\t" \
      "@pca tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%8], mk;\n\t" \
      "selp.u32 ra, 1, 0, pwa;\n\t"                                                                               \
      "selp.u32 rb, 2, 0, pwb;\n\t"                                                                               \
      "or.b32 %0, ra, rb;\n\t"                                                                                    \
      "}"                                                                                                         \
      : "=r"(rdy)                                                                                                 \
      : "r"(elected), "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc0), "r"(flags), "r"(commit_a_bar),        \
        "r"(commit_b_bar), "r"(probe_a_bar), "r"(probe_a_par), "r"(probe_b_bar), "r"(probe_b_par)                 \
      : "memory")
  if constexpr (kTf32) {
    XVEC_STEP_BODY("tf32");
  } else {
    XVEC_STEP_BODY("f16");
  }
#undef XVEC_STEP_BODY
  return rdy;
}
// The same K step with everything that is fixed per (layer shape, tap position) decided at COMPILE time (tdnn_stack.cu,
// mma_tile_fixed): what is committed / probed (kLastTap: this is the last tap of a channel chunk — hand the slab slot back,
// probe the next slab), so no flag tests or predicate logic at run time; one predicate (the elected lane) on all six issue
// instructions; and the operand descriptors advance in their low 32-bit word only (start address >> 4 in bits [0,14): + 2 per
// 32 bytes of K, which cannot carry out of the field below 256 KiB of shared memory), so the uniform datapath does 32-bit adds
// instead of 64-bit add-with-carry pairs chained through a carry predicate.
template <bool kTf32, bool kLastTap>
__device__ __forceinline__ uint32_t umma_step_fixed(uint32_t elected, uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                                    uint32_t acc0, uint32_t commit_a_bar, uint32_t commit_b_bar, uint32_t probe_a_bar,
                                                    uint32_t probe_a_par, uint32_t probe_b_bar, uint32_t probe_b_par) {
  uint32_t rdy;
#define XVEC_FIXED_BODY(KIND, PROBE_A, COMMIT_A)                                                                  \
  asm volatile(                                                                                                   \
      "{\n\t"                                                                                                     \
      ".reg .pred pe, pacc, pt, pwa, pwb;\n\t"                                                                    \
      ".reg .b64 a0, a1, a2, a3, b0, b1, b2, b3;\n\t"                                                             \
      ".reg .b32 ra, rb, t;\n\t"                                                                                  \
      ".reg .b16 mk;\n\t"                                                                                         \
      "mov.b16 mk, 3;\n\t"                                                                                        \
      "setp.ne.b32 pe, %13, 0;\n\t"                                                                               \
      "setp.ne.b32 pacc, %6, 0;\n\t"                                                                              \
      "setp.eq.b32 pt, 0, 0;\n\t"                                                                                 \
      "setp.ne.b32 pwa, 0, 0;\n\t"                                                                                \
      PROBE_A                                                                                                     \
      "mbarrier.test_wait.parity.shared::cta.b64 pwb, [%11], %12;\n\t"                                            \
      "mov.b64 a0, {%2, %4};\n\t"                                                                                 \
      "mov.b64 b0, {%3, %4};\n\t"                                                                                 \
      "add.u32 t, %2, 2;\n\tmov.b64 a1, {t, %4};\n\t"                                                            \
      "add.u32 t, %3, 2;\n\tmov.b64 b1, {t, %4};\n\t"                                                            \
      "add.u32 t, %2, 4;\n\tmov.b64 a2, {t, %4};\n\t"                                                            \
      "add.u32 t, %3, 4;\n\tmov.b64 b2, {t, %4};\n\t"                                                            \
      "add.u32 t, %2, 6;\n\tmov.b64 a3, {t, %4};\n\t"                                                            \
      "add.u32 t, %3, 6;\n\tmov.b64 b3, {t, %4};\n\t"                                                            \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%1], a0, b0, %5, pacc;\n\t"                                   \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%1], a1, b1, %5, pt;\n\t"                                     \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%1], a2, b2, %5, pt;\n\t"                                     \
      "@pe tcgen05.mma.cta_group::2.kind::" KIND " [%1], a3, b3, %5, pt;\n\t"                                     \
      "@pe tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%8], mk;\n\t" \
      COMMIT_A                                                                                                    \
      "selp.u32 ra, 1, 0, pwa;\n\t"                                                                               \
      "selp.u32 rb, 2, 0, pwb;\n\t"                                                                               \
      "or.b32 %0, ra, rb;\n\t"                                                                                    \
      "}"                                                                                                         \
      : "=r"(rdy)                                                                                                 \
      : "r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(acc0), "r"(commit_a_bar), "r"(commit_b_bar),  \
        "r"(probe_a_bar), "r"(probe_a_par), "r"(probe_b_bar), "r"(probe_b_par), "r"(elected)                      \
      : "memory")
#define XVEC_FIXED_PROBE_A "mbarrier.test_wait.parity.shared::cta.b64 pwa, [%9], %10;\n\t"
#define XVEC_FIXED_COMMIT_A "@pe tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%7], mk;\n\t"
  if constexpr (kTf32) {
    if constexpr (kLastTap) XVEC_FIXED_BODY("tf32", XVEC_FIXED_PROBE_A, XVEC_FIXED_COMMIT_A);
    else XVEC_FIXED_BODY("tf32", "", "");
  } else {
    if constexpr (kLastTap) XVEC_FIXED_BODY("f16", XVEC_FIXED_PROBE_A, XVEC_FIXED_COMMIT_A);
    else XVEC_FIXED_BODY("f16", "", "");
  }
#undef XVEC_FIXED_BODY
#undef XVEC_FIXED_PROBE_A
#undef XVEC_FIXED_COMMIT_A
  return rdy;
}
// Pair commit: arrives on the same-offset barrier of every CTA in `cta_mask` once the issued MMAs complete.
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread i gets lane i, v[j] = column j).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace xvec
