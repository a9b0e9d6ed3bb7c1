// The whole frame-level TDNN stack (time_context_layers, main.py:38-44) as ONE persistent dataflow kernel — sm_100a only.
//
// tdnn_gemm.cu runs one layer per launch; a step then pays five launch latencies / prologues / drain tails and five wave
// quantisations (600 tiles on 74 CTA pairs = 8.1 waves).  Here every (layer, 256-frame m-tile, 256-channel n-tile) of the
// stack is one WORK ITEM of a single launch:
//
//   * dynamic tile scheduler: a scheduler warp in the leader CTA of each pair draws the next item with one atomicAdd on a global
//     counter (while the current tile is loading) and hands it to all warp roles of both CTAs through a small shared-memory ring
//     (mbarrier full/empty; the peer's copy travels as an st.async that completes a transaction on the peer's barrier).  Items are
//     drawn strictly in order and an item only depends on EARLIER items, so any number of resident CTAs makes progress —
//     two of these kernels on two streams cannot deadlock each other.
//   * item order: bands of `band` m-tiles; inside a band layer 1, 2, ... L, the m-range of layer l skewed down by l tiles
//     (layer l+1 tile m reads layer l tiles m-1.. m+1, all in the same or an earlier band).  Bands of ~2.3 x pairs m-tiles are
//     long enough that an item's inputs are complete when it is drawn and short enough that a band's activations stay in L2
//     between the layers (see pick_band).
//   * inter-layer dependencies: once the TMA stores of a tile are COMPLETE (cp.async.bulk.wait_group per epilogue warp, deferred
//     so that it never blocks a busy warp) the last of a CTA's eight epilogue warps adds 8 to ready[layer][m_tile]
//     (fence.proxy.async.global + red.release.gpu: ONE gpu-scope release per tile and CTA); a dependency warp per
//     CTA runs ahead of the TMA producer, polls (ld.acquire.gpu) the flags of the tiles the next items touch and hands each
//     item to the producer through an mbarrier, so flag latency and the proxy fence stay off the load path.
//     The two ping-pong activation buffers are safe: tile (l, m) overwrites rows whose readers (l-1, m-1) and (l-1, m) it
//     has just waited for.
//
//   * warp roles (384 threads): 0 activation-slab producer, 1 MMA issuer (leader CTA), 2-9 epilogue, 10 scheduler (leader) +
//     dependency resolver, 11 weight-tile producer.  What paces the tensor pipe is the instruction stream of the ONE MMA warp
//     (512 cycles of tensor work per K step): its loop keeps everything in registers and probes barriers without blocking.
//
// TMEM double buffering and the tcgen05 step are the ones of tdnn_gemm.cu.  Layers 1.. run in the activation dtype kAct:
// kind::f16 with bf16 or f16 operands, or kind::tf32; layer 0 runs in its own dtype: kind::tf32 on the float32 MFCCs, or
// kind::f16 on a 16-bit copy of them in "window form" (taps = 1, cin = taps*channels over overlapping rows;
// include/xvec_b200.h).  The last layer is computed TRANSPOSED (weights as the M operand) so that its pooling epilogue reduces
// over time in registers.
#include "gemm_tile.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <mutex>
#include <type_traits>

namespace xvec {

// Operand staging: the activation ("A") side is loaded once per 128-byte channel chunk as a SLAB of 128 + max_tap_offset frame
// rows and reused by every tap of the layer — tap j's MMA reads the slab through a descriptor whose start address is shifted
// by tap_off[j] rows (the 128-byte swizzle is a function of the absolute shared-memory address, so a row shift keeps TMA's
// and UMMA's patterns in step as long as the slab base is 1024-byte aligned).  The weight ("B") side streams one 128 x 128-byte
// tile per (chunk, tap).
//
// ONE ring for both: RING_SLOTS uniform slots of SLOT_BYTES (a slab, 17 KiB; a weight tile uses the first 16 KiB), filled by
// the producer in exactly the order the MMA warp consumes them — per chunk the slab, then one weight tile per tap — each slot
// with its own full / empty mbarrier (a weight slot is handed back by its own MMA group's commit, a slab slot by its last
// tap's).  What a K step costs is set by how many steps' worth of operands are in flight per SM (measured on B200, 256 x 300,
// bf16, MMA-warp cycles per tile with separate rings of a slabs + b weight stages: 3-tap TDNN2/3 — b = 5 / 6 / 7 steps in flight:
// 14 400 / 13 460 / 12 850 of 12 288 ideal; 1-tap TDNN4/5 — min(a, b) = 4 / 5 steps: 7 110 / 6 660 of 4 096), and two separate
// rings cannot serve both layer shapes: the 3-tap layers want few slabs and many weight stages, the 1-tap layers want as many
// of one as of the other.  A single FIFO of uniform slots is as deep as the shared memory allows for EITHER consumption pattern
// (11 slots: 8.25 steps of a 3-tap layer, 5.5 of a 1-tap layer; separate rings 5 + 6: 6 and 5) and needs no drain between layers.
// Measured: MMA-warp cycles per TDNN2/3 tile 9 / 10 / 11 / 12 slots: 16 480 / 14 050 / 13 540 / 13 090; whole launch 326.8 /
// 299.2 / 295.8 / 297.1 us (debug builds) — the launch as a whole gains 1-2 % over the separate rings, within box-to-box spread.
// Shared memory per CTA: 1 KiB alignment slack + the ring + the TMA-store staging of the 8 epilogue warps.  bf16 activations:
// 10 slots + two 2 KiB boxes (32 rows x 64 bytes) per warp = 203 KiB; float32 activations: 10 slots + one 4 KiB box (32 rows x
// 128 bytes) = 203 KiB.  NOT the 227 KiB a CTA could have: the kernels of a batch's tail (pooling finalize + segment layers)
// must fit on the SM NEXT TO a resident CTA of the next batch's stack kernel (about 20 KiB of shared memory and 20 K registers
// stay free), otherwise they wait for a whole stack kernel to drain — measured in round 1: ~24 us of a 325 us step.  Measured
// here (256 x 300, bf16, us per launch on one box): 12 slots / 1 box 290.5, 11 / 2 boxes 291.9, 11 / 1 box 292.2 — the last
// slot buys less than the co-residency it would cost.
// Once the fences / publication were made cheap (round 2), the store epilogue weighs more: 10 slots + TWO boxes per bf16 warp
// (staging chunk k+1 while the store of chunk k still reads its box) 262.8 us against 11 slots + one box 263.7 (64 x 6000:
// 1 297 vs 1 303).
template <bool kAllTf32>
struct StackCfg {
  static constexpr int SLOTS = 10;
  static constexpr int BOX_W = kAllTf32 ? 128 : 64;                     // bytes per row of a store box (32 rows x 32 columns)
  static constexpr int BOX_BYTES = 32 * BOX_W;
  static constexpr int NBUF = kAllTf32 ? 1 : 2;                          // store boxes in flight per epilogue warp
  static constexpr int STAGE_BYTES = NBUF * BOX_BYTES;                   // staging per epilogue warp
};
constexpr int SLAB_ROWS_MAX = BM_CTA + XVEC_STACK_MAX_TAP_OFFSET;  // frame rows per slab (128 + the largest tap offset, <= 8)
constexpr int SLAB_BYTES = SLAB_ROWS_MAX * BK_BYTES;  // 17 KiB, a multiple of 1024
constexpr int SLOT_BYTES = SLAB_BYTES;
static_assert(SLOT_BYTES % 1024 == 0 && SLOT_BYTES >= B_BYTES, "slot bases must stay 1024-byte aligned for SWIZZLE_128B and hold a weight tile");
constexpr int SCHED_SLOTS = 8;            // work-item ring between the scheduler and the warp roles
constexpr int CREDIT_BARS = 4;            // "tile started" barriers; the scheduler's run-ahead must stay below this (see the scheduler warp)
constexpr int STACK_RUNAHEAD = 1;         // items a pair may hold that its producer has not started (p.runahead); measured: 1, 2, 3 give the same launch time
constexpr uint32_t ITEM_DONE = 0xFFFFFFFFu;
constexpr int SCHED_CONSUMERS = 2 * EPI_WARPS + 6;  // per slot: the two producer warps of both CTAs, leader MMA warp, peer dependency warp, 8 epilogue warps of each CTA
static_assert((EPI_WARPS & (EPI_WARPS - 1)) == 0, "publish() counts the epilogue warps of a CTA modulo EPI_WARPS");
constexpr int DEP_WARP = 2 + EPI_WARPS;             // warp 10
constexpr int WPROD_WARP = DEP_WARP + 1;            // warp 11: the weight-tile producer (warp 0 loads the activation slabs)
constexpr int STACK_THREADS = GEMM_THREADS + 64;
// Register cap: 384 threads x 112 registers = 42 K of the SM's 64 K, so that the tail kernels of the previous batch (fc_small: 128
// threads x 80 registers per CTA) find room next to a resident stack CTA (without a cap ptxas takes all 168 a 384-thread CTA may have).
constexpr int STACK_MAX_REGS = 112;

struct StackLayer {
  int n, n_tiles, taps, cpt;  // K loop = taps * cpt chunks of 128 bytes
  int tf32;                   // operand kind of this layer (1: float32 activations / TF32 math, 0: 16-bit, the kernel's kAct)
  int slab_rows;              // 128 + largest tap offset: frame rows one activation slab holds (= the A tensor map's box)
  int n_pad;                  // rows of one K chunk of the chunk-major packed weights (n_tiles * 256)
  int tap_off[XVEC_MAX_TAPS];
  unsigned tap_off4;          // the same, four bits each (tap j in bits [4j, 4j+4)): one constant load per tile on the MMA warp
  const float* bias;
};

struct StackMaps {
  CUtensorMap a[XVEC_MAX_STACK], b[XVEC_MAX_STACK], y[XVEC_MAX_STACK];
};

struct StackParams {
  int rows, m_tiles, n_layers;
  int band, n_bands;          // m-tiles per band; band_first[b] = first work item of band b
  unsigned total_items;
  StackLayer L[XVEC_MAX_STACK];
  unsigned* counter;          // next work item (zeroed before the launch)
  unsigned* ready;            // [(n_layers-1)][m_tiles] completed epilogue-warp stores per tile (zeroed before the launch)
  const int* row_utt;
  const int* blk_slot_base;
  float* part;
  unsigned long long pol_a, pol_b, pol_y;
  int dbg;
  int runahead;               // scheduler run-ahead depth, 1 .. CREDIT_BARS - 1
  unsigned band_first[XVEC_STACK_MAX_BANDS + 1];
};

// item -> (layer [0,3) | n_tile [3,8) | m_tile [8,32)).  stack_dispatch() builds band_first[] with the same band_layer_range().
__host__ __device__ inline int band_layer_range(int band, int m_tiles, int b, int l, int* lo) {
  int a = b * band - l, z = (b + 1) * band - l;
  if (a < 0) a = 0;
  if (z > m_tiles) z = m_tiles;
  *lo = a;
  return z > a ? z - a : 0;
}
__host__ __device__ inline uint32_t decode_item(const StackParams& p, unsigned item, int& band_cursor) {
  while (item >= p.band_first[band_cursor + 1]) ++band_cursor;
  unsigned r = item - p.band_first[band_cursor];
  for (int l = 0; l < p.n_layers; ++l) {
    int lo;
    const unsigned nt = p.L[l].n_tiles;
    const unsigned cnt = band_layer_range(p.band, p.m_tiles, band_cursor, l, &lo) * nt;
    if (r < cnt) return static_cast<uint32_t>(l) | ((r % nt) << 3) | ((lo + r / nt) << 8);
    r -= cnt;
  }
  return ITEM_DONE;  // unreachable when the host table is consistent
}

// Developer switches (-DXVEC_DEBUG builds only; XVEC_STACK_DBG): 1 skip the dependency waits, 2 skip the completion
// signalling (only together with 1 — alone it makes the dependency warps spin until the watchdog fires, which is what
// tests/test_gpu_kernels.py::test_watchdog_code_is_readable uses), 4 skip the proxy fences (results are then undefined; timing
// experiments only), 8 short watchdog limit for the dependency spin (2^12 polls instead of 2^24), 16 the dependency watchdog
// reports its code and stops waiting instead of trapping (a trap is an Xid event on the box; the test only needs the code),
// 32 timing experiment: every activation slab is loaded twice (more shared-memory write traffic, same results), 64 timing
// experiment: no epilogue work at all.  (The round's earlier bits 32 / 128 — no activation / weight loads for n-tiles > 0 of
// single-tap layers — were removed after their measurements, profiles/r02_experiments.txt: with two producer warps they no longer
// ran reliably.)
// Debug builds also accumulate counters in the spare words of the control block (read by tools/stack_bench.py; units of 64
// cycles unless stated): 1 tiles whose dependency warp had to spin on a flag (count), 2 flag polls (count), 3 producer waiting
// for its dependency warp, 4 producer waiting for the work item, 5 MMA warp waiting for operands (explicit waits only),
// 6 MMA warp waiting for a free accumulator buffer, 12 / 13 (pooled tiles) and 14 / 15 (stored tiles) one epilogue warp per pair
// waiting for the accumulator / busy until it hands the buffer back, 7 the same warp after the release (stores, partials), 8 / 9 lifetime of CTA 0 in cycles / nanoseconds (SM clock), 10 time inside
// the tcgen05 step, 11 MMA warp waiting for the work item, per layer (units of 16): 16.. accumulator wait, 24.. whole tile, 32.. work-item
// wait, 40.. K loop, 48.. explicit operand waits inside it, 56.. time inside the fused issue + probe steps.
#ifdef XVEC_DEBUG
#define XVEC_SDBG(p, bit) ((p).dbg & (bit))
#define XVEC_CNT(...) __VA_ARGS__
#else
#define XVEC_SDBG(p, bit) 0
#define XVEC_CNT(...)
#endif

// Position in the operand ring: slot index + the parity of the number of times the ring has wrapped (the mbarrier phase).
template <int kSlots>
struct RingPos {
  int slot = 0;
  uint32_t ph = 0;
  __device__ __forceinline__ RingPos next() const {
    RingPos n = *this;
    if (++n.slot == kSlots) { n.slot = 0; n.ph ^= 1u; }
    return n;
  }
  __device__ __forceinline__ RingPos skip(int k) const {  // k <= kSlots positions further
    RingPos n = *this;
    n.slot += k;
    if (n.slot >= kSlots) { n.slot -= kSlots; n.ph ^= 1u; }
    return n;
  }
};

// K loop of one tile on the MMA warp (leader CTA, warp-uniform; see tdnn_gemm.cu): for every channel chunk one activation slab,
// for every tap one weight tile, popped from the ring in the producer's push order; the slab slot goes back to the producer
// with the last tap's commit, a weight slot with its own.
template <int kSlots>
struct MmaRing {
  RingPos<kSlots> pos;  // the next slot to pop
  uint32_t rdy = 0;     // bit0 next slab seen full, bit1 next weight tile seen full
};
// The per-layer constants of the K loop, read ONCE per tile into registers: every inline-asm step carries a "memory" clobber,
// so fields of the __grid_constant__ parameter block would otherwise be re-read (indexed constant loads, ~30-60 cycles each,
// on the single-warp critical path) in every K step.  Tap offsets (<= 8) are packed four bits each.
struct TileK {
  int cpt, taps;
  uint32_t tap_off4;
  __device__ __forceinline__ explicit TileK(const StackLayer& L) : cpt(L.cpt), taps(L.taps), tap_off4(L.tap_off4) {}
};
static_assert(XVEC_MAX_TAPS <= 8 && XVEC_STACK_MAX_TAP_OFFSET < 16, "tap offsets are packed into 8 x 4 bits");

// kDtype: operand element type of the layer (XVEC_F32: kind::tf32; XVEC_BF16 / XVEC_F16: kind::f16 in that format).
template <int kDtype, int kSlots>
__device__ __forceinline__ void mma_tile(uint32_t ring_addr, uint32_t full_addr, uint32_t empty_addr, uint32_t d, const TileK k, MmaRing<kSlots>& r,
                                         bool swap_ab, unsigned long long& c_wait, unsigned long long& c_step) {
  constexpr bool kTf32 = kDtype == XVEC_F32;
  constexpr uint32_t idesc = umma_idesc(umma_format(kDtype), BM, BN);
  const uint64_t desc0 = umma_desc_sw128(ring_addr);  // descriptor of slot 0, row 0
  uint32_t acc = 0;
  for (int ch = 0; ch < k.cpt; ++ch) {
    if (!(r.rdy & 1u)) {
      XVEC_CNT(const long long t0 = clock64();)
      mbar_wait_a(full_addr + 8u * r.pos.slot, r.pos.ph, 3);
      XVEC_CNT(c_wait += clock64() - t0;)
    }
    r.rdy &= ~1u;  // bit0 is set again by the last tap's probe of the NEXT slab
    const int a_slot = r.pos.slot;
    r.pos = r.pos.next();
    // operand descriptors are linear in the slot index and the tap's row shift (start address >> 4 in the low 14 bits; shared
    // memory ends below 256 KiB, so nothing carries out of the field): one multiply-add per operand instead of mask / shift / or
    const uint64_t slab_desc = desc0 + static_cast<uint32_t>(a_slot * (SLOT_BYTES >> 4));
    for (int tap = 0; tap < k.taps; ++tap) {
      if (!(r.rdy & 2u)) {
        XVEC_CNT(const long long t0 = clock64();)
        mbar_wait_a(full_addr + 8u * r.pos.slot, r.pos.ph, 3);
        XVEC_CNT(c_wait += clock64() - t0;)
      }
      tc_fence_after();
      const int b_slot = r.pos.slot;
      r.pos = r.pos.next();
      const uint64_t x_desc = slab_desc + ((k.tap_off4 >> (4 * tap)) & 15u) * (BK_BYTES >> 4);  // the slab, shifted by the tap's rows
      const uint64_t w_desc = desc0 + static_cast<uint32_t>(b_slot * (SLOT_BYTES >> 4));
      // swap_ab: the weights are the M operand and the frames the N operand, i.e. the accumulator holds the TRANSPOSED tile
      // (TMEM lane = channel, column = frame).  Both operands are 128 rows x 128 bytes K-major, so it is only a swap.
      const uint64_t da = swap_ab ? w_desc : x_desc;
      const uint64_t db = swap_ab ? x_desc : w_desc;
      // what the next step pops: after the last tap the next chunk's slab (also across a tile boundary) and then its first
      // weight tile, otherwise the next tap's weight tile
      const bool last_tap = tap == k.taps - 1;
      const RingPos<kSlots> pa = r.pos;
      const RingPos<kSlots> pb = last_tap ? r.pos.next() : r.pos;
      const uint32_t flags = STEP_COMMIT_B | STEP_PROBE_B | (last_tap ? (STEP_COMMIT_A | STEP_PROBE_A) : 0u);
      XVEC_CNT(const long long ts = clock64();)
      const uint32_t got = umma_step_pair<kTf32>(elect_one() ? 1u : 0u, d, da, db, idesc, acc, flags, empty_addr + 8u * a_slot,
                                                 empty_addr + 8u * b_slot, full_addr + 8u * pa.slot, pa.ph, full_addr + 8u * pb.slot, pb.ph);
      XVEC_CNT(c_step += clock64() - ts;)
      r.rdy = (got & 2u) | (last_tap ? (got & 1u) : 0u);
      acc = 1u;
    }
  }
}

// The K loop for the tap counts the x-vector stack has (1: TDNN1 in window form, TDNN4, TDNN5; 3: TDNN2, TDNN3): the tap loop is
// straight-line code with compile-time commit / probe sets (umma_step_fixed), the operand swap of the pooled layer is a template
// argument, single-tap layers unroll two chunks, so the descriptor arithmetic of one step is scheduled under the issue of its
// neighbour.  Same ring protocol and the same MMAs in the same order as mma_tile (which stays for every other tap count).
// Measured against mma_tile for every layer (B200, 256 x 300, us per launch): 277.0 vs 277.9 in bf16, 509.4 vs 512.0 in TF32.
template <int kDtype, int kSlots, int kTaps, bool kSwap>
__device__ __forceinline__ void mma_tile_fixed(uint32_t ring_addr, uint32_t full_addr, uint32_t empty_addr, uint32_t d, const TileK k,
                                               MmaRing<kSlots>& r, unsigned long long& c_wait, unsigned long long& c_step) {
  constexpr bool kTf32 = kDtype == XVEC_F32;
  constexpr uint32_t idesc = umma_idesc(umma_format(kDtype), BM, BN);
  const uint64_t desc0 = umma_desc_sw128(ring_addr);  // descriptor of slot 0, row 0
  const uint32_t lo0 = static_cast<uint32_t>(desc0), hi = static_cast<uint32_t>(desc0 >> 32);
  const uint32_t elected = elect_one() ? 1u : 0u;  // the same lane issues every MMA and commit of the tile
  uint32_t acc = 0;
#pragma unroll(kTaps == 1 ? 2 : 1)
  for (int ch = 0; ch < k.cpt; ++ch) {
    if (!(r.rdy & 1u)) {
      XVEC_CNT(const long long t0 = clock64();)
      mbar_wait_a(full_addr + 8u * r.pos.slot, r.pos.ph, 3);
      XVEC_CNT(c_wait += clock64() - t0;)
    }
    r.rdy &= ~1u;
    const int a_slot = r.pos.slot;
    r.pos = r.pos.next();
    const uint32_t slab_lo = lo0 + static_cast<uint32_t>(a_slot * (SLOT_BYTES >> 4));
    auto tap_step = [&](auto tap_c) {
      constexpr int tap = decltype(tap_c)::value;
      constexpr bool last_tap = tap == kTaps - 1;
      if (!(r.rdy & 2u)) {
        XVEC_CNT(const long long t0 = clock64();)
        mbar_wait_a(full_addr + 8u * r.pos.slot, r.pos.ph, 3);
        XVEC_CNT(c_wait += clock64() - t0;)
      }
      tc_fence_after();
      const int b_slot = r.pos.slot;
      r.pos = r.pos.next();
      const uint32_t x_lo = slab_lo + ((k.tap_off4 >> (4 * tap)) & 15u) * (BK_BYTES >> 4);
      const uint32_t w_lo = lo0 + static_cast<uint32_t>(b_slot * (SLOT_BYTES >> 4));
      const RingPos<kSlots> pa = r.pos;
      const RingPos<kSlots> pb = last_tap ? r.pos.next() : r.pos;
      XVEC_CNT(const long long ts = clock64();)
      const uint32_t got = umma_step_fixed<kTf32, last_tap>(elected, d, kSwap ? w_lo : x_lo, kSwap ? x_lo : w_lo, hi, idesc, acc,
                                                            empty_addr + 8u * a_slot, empty_addr + 8u * b_slot, full_addr + 8u * pa.slot, pa.ph,
                                                            full_addr + 8u * pb.slot, pb.ph);
      XVEC_CNT(c_step += clock64() - ts;)
      r.rdy = last_tap ? got : (got & 2u);
      acc = 1u;
    };
    static_assert(kTaps == 1 || kTaps == 3, "instantiated for the tap counts of the x-vector stack");
    tap_step(std::integral_constant<int, 0>{});
    if constexpr (kTaps == 3) {
      tap_step(std::integral_constant<int, 1>{});
      tap_step(std::integral_constant<int, 2>{});
    }
  }
}

template <bool kAllTf32>
constexpr int stack_smem_bytes() { return 1024 + StackCfg<kAllTf32>::SLOTS * SLOT_BYTES + EPI_WARPS * StackCfg<kAllTf32>::STAGE_BYTES; }
static_assert(stack_smem_bytes<false>() <= 227 * 1024 - 1024 && stack_smem_bytes<true>() <= 227 * 1024 - 1024,
              "operand ring + store staging (+ 1 KiB of static barriers) exceed the 227 KiB of shared memory a CTA can have");
constexpr int STACK_SMEM_LEFT_FOR_TAIL = 20 * 1024;  // what a co-resident tail kernel may use (fc_small.cu takes 5 KiB)
static_assert(228 * 1024 - stack_smem_bytes<false>() - 2048 - 2 * 1024 >= STACK_SMEM_LEFT_FOR_TAIL &&
              228 * 1024 - stack_smem_bytes<true>() - 2048 - 2 * 1024 >= STACK_SMEM_LEFT_FOR_TAIL,
              "the stack kernel must leave room on the SM for the tail kernels of the previous batch");

// kAct: the activation dtype of layers 1.. (XVEC_F32, XVEC_BF16 or XVEC_F16).  The two 16-bit kinds share everything but the
// UMMA operand format and the convert of the store epilogue.
template <int kAct>
__global__ void __maxnreg__(STACK_MAX_REGS)
tdnn_stack_kernel(const __grid_constant__ StackMaps maps, const __grid_constant__ StackParams p) {
  constexpr bool kAllTf32 = kAct == XVEC_F32;
  extern __shared__ uint8_t smem_raw[];
  constexpr int RING_SLOTS = StackCfg<kAllTf32>::SLOTS;
  __shared__ uint64_t full_bar[RING_SLOTS], empty_bar[RING_SLOTS], tfull_bar[2], tempty_bar[2];
  __shared__ uint64_t sfull_bar[SCHED_SLOTS], sempty_bar[SCHED_SLOTS], dep_bar[SCHED_SLOTS], credit_bar[CREDIT_BARS];
  __shared__ uint32_t sched_item[SCHED_SLOTS];
  __shared__ uint32_t pub_cnt[4];  // epilogue warps that have completed the stores of a tile, per tile in flight (free-running, see publish)
  __shared__ uint32_t tmem_base_smem;

  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // SWIZZLE_128B tiles: 1024-byte alignment
  uint8_t* epi_smem = base + RING_SLOTS * SLOT_BYTES;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();  // 0 = leader of the pair

  if (warp == 0 && lane == 0) {
    for (int c = 0; c < 4; ++c) pub_cnt[c] = 0;
    for (int l = 0; l < p.n_layers; ++l) {
      tma_prefetch_desc(&maps.a[l]);
      tma_prefetch_desc(&maps.b[l]);
      if (l + 1 < p.n_layers) tma_prefetch_desc(&maps.y[l]);
    }
    for (int s = 0; s < RING_SLOTS; ++s) {
      mbar_init(&full_bar[s], 1);   // leader's arrive.expect_tx (bytes of both CTAs)
      mbar_init(&empty_bar[s], 1);  // leader's multicast commit (a weight slot: its own MMA group; a slab slot: the chunk's last tap)
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);               // leader's multicast commit
      mbar_init(&tempty_bar[b], 2 * EPI_WARPS);  // one arrive per epilogue warp of both CTAs (on the leader's barrier)
    }
    for (int s = 0; s < SCHED_SLOTS; ++s) {
      mbar_init(&sfull_bar[s], 1);                 // the scheduler's arrive (local in the leader, remote in the peer)
      mbar_init(&sempty_bar[s], SCHED_CONSUMERS);  // every consumer of both CTAs, on the leader's barrier
      mbar_init(&dep_bar[s], 1);                   // this CTA's dependency warp
    }
    for (int c = 0; c < CREDIT_BARS; ++c) mbar_init(&credit_bar[c], 1);  // leader's producer: tile j arrives on credit_bar[j % CREDIT_BARS]
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_pair<TMEM_COLS>(&tmem_base_smem);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  // shared-memory addresses the hot loops index by slot (see mbar_wait_a): the ring, its barriers, the leader's full barriers
  const uint32_t ring_addr = smem_u32(base), full_addr = smem_u32(full_bar), empty_addr = smem_u32(empty_bar);
  const uint32_t full_leader = mapa_u32(full_addr, 0);
  XVEC_CNT(long long dbg_c0 = clock64(); unsigned long long dbg_t0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t0));)

  // Consumer side of the work-item ring: wait for entry `it`, read it, hand the slot back to the scheduler.
  auto ring_read = [&](int it) -> uint32_t {
    const int slot = it % SCHED_SLOTS;
    const uint32_t sph = (it / SCHED_SLOTS) & 1u;
    mbar_wait(&sfull_bar[slot], sph, 6);  // leader: the scheduler's arrive; peer: the 4 bytes of the scheduler's st.async have landed
    const uint32_t item = *reinterpret_cast<volatile uint32_t*>(&sched_item[slot]);
    __syncwarp();
    if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&sempty_bar[slot]), 0));
    return item;
  };

  if (warp == 0 || warp == WPROD_WARP) {
    // ------------------------------------------------------------------ TMA producers (both CTAs): warp 0 loads the activation
    // slabs, warp WPROD_WARP the weight tiles.  Round 2: once the MMA warp's instruction stream was out of the way, ONE producer
    // warp issuing both operands (~120 instructions and two TMA issues per K step) could not keep the ring full — the MMA warp
    // waited ~2 500 cycles per TDNN2/3 tile for operands.  Both warps walk the same ring positions (per chunk: slab, then one
    // weight tile per tap) and each fills its own; they never talk to each other.
    // Per tile: read the work item (published by the scheduler warp while the previous tile was loading); the slab warp checks
    // that this CTA's dependency warp has resolved the tile's inputs (weights have no dependencies) and tells the scheduler that
    // the tile has started; then the K loop.
    const bool slabs = warp == 0;
    static_assert(XVEC_MAX_TAPS + 1 <= StackCfg<kAllTf32>::SLOTS, "RingPos::skip wraps at most once");
    RingPos<RING_SLOTS> pos;  // ring position of the current chunk's slab
    uint32_t rdy = 0;         // the slot this warp fills next was seen free
    XVEC_CNT(unsigned long long c_fw = 0, c_pub = 0;)
    for (int it = 0;; ++it) {
      XVEC_CNT(long long t0 = clock64();)
      const uint32_t item = ring_read(it);
      XVEC_CNT(c_pub += clock64() - t0; t0 = clock64();)
      if (item == ITEM_DONE) break;
      if (slabs) {
        mbar_wait(&dep_bar[it % SCHED_SLOTS], (it / SCHED_SLOTS) & 1u, 7);
        XVEC_CNT(c_fw += clock64() - t0;)
        if (rank == 0 && lane == 0) mbar_arrive(&credit_bar[it % CREDIT_BARS]);  // tile `it` has started: the scheduler may draw item it + run-ahead
      }
      const int layer = item & 7u, nt = (item >> 3) & 31u, mt = item >> 8;
      const StackLayer& L = p.L[layer];
      // everything the K loop needs from the parameter block, in registers (the asm steps clobber "memory": see TileK)
      const int cpt = L.cpt, taps = L.taps, n_pad = L.n_pad;
      const uint32_t is_leader = rank == 0 ? 1u : 0u;
      if (slabs) {
        const int bke = (kAllTf32 || L.tf32) ? 32 : 64;  // elements per 128-byte chunk
        const int m0 = mt * BM + static_cast<int>(rank) * BM_CTA;
        const CUtensorMap* ma = &maps.a[layer];
        // timing experiment (debug bit 32): every activation slab is loaded TWICE into its slot (same bytes, same place; the barrier
        // is armed for both) — +50 % / +26 % shared-memory write traffic on single-tap / 3-tap layers, results unchanged
        const bool twice = XVEC_SDBG(p, 32);
        const uint32_t slab_tx = (twice ? 4u : 2u) * static_cast<uint32_t>(L.slab_rows) * BK_BYTES;  // bytes of both CTAs' slabs
        const unsigned long long pol_a = p.pol_a;
        for (int ch = 0; ch < cpt; ++ch) {
          if (!rdy) mbar_wait_a(empty_addr + 8u * pos.slot, pos.ph ^ 1u, 1);
          const RingPos<RING_SLOTS> nxt = pos.skip(1 + taps);  // the next chunk's slab, also across a tile boundary
          rdy = tma_step_one(elect_one() ? 1u : 0u, is_leader, 1u, full_addr + 8u * pos.slot, full_leader + 8u * pos.slot, slab_tx,
                             ring_addr + pos.slot * SLOT_BYTES, ma, ch * bke, m0, pol_a, empty_addr + 8u * nxt.slot, nxt.ph ^ 1u);
          if (twice && elect_one()) tma_load_2d_pair(full_leader + 8u * pos.slot, ring_addr + pos.slot * SLOT_BYTES, ma, ch * bke, m0, pol_a);
          pos = nxt;
        }
      } else {
        const int n0 = nt * BN + static_cast<int>(rank) * BN_CTA;
        const CUtensorMap* mb = &maps.b[layer];
        const unsigned long long pol_b = p.pol_b;
        for (int ch = 0; ch < cpt; ++ch) {
          RingPos<RING_SLOTS> pb = pos.next();  // the chunk's first weight tile sits behind its slab
          int b_row = ch * n_pad + n0;          // row of the (tap, chunk) tile in the chunk-major packed matrix: (tap * cpt + ch) * n_pad + n0
          for (int tap = 0; tap < taps; ++tap, b_row += cpt * n_pad) {
            if (!rdy) mbar_wait_a(empty_addr + 8u * pb.slot, pb.ph ^ 1u, 1);
            const RingPos<RING_SLOTS> nxt = tap == taps - 1 ? pb.skip(2) : pb.next();  // after the last tap: over the next chunk's slab
            rdy = tma_step_one(elect_one() ? 1u : 0u, is_leader, 1u, full_addr + 8u * pb.slot, full_leader + 8u * pb.slot, 2u * B_BYTES,
                               ring_addr + pb.slot * SLOT_BYTES, mb, 0, b_row, pol_b, empty_addr + 8u * nxt.slot, nxt.ph ^ 1u);
            pb = nxt;
          }
          pos = pos.skip(1 + taps);
        }
      }
    }
    XVEC_CNT(if (slabs && lane == 0) {
      atomicAdd(p.counter + 3, static_cast<unsigned>(c_fw >> 6));
      atomicAdd(p.counter + 4, static_cast<unsigned>(c_pub >> 6));
    })
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (rank == 0) {
      MmaRing<RING_SLOTS> ring;
      unsigned long long c_full = 0, c_step = 0;  // debug counters (explicit operand waits / time inside the issue step)
      XVEC_CNT(unsigned long long c_tempty = 0, c_ring = 0;)
      for (int it = 0;; ++it) {
        XVEC_CNT(const long long tr = clock64();)
        const uint32_t item = ring_read(it);
        XVEC_CNT(c_ring += clock64() - tr;)
        if (item == ITEM_DONE) break;
        XVEC_CNT(if (lane == 0) atomicAdd(p.counter + 32 + (item & 7u), static_cast<unsigned>((clock64() - tr) >> 4));)  // work-item wait per layer
        const StackLayer& L = p.L[item & 7u];
        const int buf = it & 1;
        const uint32_t use = (it >> 1) & 1;
        XVEC_CNT(const long long t0 = clock64();)
        mbar_wait(&tempty_bar[buf], use ^ 1u, 2);  // both CTAs' epilogues have drained this accumulator buffer
        XVEC_CNT(c_tempty += clock64() - t0; const int dl = item & 7u; if (lane == 0) atomicAdd(p.counter + 16 + dl, static_cast<unsigned>((clock64() - t0) >> 4));)
        const uint32_t d = tmem_base + buf * BN;
        const bool pooled = static_cast<int>(item & 7u) == p.n_layers - 1;  // last layer: transposed accumulator (see the epilogue)
        XVEC_CNT(const long long tk = clock64(); const unsigned long long full0 = c_full, step0 = c_step;)
        const TileK tk_(L);
        auto run = [&](auto dt_c) {
          constexpr int dt = decltype(dt_c)::value;  // operand dtype of this layer
          if (tk_.taps == 1) {
            if (pooled) mma_tile_fixed<dt, RING_SLOTS, 1, true>(ring_addr, full_addr, empty_addr, d, tk_, ring, c_full, c_step);
            else mma_tile_fixed<dt, RING_SLOTS, 1, false>(ring_addr, full_addr, empty_addr, d, tk_, ring, c_full, c_step);
          } else if (tk_.taps == 3) {
            if (pooled) mma_tile_fixed<dt, RING_SLOTS, 3, true>(ring_addr, full_addr, empty_addr, d, tk_, ring, c_full, c_step);
            else mma_tile_fixed<dt, RING_SLOTS, 3, false>(ring_addr, full_addr, empty_addr, d, tk_, ring, c_full, c_step);
          } else {
            mma_tile<dt, RING_SLOTS>(ring_addr, full_addr, empty_addr, d, tk_, ring, pooled, c_full, c_step);
          }
        };
        if constexpr (kAllTf32) {
          run(std::integral_constant<int, XVEC_F32>{});
        } else {
          if (L.tf32) run(std::integral_constant<int, XVEC_F32>{});
          else run(std::integral_constant<int, kAct>{});
        }
        XVEC_CNT(if (lane == 0) {  // per layer: whole K loop, explicit operand waits, time inside the fused issue + probe step
          atomicAdd(p.counter + 40 + (item & 7u), static_cast<unsigned>((clock64() - tk) >> 4));
          atomicAdd(p.counter + 48 + (item & 7u), static_cast<unsigned>((c_full - full0) >> 4));
          atomicAdd(p.counter + 56 + (item & 7u), static_cast<unsigned>((c_step - step0) >> 4));
        })
        if (elect_one()) umma_commit_pair(&tfull_bar[buf], 0x3);  // accumulator complete (both CTAs' epilogues)
        __syncwarp();
        XVEC_CNT(if (lane == 0) atomicAdd(p.counter + 24 + (item & 7u), static_cast<unsigned>((clock64() - tr) >> 4));)
      }
      XVEC_CNT(if (lane == 0) {
        atomicAdd(p.counter + 5, static_cast<unsigned>(c_full >> 6));
        atomicAdd(p.counter + 6, static_cast<unsigned>(c_tempty >> 6));
        atomicAdd(p.counter + 10, static_cast<unsigned>(c_step >> 6));
        atomicAdd(p.counter + 11, static_cast<unsigned>(c_ring >> 6));
      })
    }
  } else if (warp == DEP_WARP) {
    // ------------------------------------------------------------------ scheduler (leader) + dependency warp (both CTAs)
    // Leader: draws work items (atomicAdd on the global counter), decodes them and publishes them in the ring of both CTAs —
    // item `it` as soon as the producer has started tile it - D (credit_bar), D = p.runahead (1: a pair never holds more than one
    // item it has not begun).  Measured on B200 (256 x 300, bf16): D = 1, 2, 3 give the same tile times and the same launch time
    // (297.7 / 298.3 / 299.6 us) — the chain "tile started -> atomic -> decode -> publication -> dependency acquire" is not what
    // the K = 512 tiles of TDNN4/5 wait for.  Near the end of the queue (fewer than (D + 1) x pairs items left) the depth falls
    // back to 1, so that no pair sits on unstarted items while others have run out of work.
    // Both CTAs: resolve the inter-layer dependencies of every item ahead of the producer: lanes 0..2 poll (ld.acquire.gpu)
    // the flags of the tiles the item touches — reads: this CTA's 128 rows + the taps' reach (rank 1 runs into tile mt+1);
    // writes: rows whose old contents (two layers back, same ping-pong buffer) tiles mt-1 and mt of the previous layer were
    // reading — then fence.proxy.async (flag in the generic proxy -> tile data in the async proxy), one arrive on dep_bar.
    XVEC_CNT(unsigned long long c_spun = 0, c_polls = 0;)
    int band_cursor = 0;
    unsigned raw_prev = 0;  // the last item this pair drew
    for (int it = 0;; ++it) {
      uint32_t item;
      if (rank == 0) {
        const int slot = it % SCHED_SLOTS;
        const uint32_t sph = (it / SCHED_SLOTS) & 1u;
        {
          const int depth = (raw_prev + static_cast<unsigned>(p.runahead + 1) * (gridDim.x >> 1) >= p.total_items) ? 1 : p.runahead;
          const int j = it - depth;  // the tile whose start is awaited; tile j arrives in phase j / CREDIT_BARS of credit_bar[j % CREDIT_BARS]
          if (j >= 0) mbar_wait(&credit_bar[j % CREDIT_BARS], static_cast<uint32_t>(j / CREDIT_BARS) & 1u, 8);
        }
        unsigned raw = 0;
        if (lane == 0) raw = atomicAdd(p.counter, 1u);
        raw = __shfl_sync(0xffffffffu, raw, 0);
        raw_prev = raw;
        item = raw < p.total_items ? decode_item(p, raw, band_cursor) : ITEM_DONE;
        mbar_wait(&sempty_bar[slot], sph ^ 1u, 5);
        if (lane == 0) {
          sched_item[slot] = item;
          mbar_arrive(&sfull_bar[slot]);
          const uint32_t peer_bar = mapa_u32(smem_u32(&sfull_bar[slot]), 1);
          mbar_arrive_expect_tx_cluster(peer_bar, 4);
          st_async_cluster_u32(mapa_u32(smem_u32(&sched_item[slot]), 1), item, peer_bar);
        }
        __syncwarp();
      } else {
        item = ring_read(it);
      }
      if (item == ITEM_DONE) break;
      const int layer = item & 7u, mt = item >> 8;
      if (layer > 0 && !XVEC_SDBG(p, 1)) {
        const unsigned target = static_cast<unsigned>(p.L[layer - 1].n_tiles) * 2u * EPI_WARPS;
        const int d = lane - 1;  // lanes 0..2 -> tiles mt-1, mt, mt+1
        const bool mine = lane < 3 && mt + d >= 0 && mt + d < p.m_tiles && (d < 1 || rank == 1);
        const unsigned* f = p.ready + static_cast<size_t>(layer - 1) * p.m_tiles + (mine ? mt + d : mt);
        uint32_t spins = 0;
        while (__any_sync(0xffffffffu, mine && ld_acquire_gpu_u32(f) < target)) {
          if (++spins > (XVEC_SDBG(p, 8) ? (1u << 12) : (1u << 24))) {
            if (XVEC_SDBG(p, 16)) {  // test mode: report, do not trap, stop waiting (the results are then garbage)
              watchdog_report(7u);
              break;
            }
            watchdog_trip(7u);
          }
        }
        XVEC_CNT(c_polls += spins; c_spun += spins ? 1 : 0;)
        if (!XVEC_SDBG(p, 4)) fence_proxy_async_global();
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&dep_bar[it % SCHED_SLOTS]);
    }
    XVEC_CNT(if (lane == 0) {
      atomicAdd(p.counter + 1, static_cast<unsigned>(c_spun));
      atomicAdd(p.counter + 2, static_cast<unsigned>(c_polls));
    })
  } else {
    // ------------------------------------------------------------------ epilogue warps (both CTAs, 128 rows each)
    const int q = warp & 3;                         // TMEM lane quarter this warp may read
    const int cbeg = ((warp - 2) >> 2) * (BN / 2);  // this warp's half of the tile's columns
    uint8_t* out_stage = epi_smem + (warp - 2) * StackCfg<kAllTf32>::STAGE_BYTES;
    int store_seq = 0;
    // Store staging: one TMA-store box per tcgen05.ld chunk (32 rows x 32 columns).  16-bit: 64-byte rows (SWIZZLE_64B), the warp's
    // 4 KiB hold two boxes, so staging chunk k+1 overlaps the store of chunk k; float32: 128-byte rows, one box.
    constexpr int BOX_W = kAllTf32 ? 128 : 64;                              // bytes per box row
    constexpr int BOX_BYTES = 32 * BOX_W;
    constexpr int NBUF = StackCfg<kAllTf32>::NBUF;                          // boxes in flight per warp
    constexpr int BOXES = (BN / 2) / 32;                                    // boxes (= bulk groups) per tile and warp
    unsigned* pend = nullptr;  // ready counter of the last stored tile whose completion has not been published yet (warp-uniform)
    int pend_it = 0;           // ... and the work-item index it was processed at (all epilogue warps of a CTA see the same sequence)
    // Publish `pend`: lane 0 owns the warp's bulk groups; once they are complete the tile's rows are in global memory.  The eight
    // epilogue warps of a CTA count themselves in shared memory (acq_rel at CTA scope), and the LAST one to arrive publishes for
    // all: one fence + one red.release.gpu (+ 8) per tile and CTA instead of eight — a gpu-scope release is a MEMBAR.ALL.GPU
    // (measured on a B200: 262.3 vs 264.5 us per launch against one release per warp; 256 x 300, bf16).
    // A tile's counter is free-running (8 arrivals per use; at most three stored tiles of a CTA are unpublished at any time: a
    // warp publishes tile i before it leaves tile i + 1, and nobody enters tile i + 2 before every warp has released tile i).
    // kAll: wait for every bulk group of this thread; otherwise for all but the BOXES most recent (the current tile's).
    auto publish = [&](bool all) {
      if (lane == 0 && !XVEC_SDBG(p, 2)) {
        if (all) tma_store_wait_all();
        else tma_store_wait_done<BOXES>();
        if ((atom_add_acq_rel_cta_shared_u32(smem_u32(&pub_cnt[pend_it & 3]), 1u) & (EPI_WARPS - 1)) == EPI_WARPS - 1) {
          if (!XVEC_SDBG(p, 4)) fence_proxy_async_global();
          red_release_gpu_add_u32(pend, static_cast<uint32_t>(EPI_WARPS));
        }
      }
      pend = nullptr;
    };
    auto flush = [&]() { publish(true); };
    // The epilogue warps' per-tile chain — read the work item (~500 cycles), wait for the accumulator, fetch the pooling
    // bookkeeping from L2 (~700 cycles), then four dependent tcgen05.ld + math rounds — is what the MMA warp ends up waiting
    // for once the mainloop is fast (round 2).  So the chain is software-pipelined: item `it` is in hand when iteration `it`
    // starts (read during iteration it - 1), its global loads are issued first, then item it + 1 is read while they are in
    // flight, and only then does the warp wait for the accumulator.
    // Never sleep on future work with an unpublished tile: a consumer of that tile may be what the future work waits for.
    XVEC_CNT(unsigned long long e_wait[2] = {0, 0}, e_busy[2] = {0, 0}, e_tail = 0; long long e_t0 = 0, e_t1 = 0;)
    uint32_t item = ring_read(0);
    for (int it = 0;; ++it) {
      if (item == ITEM_DONE) break;
      const int layer = item & 7u, nt = (item >> 3) & 31u, mt = item >> 8;
      const StackLayer& L = p.L[layer];
      const int m0 = mt * BM + static_cast<int>(rank) * BM_CTA;
      const int n0 = nt * BN;
      const int buf = it & 1;
      const uint32_t use = (it >> 1) & 1;
      const bool pooled_tile = layer == p.n_layers - 1;
      const PoolArgs pa{p.rows, L.n, L.bias, p.row_utt, p.blk_slot_base, p.part};
      const int pch = n0 + static_cast<int>(rank) * BN_CTA + q * 32 + lane, pf0 = mt * BM + cbeg;
      PoolPrefetch pre{};
      if (pooled_tile) pre = pool_prefetch(pa, pch, pf0, lane);
      uint32_t next_item;
      {
        const int nslot = (it + 1) % SCHED_SLOTS;
        const uint32_t nph = ((it + 1) / SCHED_SLOTS) & 1u;
        if (pend && !mbar_test_wait(&sfull_bar[nslot], nph)) flush();
        next_item = ring_read(it + 1);
      }
      if (pend && !mbar_test_wait(&tfull_bar[buf], use)) flush();
      XVEC_CNT(e_t0 = clock64();)
      mbar_wait(&tfull_bar[buf], use, 4);
      tc_fence_after();
      XVEC_CNT(e_t1 = clock64(); e_wait[pooled_tile ? 0 : 1] += e_t1 - e_t0;)
      const uint32_t tbase = tmem_base + buf * BN + (static_cast<uint32_t>(q * 32) << 16);
      const int row0 = m0 + q * 32;
      bool released = false;
      auto release_tmem = [&]() {  // right after this warp's LAST tcgen05.ld of the tile
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[buf]), 0));
        released = true;
        XVEC_CNT(e_t0 = clock64(); e_busy[pooled_tile ? 0 : 1] += e_t0 - e_t1;)
      };

      if (XVEC_SDBG(p, 64)) {  // timing experiment: no epilogue at all (no tcgen05.ld, no math, no stores); completion is still published
        release_tmem();
        if (pend) flush();
        if (layer != p.n_layers - 1) {
          pend = p.ready + static_cast<size_t>(layer) * p.m_tiles + mt;
          pend_it = it;
        }
        item = next_item;
        continue;
      }
      if (pooled_tile) {
        // Last layer: statistics-pooling partials; nothing is stored and nobody waits for this tile.  The accumulator is
        // TRANSPOSED (the MMA warp swapped the operands): TMEM lane = output channel, column = frame (gemm_tile.cuh).
        pool_epilogue_tile_t(pa, pre, tmem_base + buf * BN + (static_cast<uint32_t>(q * 32) << 16) + cbeg, pch, pf0, lane, release_tmem);
        if (!released) release_tmem();
        if (pend) flush();  // its stores were issued a whole tile ago
      } else {
        const CUtensorMap* my = &maps.y[layer];
        // tcgen05.ld of chunk k+1 is in flight while chunk k is converted, staged and stored
        uint32_t va[32], vb[32];
        tmem_ld_32x32(tbase + cbeg, va);
        tmem_ld_wait();
#pragma unroll
        for (int k = 0; k < BOXES; ++k) {
          uint32_t(&v)[32] = (k & 1) ? vb : va;
          if (k + 1 < BOXES) tmem_ld_32x32(tbase + cbeg + 32 * (k + 1), (k & 1) ? va : vb);
          uint8_t* ob = out_stage + (store_seq % NBUF) * BOX_BYTES;
          const int col0 = n0 + cbeg + k * 32;
          // r = relu(acc + bias') — every BatchNorm is folded forward into the next layer's weights (xvector.py)
          float o[32];
          const float4* bp = reinterpret_cast<const float4*>(L.bias + col0);
#pragma unroll
          for (int j4 = 0; j4 < 32; j4 += 4) {
            const float4 bb = __ldg(bp + (j4 >> 2));
            const float2 a = __fadd2_rn(make_float2(__uint_as_float(v[j4 + 0]), __uint_as_float(v[j4 + 1])), make_float2(bb.x, bb.y));
            const float2 d = __fadd2_rn(make_float2(__uint_as_float(v[j4 + 2]), __uint_as_float(v[j4 + 3])), make_float2(bb.z, bb.w));
            o[j4 + 0] = a.x; o[j4 + 1] = a.y; o[j4 + 2] = d.x; o[j4 + 3] = d.y;
          }
          // the store that last used this box must have read it — checked only now, after the bias / ReLU math of this chunk
          // (measured on a B200: 263.7 vs 264.3 us per launch against the wait before the math; 256 x 300, bf16)
          if (lane == 0) tma_store_wait_read<NBUF - 1>();
          __syncwarp();
          // row `lane` of the box, 16-byte pieces XOR-swizzled like the tensor map's swizzle mode expects
          uint8_t* orow = ob + lane * BOX_W;
          if constexpr (!kAllTf32) {  // SWIZZLE_64B: piece index ^ address bits [7,9) = (row / 2) % 4
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 w;
              w.x = pack16x2_relu<kAct>(o[8 * j + 0], o[8 * j + 1]);
              w.y = pack16x2_relu<kAct>(o[8 * j + 2], o[8 * j + 3]);
              w.z = pack16x2_relu<kAct>(o[8 * j + 4], o[8 * j + 5]);
              w.w = pack16x2_relu<kAct>(o[8 * j + 6], o[8 * j + 7]);
              *reinterpret_cast<uint4*>(orow + ((j ^ ((lane >> 1) & 3)) << 4)) = w;
            }
          } else {                    // SWIZZLE_128B: piece index ^ address bits [7,10) = row % 8
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 w = make_float4(fmaxf(o[4 * j], 0.f), fmaxf(o[4 * j + 1], 0.f), fmaxf(o[4 * j + 2], 0.f), fmaxf(o[4 * j + 3], 0.f));
              *reinterpret_cast<float4*>(orow + ((j ^ (lane & 7)) << 4)) = w;
            }
          }
          if (k + 1 < BOXES) tmem_ld_wait();
          if (k == BOXES - 2) release_tmem();  // the last tcgen05.ld of the tile has landed
          fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
          __syncwarp();
          if (lane == 0) {
            if (row0 < p.rows) tma_store_2d(my, ob, col0, row0, p.pol_y);  // rows past the matrix are clipped
            tma_store_commit();  // one group per box, also when nothing was stored, so that the group arithmetic below holds
          }
          ++store_seq;
        }
        if (pend) publish(false);  // the previous stored tile's groups are older than this tile's BOXES groups
        pend = p.ready + static_cast<size_t>(layer) * p.m_tiles + mt;
        pend_it = it;
      }
      XVEC_CNT(e_tail += clock64() - e_t0;)
      item = next_item;
    }
    // which epilogue warp reports: XVEC_STACK_DBG bits [8,12) = warp (0: warp 2), bit 13 = CTA rank of the pair
    XVEC_CNT(if (static_cast<int>(rank) == ((p.dbg >> 13) & 1) && warp == (((p.dbg >> 8) & 15) ? ((p.dbg >> 8) & 15) : 2) && lane == 0) {  // one epilogue warp per pair: accumulator wait / busy until the release / after it (units of 64 cycles)
      atomicAdd(p.counter + 12, static_cast<unsigned>(e_wait[0] >> 6));
      atomicAdd(p.counter + 13, static_cast<unsigned>(e_busy[0] >> 6));
      atomicAdd(p.counter + 14, static_cast<unsigned>(e_wait[1] >> 6));
      atomicAdd(p.counter + 15, static_cast<unsigned>(e_busy[1] >> 6));
      atomicAdd(p.counter + 7, static_cast<unsigned>(e_tail >> 6));
    })
    if (pend) flush();
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  XVEC_CNT(if (blockIdx.x == 0 && threadIdx.x == 0) {  // SM clock during the launch: cycles (>>6) and nanoseconds of CTA 0
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    p.counter[8] = static_cast<unsigned>((clock64() - dbg_c0) >> 6);
    p.counter[9] = static_cast<unsigned>(t1 - dbg_t0);
  })
  cluster_sync_all();  // the peer may still be reading our smem / signalling our barriers until here
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair<TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ host side
// Band height.  Two opposing effects, both measured on B200 (256 x 300 frames = 300 m-tiles, bf16, 74 pairs):
//   * producers run 3-4 tiles ahead of the published completions, so an item's inputs are only certain to be complete when they
//     were drawn >= ~4 x pairs items earlier — bands of 100 / 148 m-tiles stall (364 us sustained, dependency warps spinning);
//   * a band's activations (band x 256 KiB per ping-pong buffer in bf16: 2 x 43.5 MB at 170 m-tiles, of 126 MB of L2) stay in
//     L2 between the layers when the band is short enough,
//     which saves the HBM round trip of every activation and the power that goes with it — the kernel runs at the 1000 W cap,
//     so this is throughput: one band 294 / 336 us (burst / sustained), bands of 160-170: 278 / 322 us, 180-200: 282-284 /
//     326-328 us, 225: 292 / 332 us, 250: 311 / 347 us.  64 x 6000 frames (1500 m-tiles): 1474 -> 1382 us; 437 x 300: 519 -> 467 us.
// Hence equal bands of about 2.3 x pairs m-tiles.  `want` > 0 (xvec_tdnn_stack's band argument; tests and tools) overrides.
static int pick_band(int m_tiles, int n_layers, int pairs, int want) {
  int band = want;
  if (band <= 0) {
    // equal bands of about 2.3 x pairs m-tiles: a short last band runs its five layers as a serial chain of a few tiles each
    // (437 x 300 frames = 512 m-tiles: bands 170+170+170+6 take 525 us, 3 x 172 take 487 us)
    const int target = (23 * pairs + 5) / 10, span = m_tiles + n_layers - 1;
    const int n_bands = span < target ? 1 : (span + target / 2) / target;
    band = (span + n_bands - 1) / n_bands;
  }
  if (band < n_layers) band = n_layers;
  while ((m_tiles + n_layers - 1 + band - 1) / band > XVEC_STACK_MAX_BANDS) band *= 2;
  return band;
}

// Work-item order of a stack whose m_tiles / n_layers / L[].n_tiles are set: band table + total (see decode_item).
static int fill_schedule(StackParams& p, int band) {
  p.band = band;
  p.n_bands = (p.m_tiles + p.n_layers - 1 + p.band - 1) / p.band;
  if (p.n_bands > XVEC_STACK_MAX_BANDS) return set_error(XVEC_E_ARG, "internal: too many bands");
  unsigned acc = 0;
  int64_t items_per_mtile = 0;
  for (int l = 0; l < p.n_layers; ++l) items_per_mtile += p.L[l].n_tiles;
  for (int b = 0; b < p.n_bands; ++b) {
    p.band_first[b] = acc;
    for (int l = 0; l < p.n_layers; ++l) {
      int lo;
      acc += static_cast<unsigned>(band_layer_range(p.band, p.m_tiles, b, l, &lo)) * p.L[l].n_tiles;
    }
  }
  p.band_first[p.n_bands] = acc;
  if (static_cast<int64_t>(acc) != items_per_mtile * p.m_tiles) return set_error(XVEC_E_ARG, "internal: band table does not cover the stack");
  p.total_items = acc;
  return XVEC_OK;
}

// Host-side replay of the device scheduler's decode (no GPU needed): items_out[i] = (layer | n_tile << 3 | m_tile << 8) of the
// i-th work item for a stack of n_layers layers with n_tiles_per_layer[] 256-channel tiles over `rows` frame rows.
int64_t stack_plan(int64_t rows, int n_layers, const int32_t* n_tiles_per_layer, int band, uint32_t* items_out, int64_t capacity) {
  if (rows <= 0 || n_layers < 2 || n_layers > XVEC_MAX_STACK || !n_tiles_per_layer) return set_error(XVEC_E_ARG, "bad stack shape");
  static thread_local StackParams p;
  p = StackParams{};
  p.m_tiles = static_cast<int>((rows + BM - 1) / BM);
  p.n_layers = n_layers;
  for (int l = 0; l < n_layers; ++l) {
    if (n_tiles_per_layer[l] < 1 || n_tiles_per_layer[l] > 31) return set_error(XVEC_E_ARG, "bad n_tiles");
    p.L[l].n_tiles = n_tiles_per_layer[l];
  }
  int rc = fill_schedule(p, pick_band(p.m_tiles, n_layers, 74, band));
  if (rc) return rc;
  if (items_out) {
    int cursor = 0;
    for (unsigned i = 0; i < p.total_items && static_cast<int64_t>(i) < capacity; ++i) items_out[i] = decode_item(p, i, cursor);
  }
  return p.total_items;
}

int64_t stack_ctrl_bytes(int64_t rows, int n_layers) {
  if (rows <= 0 || n_layers < 2) return 0;
  const int64_t m_tiles = (rows + BM - 1) / BM;
  return 256 + (n_layers - 1) * m_tiles * 4;  // counters (64 words) | ready[layers - 1][m_tiles]
}

XVEC_DEFINE_WATCHDOG_BINDER(bind_watchdog_stack)

bool stack_supported(const XvecLayerDesc* tdnn, int n_tdnn, int64_t rows) {
  if (n_tdnn < 2 || n_tdnn > XVEC_MAX_STACK || rows <= 0 || rows > 0x7fffff00LL) return false;
  if (!valid_dtype(tdnn[0].dtype) || !valid_dtype(tdnn[1].dtype)) return false;
  // float16 runs in its own kernel instance: layer 0 is then TF32 or float16 as well, and float16 activations take no bf16 layer 0
  if ((tdnn[0].dtype == XVEC_F16 || tdnn[1].dtype == XVEC_F16) && tdnn[0].dtype != XVEC_F32 && tdnn[0].dtype != tdnn[1].dtype) return false;
  for (int i = 0; i < n_tdnn; ++i) {
    if (tdnn[i].taps < 1 || tdnn[i].taps > XVEC_MAX_TAPS) return false;
    if (i > 0 && (tdnn[i].dtype != tdnn[1].dtype || tdnn[i].cin != tdnn[i - 1].n)) return false;
    if (i + 1 < n_tdnn && (tdnn[i].n % BN != 0 || !tdnn[i].bias_dev)) return false;  // stored layers: full tiles, bias vector
    if ((tdnn[i].n + BN - 1) / BN > 31) return false;
    int max_off = 0;
    for (int j = 0; j < tdnn[i].taps; ++j) {
      if (tdnn[i].tap_offsets[j] < 0) return false;
      if (tdnn[i].tap_offsets[j] > max_off) max_off = tdnn[i].tap_offsets[j];
    }
    if (max_off > SLAB_ROWS_MAX - BM_CTA) return false;  // one activation slab holds 128 + max_off <= 136 frame rows
  }
  return true;
}

// Everything stack_dispatch derives from its arguments except the per-call pointers: the 3 x n_layers tensor maps (a
// cuTensorMapEncodeTiled each — together most of the host time of a call) and the kernel parameters.  A pipeline calls with
// the same few (input, scratch, weights, rows) combinations over and over — one per slot — so the last STACK_PLAN_CACHE of
// them are kept, keyed by every argument a map or a parameter depends on.  A key describes pointers AND extents, so an entry
// stays valid for as long as its key can recur.
struct StackKey {
  int dev, n_tdnn, band;
  int64_t rows, x_ld, act_ld;
  const void *x, *act0, *act1;
  XvecLayerDesc L[XVEC_MAX_STACK];
};
struct StackPlan {
  StackKey key;
  StackMaps maps;
  StackParams p;
  int grid;
  int act_dtype;   // kernel instance: the dtype of layers 1..
  uint64_t stamp;  // 0 = empty
};
constexpr int STACK_PLAN_CACHE = 64;
static std::mutex g_plan_mu;
static StackPlan g_plans[STACK_PLAN_CACHE];
static uint64_t g_plan_clock = 0;

static int build_plan(StackPlan& pl, const XvecLayerDesc* tdnn, int n_tdnn, const void* x, int64_t rows, int64_t x_ld, void* act0, void* act1,
                      int64_t act_ld, int band) {
  const int act_dtype = pl.act_dtype = tdnn[1].dtype;
  StackMaps& maps = pl.maps;
  StackParams& p = pl.p;
  p = StackParams{};
  p.rows = static_cast<int>(rows);
  p.m_tiles = static_cast<int>((rows + BM - 1) / BM);
  p.n_layers = n_tdnn;
  void* act[2] = {act0, act1};
  const void* h = x;
  int64_t h_ld = x_ld;
  int h_dtype = tdnn[0].dtype;
  int rc;
  for (int l = 0; l < n_tdnn; ++l) {
    const XvecLayerDesc& d = tdnn[l];
    StackLayer& L = p.L[l];
    const int bke = chunk_elems(d.dtype);
    L.n = d.n;
    L.n_tiles = (d.n + BN - 1) / BN;
    L.taps = d.taps;
    L.cpt = (d.cin + bke - 1) / bke;
    L.tf32 = d.dtype == XVEC_F32 ? 1 : 0;
    int max_off = 0;
    for (int j = 0; j < d.taps; ++j) {
      L.tap_off[j] = d.tap_offsets[j];
      if (d.tap_offsets[j] > max_off) max_off = d.tap_offsets[j];
    }
    L.tap_off4 = 0;
    for (int j = 0; j < d.taps; ++j) L.tap_off4 |= static_cast<unsigned>(d.tap_offsets[j]) << (4 * j);
    L.slab_rows = BM_CTA + max_off;
    L.bias = d.bias_dev;
    if (reinterpret_cast<uintptr_t>(d.bias_dev) & 15u) return set_error(XVEC_E_ARG, "bias must be 16-byte aligned");
    const int64_t h_rows = window_rows(rows, d.cin, h_ld);
    if (h_rows < 0) return static_cast<int>(h_rows);
    rc = make_tmap_2d(&maps.a[l], h, h_dtype, static_cast<uint64_t>(d.cin), static_cast<uint64_t>(h_rows), static_cast<uint64_t>(h_ld),
                      bke, static_cast<uint32_t>(L.slab_rows));
    if (rc) return rc;
    L.n_pad = L.n_tiles * BN;
    rc = make_weight_tmap(&maps.b[l], d);
    if (rc) return rc;
    if (l + 1 < n_tdnn) {
      // store boxes: 32 rows x 32 columns (64-byte rows / SWIZZLE_64B for 16-bit, 128-byte rows / SWIZZLE_128B for float32)
      rc = make_tmap_2d(&maps.y[l], act[l & 1], act_dtype, static_cast<uint64_t>(d.n), static_cast<uint64_t>(rows),
                        static_cast<uint64_t>(act_ld), 32, 32, act_dtype == XVEC_F32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
      if (rc) return rc;
      h = act[l & 1];
      h_ld = act_ld;
      h_dtype = act_dtype;
    } else {
      maps.y[l] = maps.a[l];  // unused
    }
  }
  for (int l = n_tdnn; l < XVEC_MAX_STACK; ++l) {
    maps.a[l] = maps.a[0];
    maps.b[l] = maps.b[0];
    maps.y[l] = maps.a[0];
  }
  const int max_pairs = num_sms() / 2;
  rc = fill_schedule(p, pick_band(p.m_tiles, n_tdnn, max_pairs, band));
  if (rc) return rc;
  l2_policies(&p.pol_a, &p.pol_b, &p.pol_y);
  p.runahead = STACK_RUNAHEAD;
  const int64_t pairs = static_cast<int64_t>(p.total_items) < max_pairs ? p.total_items : max_pairs;
  pl.grid = 2 * static_cast<int>(pairs);
  return XVEC_OK;
}

int stack_dispatch(const XvecLayerDesc* tdnn, int n_tdnn, const void* x, int64_t rows, int64_t x_ld, void* act0, void* act1,
                   int64_t act_ld, const int32_t* row_utt, const int32_t* blk_slot_base, float* part, void* ctrl, int64_t ctrl_bytes,
                   int band, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!stack_supported(tdnn, n_tdnn, rows)) return set_error(XVEC_E_ARG, "layer stack is not supported by the fused stack kernel");
  if (!x || !act0 || !act1 || !row_utt || !blk_slot_base || !part || !ctrl) return set_error(XVEC_E_ARG, "null pointer argument");
  if (ctrl_bytes < stack_ctrl_bytes(rows, n_tdnn) || (reinterpret_cast<uintptr_t>(ctrl) & 127u))
    return set_error(XVEC_E_ARG, "ctrl_dev must be 128-byte aligned and hold xvec_stack_ctrl_bytes() bytes");
  StackKey key;
  memset(&key, 0, sizeof(key));  // padding bytes too: keys are compared with memcmp
  cudaGetDevice(&key.dev);
  key.n_tdnn = n_tdnn;
  key.band = band > 0 ? band : 0;
  key.rows = rows;
  key.x_ld = x_ld;
  key.act_ld = act_ld;
  key.x = x;
  key.act0 = act0;
  key.act1 = act1;
  for (int l = 0; l < n_tdnn; ++l) {  // without the garbage the caller's struct may carry in unused tap slots
    rc = layer_desc(&key.L[l], tdnn[l].w_packed_dev, tdnn[l].bias_dev, tdnn[l].n, tdnn[l].cin, tdnn[l].taps, tdnn[l].dtype, tdnn[l].tap_offsets);
    if (rc) return rc;
  }
  StackMaps maps;
  StackParams p;
  int grid;
  int act_dtype;
  {
    std::lock_guard<std::mutex> lock(g_plan_mu);
    StackPlan* hit = nullptr;
    StackPlan* victim = &g_plans[0];
    for (StackPlan& pl : g_plans) {
      if (pl.stamp && memcmp(&pl.key, &key, sizeof(key)) == 0) {
        hit = &pl;
        break;
      }
      if (pl.stamp < victim->stamp) victim = &pl;
    }
    if (!hit) {
      victim->stamp = 0;
      rc = build_plan(*victim, tdnn, n_tdnn, x, rows, x_ld, act0, act1, act_ld, band);
      if (rc) return rc;
      victim->key = key;
      hit = victim;
    }
    hit->stamp = ++g_plan_clock;
    maps = hit->maps;
    p = hit->p;
    grid = hit->grid;
    act_dtype = hit->act_dtype;
  }
  p.counter = static_cast<unsigned*>(ctrl);
  p.ready = reinterpret_cast<unsigned*>(static_cast<char*>(ctrl) + 256);
  p.row_utt = row_utt;
  p.blk_slot_base = blk_slot_base;
  p.part = part;
#ifdef XVEC_DEBUG
  {
    const char* e = getenv("XVEC_STACK_DBG");
    p.dbg = e ? atoi(e) : 0;
  }
#endif
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(ctrl, 0, static_cast<size_t>(stack_ctrl_bytes(rows, n_tdnn)), st);
  if (e != cudaSuccess) return set_error(XVEC_E_CUDA, "cudaMemsetAsync(ctrl): %s", cudaGetErrorString(e));
  if (act_dtype == XVEC_F32)
    return launch_pair<tdnn_stack_kernel<XVEC_F32>>("tdnn_stack_kernel", STACK_THREADS, stack_smem_bytes<true>(), grid, bind_watchdog_stack, st, maps, p);
  if (act_dtype == XVEC_F16)
    return launch_pair<tdnn_stack_kernel<XVEC_F16>>("tdnn_stack_kernel", STACK_THREADS, stack_smem_bytes<false>(), grid, bind_watchdog_stack, st, maps, p);
  return launch_pair<tdnn_stack_kernel<XVEC_BF16>>("tdnn_stack_kernel", STACK_THREADS, stack_smem_bytes<false>(), grid, bind_watchdog_stack, st, maps, p);
}

}  // namespace xvec
