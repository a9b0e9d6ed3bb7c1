// TDNN layer as a tcgen05 GEMM over the flat frame matrix — sm_100a only.
//
//   y[r, n] = epi( sum_{tap j} sum_{ch} x[r + off_j, ch] * W[n, j*Cin + ch] )
//
// replaces tdnn_layer.py:26-41 (get_time_context + torch.cat + nn.Linear + ReLU + eval BatchNorm1d) without ever
// materialising the unfolded (rows x taps*Cin) tensor: the K loop runs over (128-byte channel chunk, tap) and the
// TMA producer simply shifts the row coordinate of the A tile by the tap's frame offset.  Rows past the end of the
// matrix and channels past Cin are zero-filled by TMA, the packed weights carry matching zero padding.
//
// One output tile = 256 frames x 256 channels, computed by a CTA PAIR (cluster of 2, tcgen05 cta_group::2): each CTA
// stages its own 128 frame rows (A) and HALF of the weight tile (B, 128 channels) per 128-byte K chunk, so a CTA moves
// 32 KiB through shared memory per 128x256x{64 bf16|32 tf32} of its MMA work instead of the 48 KiB of a single-CTA
// 128x256 tile (measurements and the alternatives that were tried are in DESIGN.md §3).
//
// Persistent, warp-specialised CTA (320 threads, 1 CTA/SM, 74 pairs):
//   warp 0      TMA producer (both CTAs; completion bytes of both land on the LEADER's full barrier)
//   warp 1      TMEM owner; in the leader CTA it issues tcgen05.mma.cta_group::2 (UMMA 256x256xK, fp32 accumulators in
//               TMEM, two 256-column buffers so the epilogue of tile i overlaps the MMAs of tile i+1)
//               Both run warp-uniform loops (addresses / descriptors stay in uniform registers) and predicate only the
//               single-thread instructions on one elected lane; each step ends with a probe of the NEXT stage's barrier
//               (ptx.cuh: tma_step_pair, umma_step_pair).
//   warps 2-9   epilogue (both CTAs, 128 rows each; 2 warps per TMEM lane quarter, each half of the columns):
//               tcgen05.ld -> bias/ReLU (packed f32x2, cvt.relu) / BatchNorm affine -> 128B-swizzled smem staging
//               -> TMA store                                                                  (EPI_STORE_*)
//               or (tile computed TRANSPOSED: weights = M operand) -> per-utterance sums over time of r and r^2 in
//               registers, statistics pooling partials (gemm_tile.cuh: pool_epilogue_tile_t)   (EPI_POOL)
// The whole five-layer stack of the extraction path runs through tdnn_stack.cu instead (one persistent launch); this kernel
// serves the segment layers of the TF32 pipeline (split-K), the standalone TdnnLayer module, the PLDA GEMMs and stacks the
// fused kernel does not take.
#include "gemm_tile.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace xvec {

enum { EPI_STORE_F32 = 0, EPI_STORE_BF16 = 1, EPI_POOL = 2, EPI_STORE_F16 = 3 };
// Flag of the kernel's epilogue argument: the operands are float16 (kind::f16 in f16 format) instead of bfloat16.  A flag rather
// than a third template parameter, so that the bf16 / TF32 kernels keep their template arguments and symbol names.
constexpr int EPI_IN_F16 = 8;

struct GemmParams {
  int rows;     // output rows
  int n;        // valid output columns
  int m_tiles, n_tiles;
  int taps, cpt;  // K loop = taps * cpt chunks of 128 bytes
  int tap_off[XVEC_MAX_TAPS];
  const float* bias;
  const float* scale;
  const float* shift;
  int relu;
  void* out;
  long long ldo;
  int vec_store;  // output rows are 16-byte aligned -> swizzled smem staging + TMA store; else scalar stores
  const int* row_utt;
  const int* blk_slot_base;
  float* part;
  int ksplit, kb_per_split, rows_pad;  // split-K: tile t also selects a K range; partial sums go to row s*rows_pad + r
  unsigned long long pol_a, pol_b, pol_y;  // L2 eviction hints: activations in, weights, activations out
  long long* trace;  // debug: per-tile clock64 stamps of pair 0 (XVEC_TRACE=1)
  int dbg;  // debug: bit0 skip tmem loads, bit1 skip output staging+store, bit2 skip epilogue math
};

// Developer instrumentation (tools/trace_tiles.py, tools/episweep.py): only in -DXVEC_DEBUG builds
// (build.py --debug -> libxvec_b200_debug.so); the product library compiles all of it out.
constexpr int TRACE_TILES = 32;
constexpr int TRACE_SLOTS = 32;
#ifdef XVEC_DEBUG
__device__ __forceinline__ void trace(const GemmParams& p, int it, int slot) {
  if (p.trace && blockIdx.x == 0 && it < TRACE_TILES) p.trace[it * TRACE_SLOTS + slot] = clock64();
}
#define XVEC_DBG(p, bit) ((p).dbg & (bit))
#else
__device__ __forceinline__ void trace(const GemmParams&, int, int) {}
#define XVEC_DBG(p, bit) 0
#endif

template <int kEpi>
constexpr int num_stages() {
  return 5;
}
template <int kEpi>
constexpr int epi_smem_bytes() {
  return kEpi == EPI_POOL ? 0 : EPI_WARPS * OUT_BUFS * OUT_BUF_BYTES;  // the pooling epilogue works in registers
}
template <int kEpi>
constexpr int gemm_smem_bytes() {
  return 1024 + num_stages<kEpi>() * STAGE_BYTES + epi_smem_bytes<kEpi>();
}

// Operands: float32 with kind::tf32 (kTf32), else bfloat16, or float16 when kEpi carries EPI_IN_F16; kEpi & ~EPI_IN_F16 is the
// epilogue.  It is written out where it is used: a kernel-scope constexpr variable for it (or for the operand dtype) changes
// nvcc's register allocation in the bf16 / TF32 pooling kernels, whose code stays as it was measured.
template <bool kTf32, int kEpi>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
tdnn_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmY, const GemmParams p) {
  static_assert(!(kTf32 && (kEpi & EPI_IN_F16)), "float16 operands run kind::f16");
  constexpr int STAGES = num_stages<kEpi>();
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES], tfull_bar[2], tempty_bar[2];
  __shared__ uint32_t tmem_base_smem;
  __shared__ int tap_off_s[XVEC_MAX_TAPS];

  // SWIZZLE_128B tiles need 1024-byte alignment (same offset in both CTAs of the pair)
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* epi_smem = base + STAGES * STAGE_BYTES;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();  // 0 = leader of the pair
  const int pair = blockIdx.x >> 1;
  const int n_pairs = gridDim.x >> 1;
  constexpr int BKE = kTf32 ? 32 : 64;  // elements per 128-byte chunk
  const int kblocks = p.taps * p.cpt;
  const int mn_tiles = p.m_tiles * p.n_tiles;
  const int total_tiles = mn_tiles * p.ksplit;

  if (threadIdx.x < XVEC_MAX_TAPS) tap_off_s[threadIdx.x] = p.tap_off[threadIdx.x];
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if constexpr ((kEpi & ~EPI_IN_F16) != EPI_POOL) tma_prefetch_desc(&tmY);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);   // leader's arrive.expect_tx (bytes of both CTAs)
      mbar_init(&empty_bar[s], 1);  // leader's multicast commit
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);   // leader's multicast commit
      mbar_init(&tempty_bar[b], 2 * EPI_WARPS);  // one arrive per epilogue warp of both CTAs (on the leader's barrier)
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_pair<TMEM_COLS>(&tmem_base_smem);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // barriers of both CTAs are initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    // The whole warp runs the loop with warp-uniform control flow (addresses, coordinates, barrier state live in uniform
    // registers); only expect_tx / TMA are predicated on one elected lane.
    int stage = 0;
    uint32_t phase = 0;
    int pit = 0;
    uint32_t rdy = 0;
    uint32_t leader_full[STAGES];  // shared::cluster addresses of the leader's full barriers
#pragma unroll
    for (int i = 0; i < STAGES; ++i) leader_full[i] = mapa_u32(smem_u32(&full_bar[i]), 0);
    for (int t = pair; t < total_tiles; t += n_pairs, ++pit) {
      const int ks = t / mn_tiles, tt = t - ks * mn_tiles;
      const int m0 = (tt / p.n_tiles) * BM + static_cast<int>(rank) * BM_CTA;
      const int n0 = (tt % p.n_tiles) * BN + static_cast<int>(rank) * BN_CTA;
      const int kb0 = ks * p.kb_per_split, kb1 = min(kblocks, kb0 + p.kb_per_split);
      for (int kb = kb0; kb < kb1; ++kb) {
        const int ch = kb / p.taps;  // channel chunk outermost, taps innermost: the K order of tdnn_stack.cu (bit-identical sums)
        const int tap = kb - ch * p.taps;
        if (!rdy) mbar_wait(&empty_bar[stage], phase ^ 1u, 1);
        if (kb == kb0 && lane == 0) trace(p, pit, 0);
        const int arow = m0 + tap_off_s[tap];
        int stage_n = stage + 1;
        uint32_t phase_n = phase;
        if (stage_n == STAGES) { stage_n = 0; phase_n ^= 1u; }
        uint32_t lf = leader_full[0];
#pragma unroll
        for (int i = 1; i < STAGES; ++i) lf = (stage == i) ? leader_full[i] : lf;
        const uint32_t sa = smem_u32(base + stage * STAGE_BYTES);
        if (XVEC_DBG(p, 8)) {  // debug: no loads at all, only the barrier protocol
          if (elect_one() && rank == 0) mbar_expect_tx(&full_bar[stage], 0);
          __syncwarp();
          rdy = 0;
          stage = stage_n;
          phase = phase_n;
          continue;
        }
        rdy = tma_step_pair(elect_one() ? 1u : 0u, rank == 0 ? 1u : 0u, smem_u32(&full_bar[stage]), lf, 2 * STAGE_BYTES, sa, &tmA,
                            ch * BKE, arow, p.pol_a, sa + A_BYTES, &tmB, 0, (tap * p.cpt + ch) * (p.n_tiles * BN) + n0, p.pol_b, smem_u32(&empty_bar[stage_n]),
                            phase_n ^ 1u);
        stage = stage_n;
        phase = phase_n;
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA; warp-uniform loop, one
    // elected lane issues tcgen05.mma / tcgen05.commit; the readiness of the NEXT stage is probed before the MMAs are
    // issued so the probe latency is off the critical path)
    if (rank == 0) {
      constexpr uint32_t idesc = umma_idesc(umma_format(kTf32 ? XVEC_F32 : (kEpi & EPI_IN_F16) ? XVEC_F16 : XVEC_BF16), BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      uint32_t rdy = 0;
      for (int t = pair; t < total_tiles; t += n_pairs, ++it) {
        const int buf = it & 1;
        const uint32_t use = (it >> 1) & 1;
        if (lane == 0) trace(p, it, 1);
        mbar_wait(&tempty_bar[buf], use ^ 1u, 2);  // both CTAs' epilogues have drained this accumulator buffer
        if (lane == 0) trace(p, it, 2);
        const uint32_t d = tmem_base + buf * BN;
        const int kb0 = (t / mn_tiles) * p.kb_per_split, kb1 = min(kblocks, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          if (!(rdy & 1u)) mbar_wait(&full_bar[stage], phase, 3);
          tc_fence_after();
          if (kb == kb0 && lane == 0) trace(p, it, 3);
          const uint32_t a_addr = smem_u32(base + stage * STAGE_BYTES);
          // EPI_POOL computes the tile transposed (weights = M operand): see pool_epilogue_tile_t
          const uint64_t da = umma_desc_sw128((kEpi & ~EPI_IN_F16) == EPI_POOL ? a_addr + A_BYTES : a_addr);
          const uint64_t db = umma_desc_sw128((kEpi & ~EPI_IN_F16) == EPI_POOL ? a_addr : a_addr + A_BYTES);
          int stage_n = stage + 1;
          uint32_t phase_n = phase;
          if (stage_n == STAGES) { stage_n = 0; phase_n ^= 1u; }
          if (XVEC_DBG(p, 16)) {  // debug: no MMAs, only the barrier protocol
            if (elect_one()) umma_commit_pair(&empty_bar[stage], 0x3);
            __syncwarp();
            rdy = 0;
            stage = stage_n;
            phase = phase_n;
            continue;
          }
          rdy = umma_step_pair<kTf32>(elect_one() ? 1u : 0u, d, da, db, idesc, kb > kb0 ? 1u : 0u, STEP_COMMIT_A | STEP_PROBE_A,
                                      smem_u32(&empty_bar[stage]), 0u, smem_u32(&full_bar[stage_n]), phase_n, 0u, 0u);
          stage = stage_n;
          phase = phase_n;
        }
        if (elect_one()) umma_commit_pair(&tfull_bar[buf], 0x3);  // accumulator complete (both CTAs' epilogues)
        __syncwarp();
        if (lane == 0) trace(p, it, 4);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (both CTAs, 128 rows each)
    const int q = warp & 3;             // TMEM lane quarter this warp may read
    const int cbeg = ((warp - 2) >> 2) * (BN / 2);  // this warp's half of the tile's columns
    const int cend = cbeg + BN / 2;
    int it = 0;
    int store_seq = 0;
    for (int t = pair; t < total_tiles; t += n_pairs, ++it) {
      const int ks = t / mn_tiles, tt = t - ks * mn_tiles;
      const int m0 = (tt / p.n_tiles) * BM + static_cast<int>(rank) * BM_CTA;
      const int n0 = (tt % p.n_tiles) * BN;
      const int buf = it & 1;
      const uint32_t use = (it >> 1) & 1;
      if (warp == 2 && lane == 0) trace(p, it, 5);
      mbar_wait(&tfull_bar[buf], use, 4);
      tc_fence_after();
      if (warp == 2 && lane == 0) trace(p, it, 6);
      const uint32_t tbase = tmem_base + buf * BN + (static_cast<uint32_t>(q * 32) << 16);
      const int row0 = m0 + q * 32;
      const int row = row0 + lane;
      // The accumulator buffer goes back to the MMA issuer as soon as this warp's LAST tcgen05.ld of the tile has landed in
      // registers — the math / staging / stores of that last chunk then overlap the MMAs of tile i+2.
      bool released = false;
      auto release_tmem = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[buf]), 0));
        released = true;
      };
      const int c_last = min(cend, p.n - n0) - 1;  // last valid column of this warp's range (may be < cbeg)

      if constexpr ((kEpi & ~EPI_IN_F16) == EPI_POOL) {
        const PoolArgs pa{p.rows, p.n, p.bias, p.row_utt, p.blk_slot_base, p.part};
        const int pch = n0 + static_cast<int>(rank) * BN_CTA + q * 32 + lane, pf0 = (tt / p.n_tiles) * BM + cbeg;
        pool_epilogue_tile_t(pa, pool_prefetch(pa, pch, pf0, lane), tmem_base + buf * BN + (static_cast<uint32_t>(q * 32) << 16) + cbeg, pch,
                             pf0, lane, release_tmem);
      } else {
        uint8_t* out_stage = epi_smem + (warp - 2) * (OUT_BUFS * OUT_BUF_BYTES);  // 32-row x 128-byte staging boxes
        constexpr int kStore = kEpi & ~EPI_IN_F16;
        constexpr bool k16 = kStore == EPI_STORE_BF16 || kStore == EPI_STORE_F16;  // 16-bit output
        constexpr int kOut = kStore == EPI_STORE_F16 ? XVEC_F16 : XVEC_BF16;        // ... and its type
        constexpr int OUT_ES = k16 ? 2 : 4;
        constexpr int GROUP_COLS = 128 / OUT_ES;     // columns per TMA-store box (128 bytes per row)
        constexpr int CHUNKS = GROUP_COLS / 32;      // tcgen05.ld chunks per box
        for (int c = cbeg; c < cend && n0 + c < p.n; c += GROUP_COLS) {
          uint8_t* ob = out_stage + (store_seq % OUT_BUFS) * OUT_BUF_BYTES;
          if (p.vec_store && !(XVEC_DBG(p, 2))) {
            if (lane == 0) tma_store_wait_read<OUT_BUFS - 1>();  // the store that last used this box has read it
            __syncwarp();
          }
#pragma unroll
          for (int cc = 0; cc < CHUNKS; ++cc) {
            const int col0 = n0 + c + cc * 32;
            if (col0 >= p.n) break;  // warp-uniform; the box is clipped by TMA
            uint32_t v[32];
            if (!(XVEC_DBG(p, 1))) {
              if (warp == 2 && lane == 0 && c == cbeg && cc == 0) trace(p, it, 8);
              tmem_ld_32x32(tbase + c + cc * 32, v);
              tmem_ld_wait();
              if (c + cc * 32 + 32 > c_last) release_tmem();
              if (warp == 2 && lane == 0 && c == cbeg && cc == 0) trace(p, it, 9);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = lane + j;
            }
            // bias (+ReLU, + optional BatchNorm affine); column parameters are warp-uniform read-only loads
            float o[32];
            const float4* bp = reinterpret_cast<const float4*>(p.bias + col0);
            if (p.scale == nullptr) {
#pragma unroll
              for (int j4 = 0; j4 < 32; j4 += 4) {
                const float4 bb = p.bias ? __ldg(bp + (j4 >> 2)) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float2 a = __fadd2_rn(make_float2(__uint_as_float(v[j4 + 0]), __uint_as_float(v[j4 + 1])), make_float2(bb.x, bb.y));
                const float2 d = __fadd2_rn(make_float2(__uint_as_float(v[j4 + 2]), __uint_as_float(v[j4 + 3])), make_float2(bb.z, bb.w));
                o[j4 + 0] = a.x; o[j4 + 1] = a.y; o[j4 + 2] = d.x; o[j4 + 3] = d.y;
              }
              if (p.relu && !k16) {  // 16-bit output: ReLU is folded into the convert below
#pragma unroll
                for (int j = 0; j < 32; ++j) o[j] = relu_keep_nan(o[j]);
              }
            } else {
              const float4* sp = reinterpret_cast<const float4*>(p.scale + col0);
              const float4* hp = reinterpret_cast<const float4*>(p.shift + col0);
#pragma unroll
              for (int j4 = 0; j4 < 32; j4 += 4) {
                const float4 bb = p.bias ? __ldg(bp + (j4 >> 2)) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float4 sc = __ldg(sp + (j4 >> 2));
                const float4 sh = __ldg(hp + (j4 >> 2));
                float2 a = __fadd2_rn(make_float2(__uint_as_float(v[j4 + 0]), __uint_as_float(v[j4 + 1])), make_float2(bb.x, bb.y));
                float2 d = __fadd2_rn(make_float2(__uint_as_float(v[j4 + 2]), __uint_as_float(v[j4 + 3])), make_float2(bb.z, bb.w));
                if (p.relu) { a.x = relu_keep_nan(a.x); a.y = relu_keep_nan(a.y); d.x = relu_keep_nan(d.x); d.y = relu_keep_nan(d.y); }
                a = __ffma2_rn(a, make_float2(sc.x, sc.y), make_float2(sh.x, sh.y));
                d = __ffma2_rn(d, make_float2(sc.z, sc.w), make_float2(sh.z, sh.w));
                o[j4 + 0] = a.x; o[j4 + 1] = a.y; o[j4 + 2] = d.x; o[j4 + 3] = d.y;
              }
            }
            const bool cvt_relu = p.relu && p.scale == nullptr;  // ReLU not applied yet (16-bit fast path)
            if (warp == 2 && lane == 0 && c == cbeg && cc == 0) trace(p, it, 10);
            if (XVEC_DBG(p, 2)) {
              if (o[0] == 123.456f && o[31] == 1.f) ob[lane] = 1;
            } else if (p.vec_store) {
              // row `lane` of the box, 16-byte pieces XOR-swizzled like CU_TENSOR_MAP_SWIZZLE_128B expects
              uint8_t* orow = ob + lane * 128;
              if constexpr (k16) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  uint4 w;
                  if (cvt_relu) {
                    w.x = pack16x2_relu<kOut>(o[8 * j + 0], o[8 * j + 1]);
                    w.y = pack16x2_relu<kOut>(o[8 * j + 2], o[8 * j + 3]);
                    w.z = pack16x2_relu<kOut>(o[8 * j + 4], o[8 * j + 5]);
                    w.w = pack16x2_relu<kOut>(o[8 * j + 6], o[8 * j + 7]);
                  } else {
                    w.x = pack16x2<kOut>(o[8 * j + 0], o[8 * j + 1]);
                    w.y = pack16x2<kOut>(o[8 * j + 2], o[8 * j + 3]);
                    w.z = pack16x2<kOut>(o[8 * j + 4], o[8 * j + 5]);
                    w.w = pack16x2<kOut>(o[8 * j + 6], o[8 * j + 7]);
                  }
                  const int piece = cc * 4 + j;
                  *reinterpret_cast<uint4*>(orow + ((piece ^ (lane & 7)) << 4)) = w;
                }
              } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 w = make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
                  *reinterpret_cast<float4*>(orow + ((j ^ (lane & 7)) << 4)) = w;
                }
              }
            } else if (row < p.rows) {
              if constexpr (kStore == EPI_STORE_BF16) {
                __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<size_t>(row) * p.ldo + col0;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + j < p.n) dst[j] = __float2bfloat16_rn(cvt_relu ? relu_keep_nan(o[j]) : o[j]);
              } else if constexpr (kStore == EPI_STORE_F16) {
                __half* dst = reinterpret_cast<__half*>(p.out) + static_cast<size_t>(row) * p.ldo + col0;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + j < p.n) dst[j] = __float2half_rn(cvt_relu ? relu_keep_nan(o[j]) : o[j]);
              } else {
                float* dst = reinterpret_cast<float*>(p.out) + static_cast<size_t>(row) * p.ldo + col0;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + j < p.n) dst[j] = o[j];
              }
            }
          }
          if (p.vec_store && !(XVEC_DBG(p, 2))) {
            if (warp == 2 && lane == 0 && c == cbeg) trace(p, it, 14);
            fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
            __syncwarp();
            if (warp == 2 && lane == 0 && c == cbeg) trace(p, it, 15);
            if (lane == 0) {
              if (row0 < p.rows) tma_store_2d(&tmY, ob, n0 + c, ks * p.rows_pad + row0, p.pol_y);  // rows / columns past the matrix are clipped
              tma_store_commit();
            }
            if (warp == 2 && lane == 0 && c == cbeg) trace(p, it, 11);
            ++store_seq;
          }
        }
      }
      if (!released) release_tmem();  // nothing was read (no pooled rows / no valid columns in this warp's range)
      if (warp == 2 && lane == 0) trace(p, it, 7);
    }
    if constexpr ((kEpi & ~EPI_IN_F16) != EPI_POOL) {
      if (lane == 0) tma_store_wait_all();
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer may still be reading our smem / signalling our barriers until here
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair<TMEM_COLS>(tmem_base);
  }
}

// Split-K second pass: y[r, c] = epi( sum_s ws[s*rows_pad + r, c] ) in fixed split order (deterministic).
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ ws, int ksplit, int rows, int rows_pad, int n, int ws_ld, const float* __restrict__ bias,
                     const float* __restrict__ scale, const float* __restrict__ shift, int relu, void* __restrict__ out, int out_dtype,
                     long long ldo) {
  const long long total = static_cast<long long>(rows) * n;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / n);
    const int c = static_cast<int>(i - static_cast<long long>(r) * n);
    float a = 0.f;
    for (int s = 0; s < ksplit; ++s) a += ws[(static_cast<size_t>(s) * rows_pad + r) * ws_ld + c];
    if (bias) a += bias[c];
    if (relu) a = a < 0.f ? 0.f : a;  // keeps NaN like torch.relu
    if (scale) a = fmaf(a, scale[c], shift[c]);
    if (out_dtype == XVEC_BF16)
      reinterpret_cast<__nv_bfloat16*>(out)[static_cast<size_t>(r) * ldo + c] = __float2bfloat16_rn(a);
    else if (out_dtype == XVEC_F16)
      reinterpret_cast<__half*>(out)[static_cast<size_t>(r) * ldo + c] = __float2half_rn(a);
    else
      reinterpret_cast<float*>(out)[static_cast<size_t>(r) * ldo + c] = a;
  }
}

// ------------------------------------------------------------------------------------------------ host side
static long long* g_trace_buf = nullptr;

// Persistent grid: one CTA pair per tile, at most one pair per two SMs.
template <int kEpi>
static int launch(int dtype, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ty, const GemmParams& p, cudaStream_t st) {
  const int64_t tiles = static_cast<int64_t>(p.m_tiles) * p.n_tiles * p.ksplit;
  const int max_pairs = num_sms() / 2;
  const int grid = 2 * static_cast<int>(tiles < max_pairs ? tiles : max_pairs);
  constexpr int smem = gemm_smem_bytes<kEpi>();
  if (dtype == XVEC_F32)
    return launch_pair<tdnn_gemm_kernel<true, kEpi>>("tdnn_gemm_kernel", GEMM_THREADS, smem, grid, bind_watchdog_gemm, st, ta, tb, ty, p);
  if (dtype == XVEC_BF16)
    return launch_pair<tdnn_gemm_kernel<false, kEpi>>("tdnn_gemm_kernel", GEMM_THREADS, smem, grid, bind_watchdog_gemm, st, ta, tb, ty, p);
  return launch_pair<tdnn_gemm_kernel<false, kEpi | EPI_IN_F16>>("tdnn_gemm_kernel", GEMM_THREADS, smem, grid, bind_watchdog_gemm, st, ta, tb, ty, p);
}

// Split-K plan for GEMMs with too few output tiles to fill the machine (segment6/7: a few hundred rows, K = 3000).
static void splitk_plan(int64_t rows, int n, int kblocks, int* ksplit, int* kb_per_split) {
  const int64_t mn = ((rows + BM - 1) / BM) * ((n + BN - 1) / BN);
  const int pairs = num_sms() / 2;
  *ksplit = 1;
  *kb_per_split = kblocks;
  if (mn * 4 > pairs || kblocks < 8) return;
  int want = static_cast<int>(pairs / mn);
  if (want > kblocks / 2) want = kblocks / 2;
  if (want < 2) return;
  *kb_per_split = (kblocks + want - 1) / want;
  *ksplit = (kblocks + *kb_per_split - 1) / *kb_per_split;
}

int64_t splitk_workspace_bytes(int64_t rows, int cin, int taps, int n, int dtype) {
  const int bke = chunk_elems(dtype);
  int ksplit, kbs;
  splitk_plan(rows, n, taps * ((cin + bke - 1) / bke), &ksplit, &kbs);
  if (ksplit <= 1) return 0;
  const int64_t rows_pad = (rows + BM - 1) / BM * BM;
  return static_cast<int64_t>(ksplit) * rows_pad * ((n + BN - 1) / BN * BN) * 4;
}

// What both epilogues share: the checks of the layer and its input, the kernel parameters of the whole K loop with the bias and
// no other epilogue operand, and the tensor maps of the input (ta) and the packed weights (tb).  ty is a placeholder until an
// epilogue stores through TMA.
static int gemm_setup(const XvecLayerDesc& l, const void* x, int64_t x_rows, int64_t x_ld, int64_t rows, GemmParams& p, CUtensorMap& ta,
                      CUtensorMap& tb, CUtensorMap& ty) {
  int rc = device_check();
  if (rc) return rc;
  if (!x || !l.w_packed_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (!valid_dtype(l.dtype)) return set_error(XVEC_E_ARG, "bad x_dtype %d", l.dtype);
  if (l.taps < 1 || l.taps > XVEC_MAX_TAPS) return set_error(XVEC_E_ARG, "taps must be in [1,%d]", XVEC_MAX_TAPS);
  if (rows <= 0 || x_rows <= 0 || l.cin <= 0 || l.n <= 0) return set_error(XVEC_E_ARG, "non-positive size");
  if (rows > 0x7fffff00LL || x_rows > 0x7fffff00LL) return set_error(XVEC_E_ARG, "too many rows");
  const int bke = chunk_elems(l.dtype);
  p = GemmParams{};
  p.rows = static_cast<int>(rows);
  p.n = l.n;
  p.m_tiles = static_cast<int>((rows + BM - 1) / BM);
  p.n_tiles = (l.n + BN - 1) / BN;
  p.taps = l.taps;
  p.cpt = (l.cin + bke - 1) / bke;
  for (int j = 0; j < l.taps; ++j) {
    if (l.tap_offsets[j] < 0) return set_error(XVEC_E_ARG, "tap offsets must be non-negative");
    p.tap_off[j] = l.tap_offsets[j];
  }
  p.bias = l.bias_dev;
  p.ksplit = 1;
  p.kb_per_split = l.taps * p.cpt;
  p.rows_pad = p.m_tiles * BM;
  l2_policies(&p.pol_a, &p.pol_b, &p.pol_y);
#ifdef XVEC_DEBUG
  {  // developer instrumentation (XVEC_DBG epilogue/mainloop skip switches, XVEC_TRACE per-tile clock stamps): debug builds only
    static int dbg = -1;
    static long long* trace_buf = nullptr;
    if (dbg < 0) {
      const char* e = getenv("XVEC_DBG");
      dbg = e ? atoi(e) : 0;
      if (getenv("XVEC_TRACE")) cudaMalloc(&trace_buf, TRACE_TILES * TRACE_SLOTS * sizeof(long long));
    }
    p.dbg = dbg;
    p.trace = trace_buf;
    g_trace_buf = trace_buf;
  }
#endif
  const int64_t a_rows = window_rows(x_rows, l.cin, x_ld);
  if (a_rows < 0) return static_cast<int>(a_rows);
  rc = make_tmap_2d(&ta, x, l.dtype, static_cast<uint64_t>(l.cin), static_cast<uint64_t>(a_rows), static_cast<uint64_t>(x_ld), bke, BM_CTA);
  if (rc) return rc;
  ty = ta;
  return make_weight_tmap(&tb, l);
}

// Destination of a store epilogue: y_rows x n of y_dtype, row stride y_ld.  16-byte aligned rows are staged in swizzled shared
// memory and TMA-stored through ty; other rows are stored element by element.
static int set_store_output(GemmParams& p, CUtensorMap& ty, void* y, int y_dtype, int64_t y_ld, int64_t y_rows) {
  const int64_t es = elem_bytes(y_dtype);
  p.out = y;
  p.ldo = y_ld;
  p.vec_store = ((reinterpret_cast<uintptr_t>(y) & 15u) == 0 && (y_ld * es) % 16 == 0) ? 1 : 0;
  if (!p.vec_store) return XVEC_OK;
  return make_tmap_2d(&ty, y, y_dtype, static_cast<uint64_t>(p.n), static_cast<uint64_t>(y_rows), static_cast<uint64_t>(y_ld),
                      static_cast<uint32_t>(128 / es), 32);
}

int gemm_pool(const XvecLayerDesc& l, const void* x, int64_t x_rows, int64_t x_ld, int64_t rows, const int32_t* row_utt,
              const int32_t* blk_slot_base, float* part, void* stream) {
  GemmParams p;
  CUtensorMap ta, tb, ty;
  int rc = gemm_setup(l, x, x_rows, x_ld, rows, p, ta, tb, ty);
  if (rc) return rc;
  if (!row_utt || !blk_slot_base || !part) return set_error(XVEC_E_ARG, "null pointer argument");
  p.row_utt = row_utt;
  p.blk_slot_base = blk_slot_base;
  p.part = part;
  return launch<EPI_POOL>(l.dtype, ta, tb, ty, p, static_cast<cudaStream_t>(stream));
}

int gemm_store(const XvecLayerDesc& l, const void* x, int64_t x_rows, int64_t x_ld, int64_t rows, const float* bn_scale,
               const float* bn_shift, int relu, void* y, int y_dtype, int64_t y_ld, void* ws, int64_t ws_bytes, void* stream) {
  GemmParams p;
  CUtensorMap ta, tb, ty;
  int rc = gemm_setup(l, x, x_rows, x_ld, rows, p, ta, tb, ty);
  if (rc) return rc;
  if (!y) return set_error(XVEC_E_ARG, "null pointer argument");
  if (!valid_dtype(y_dtype)) return set_error(XVEC_E_ARG, "bad y_dtype %d", y_dtype);
  if ((bn_scale == nullptr) != (bn_shift == nullptr)) return set_error(XVEC_E_ARG, "bn_scale and bn_shift must be given together");
  if ((reinterpret_cast<uintptr_t>(l.bias_dev) & 15u) || (reinterpret_cast<uintptr_t>(bn_scale) & 15u) || (reinterpret_cast<uintptr_t>(bn_shift) & 15u))
    return set_error(XVEC_E_ARG, "bias / bn_scale / bn_shift must be 16-byte aligned (and hold ceil(n/32)*32 floats)");
  if (y_ld < l.n) return set_error(XVEC_E_ARG, "y_ld < n");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t ws_need = splitk_workspace_bytes(rows, l.cin, l.taps, l.n, l.dtype);
  if (ws_need == 0 || !ws || ws_bytes < ws_need || (reinterpret_cast<uintptr_t>(ws) & 15u)) {
    p.scale = bn_scale;
    p.shift = bn_shift;
    p.relu = relu;
    rc = set_store_output(p, ty, y, y_dtype, y_ld, rows);
    if (rc) return rc;
    if (y_dtype == XVEC_BF16) return launch<EPI_STORE_BF16>(l.dtype, ta, tb, ty, p, st);
    if (y_dtype == XVEC_F16) return launch<EPI_STORE_F16>(l.dtype, ta, tb, ty, p, st);
    return launch<EPI_STORE_F32>(l.dtype, ta, tb, ty, p, st);
  }
  // split-K, step 1: a GEMM with no epilogue; split s of the K loop writes the sums of output row r to workspace row s * rows_pad + r
  splitk_plan(rows, l.n, l.taps * p.cpt, &p.ksplit, &p.kb_per_split);
  p.bias = nullptr;
  const int ws_ld = p.n_tiles * BN;
  rc = set_store_output(p, ty, ws, XVEC_F32, ws_ld, static_cast<int64_t>(p.ksplit) * p.rows_pad);
  if (rc) return rc;
  rc = launch<EPI_STORE_F32>(l.dtype, ta, tb, ty, p, st);
  if (rc) return rc;
  // step 2: the splits summed in fixed order (deterministic), then the caller's epilogue into y
  const long long total = rows * static_cast<long long>(l.n);
  long long blocks = (total + 255) / 256;
  if (blocks > num_sms() * 8LL) blocks = num_sms() * 8LL;
  splitk_reduce_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(static_cast<const float*>(ws), p.ksplit, p.rows, p.rows_pad, l.n, ws_ld,
                                                                    l.bias_dev, bn_scale, bn_shift, relu, y, y_dtype, y_ld);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(XVEC_E_CUDA, "splitk_reduce_kernel launch: %s", cudaGetErrorString(e));
  return XVEC_OK;
}

int read_trace(long long* out_host, int n) {
  if (!g_trace_buf) return 0;
  const int m = n < TRACE_TILES * TRACE_SLOTS ? n : TRACE_TILES * TRACE_SLOTS;
  cudaDeviceSynchronize();
  cudaMemcpy(out_host, g_trace_buf, m * sizeof(long long), cudaMemcpyDeviceToHost);
  return m;
}

XVEC_DEFINE_WATCHDOG_BINDER(bind_watchdog_gemm)

}  // namespace xvec
