// Tile geometry and device/host pieces shared by the per-layer kernel (tdnn_gemm.cu) and the whole-stack kernel
// (tdnn_stack.cu): one output tile = 256 frames x 256 channels per CTA pair, 128-byte K chunks, 8 epilogue warps.
#pragma once
#include <stdlib.h>
#include <string.h>

#include "ptx.cuh"
#include "xvec_internal.h"

namespace xvec {

constexpr int BM_CTA = 128;            // frame rows per CTA
constexpr int BM = 2 * BM_CTA;         // frame rows per tile (CTA pair)
constexpr int BN = XVEC_TILE_N;        // 256 output channels per tile
constexpr int BN_CTA = BN / 2;         // weight rows staged by each CTA
constexpr int BK_BYTES = 128;          // one 128B-swizzle atom row: 64 bf16 or 32 tf32 channels
constexpr int A_BYTES = BM_CTA * BK_BYTES;  // 16 KiB
constexpr int B_BYTES = BN_CTA * BK_BYTES;  // 16 KiB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int EPI_WARPS = 8;             // two per TMEM lane quarter, each owning half (128) of the tile's columns
constexpr int GEMM_THREADS = 64 + 32 * EPI_WARPS;
constexpr int TMEM_COLS = 512;
constexpr int OUT_BUF_BYTES = 32 * 128;  // one TMA-store box: 32 rows x 128 bytes
constexpr int OUT_BUFS = 2;              // staging boxes per epilogue warp (TMA stores in flight)

// ReLU that keeps NaN like torch.relu (fmaxf(NaN, 0) is 0): the std of a single-frame utterance is NaN (torch.std, main.py:61) and
// has to stay NaN through relu(segment6) (main.py:72, 89).
__device__ __forceinline__ float relu_keep_nan(float v) { return v < 0.f ? 0.f : v; }

// {lo, hi} floats -> packed bf16x2 (lo in the low half), round-to-nearest; the _relu form clamps negatives to 0.
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// The same for float16.  No .satfinite: a value beyond the float16 range becomes +inf and reaches the x-vector as a non-finite
// value instead of a plausible wrong number (DESIGN.md section 4).
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// 16-bit pair packs of activation dtype kDtype (XVEC_BF16 or XVEC_F16).
template <int kDtype>
__device__ __forceinline__ uint32_t pack16x2(float lo, float hi) {
  if constexpr (kDtype == XVEC_F16) return pack_f16x2(lo, hi);
  else return pack_bf16x2(lo, hi);
}
template <int kDtype>
__device__ __forceinline__ uint32_t pack16x2_relu(float lo, float hi) {
  if constexpr (kDtype == XVEC_F16) return pack_f16x2_relu(lo, hi);
  else return pack_bf16x2_relu(lo, hi);
}

// Operand format of the UMMA instruction descriptor for operands of element type `dtype` (umma_idesc, ptx.cuh).
__host__ __device__ constexpr uint32_t umma_format(int dtype) { return dtype == XVEC_F32 ? 2u : dtype == XVEC_BF16 ? 1u : 0u; }

// Statistics-pooling epilogue of one TRANSPOSED accumulator tile for one epilogue warp (replaces the reads of torch.mean /
// torch.std in stat_pool, main.py:59-63).  The MMA warp swaps the operands of the pooled layer (weights = M operand, frames = N
// operand; both are 128 rows x 128 bytes K-major, so it is only a swap of the two descriptors): TMEM lane = output channel,
// column = frame.  A thread then owns ONE channel and reads 32 consecutive frames per tcgen05.ld, so the sums over time are
// plain register adds — no shared-memory transpose, no shuffles.  The warp covers XVEC_POOL_BLOCK = 128 consecutive frames
// (4 loads, load k+1 in flight while block k is reduced) and emits, per utterance with a pooled frame among them, the sum and
// the sum of squares of r = relu(acc + bias) into part[slot][2][n]; slots of a 128-frame group are consecutive in row order
// (blk_slot_base), the summation order is fixed (frame pairs in increasing order), nothing is atomic.
struct PoolArgs {
  int rows, n;
  const float* bias;
  const int* row_utt;
  const int* blk_slot_base;
  float* part;
};
// tcol: TMEM address of (this warp's lane quarter, first of its 128 columns); ch: this thread's channel; f0: frame of column 0
// (a multiple of 128); release(): called once, right after the warp's last tcgen05.ld of the tile has landed (NOT called when
// none of the warp's channels exist — the caller then releases the buffer itself).
// What a pooling tile reads from global memory before it can start: this thread's bias, the utterance of its frame in each of
// the four 32-frame blocks, the first partial slot of the 128-frame group.  pool_prefetch() issues these loads; calling it
// BEFORE the wait for the accumulator puts their ~700 cycles of L2 latency behind that wait instead of in front of the first
// tcgen05.ld (the epilogue warps' per-tile latency chain is what the MMA warp ends up waiting for).
struct PoolPrefetch {
  float bch;
  int my_u[4];
  int slot;
};
__device__ __forceinline__ PoolPrefetch pool_prefetch(const PoolArgs& p, int ch, int f0, int lane) {
  PoolPrefetch q;
  q.bch = (ch < p.n && p.bias) ? __ldg(p.bias + ch) : 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {  // frame -> utterance of the four 32-frame blocks (lane = frame within the block)
    const int f = f0 + 32 * k + lane;
    q.my_u[k] = f < p.rows ? __ldg(p.row_utt + f) : -1;
  }
  q.slot = __ldg(p.blk_slot_base + (f0 / XVEC_POOL_BLOCK));
  return q;
}
template <class Release>
__device__ __forceinline__ void pool_epilogue_tile_t(const PoolArgs& p, const PoolPrefetch& pre, uint32_t tcol, int ch, int f0, int lane,
                                                     Release&& release) {
  if (ch - lane >= p.n) return;  // warp-uniform: none of the warp's 32 channels exist
  const float bch = pre.bch;
  const float2 b2 = make_float2(bch, bch);
  int my_u[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) my_u[k] = pre.my_u[k];
  int slot = pre.slot;
  float* const part_ch = p.part + ch;
  const size_t slot_stride = 2 * static_cast<size_t>(p.n);
  uint32_t va[32], vb[32];
  tmem_ld_32x32(tcol, va);
  tmem_ld_wait();
  int cur_u = -1;  // utterance whose sums are being accumulated (frames of an utterance are consecutive rows)
  float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    uint32_t(&v)[32] = (k & 1) ? vb : va;
    if (k + 1 < 4) tmem_ld_32x32(tcol + 32 * (k + 1), (k & 1) ? va : vb);
    unsigned remaining = __ballot_sync(0xffffffffu, my_u[k] >= 0);
    while (remaining) {  // one pass per utterance present in this 32-frame block (warp-uniform)
      const int lo = __ffs(remaining) - 1;
      const int u = __shfl_sync(0xffffffffu, my_u[k], lo);
      const unsigned m = __ballot_sync(0xffffffffu, my_u[k] == u);
      if (u != cur_u) {
        if (cur_u >= 0) {
          if (ch < p.n) {
            part_ch[slot * slot_stride] = s2.x + s2.y;
            part_ch[slot * slot_stride + p.n] = q2.x + q2.y;
          }
          ++slot;
        }
        cur_u = u;
        s2 = make_float2(0.f, 0.f);
        q2 = make_float2(0.f, 0.f);
      }
      if (m == 0xffffffffu) {
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float2 a = __fadd2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), b2);
          a.x = fmaxf(a.x, 0.f);
          a.y = fmaxf(a.y, 0.f);
          s2 = __fadd2_rn(s2, a);
          q2 = __ffma2_rn(a, a, q2);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float2 a = __fadd2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), b2);
          a.x = ((m >> j) & 1u) ? fmaxf(a.x, 0.f) : 0.f;
          a.y = ((m >> (j + 1)) & 1u) ? fmaxf(a.y, 0.f) : 0.f;
          s2 = __fadd2_rn(s2, a);
          q2 = __ffma2_rn(a, a, q2);
        }
      }
      remaining &= ~m;
    }
    if (k + 1 < 4) tmem_ld_wait();
    if (k == 2) release();  // the last tcgen05.ld of the tile has landed
  }
  if (cur_u >= 0 && ch < p.n) {
    part_ch[slot * slot_stride] = s2.x + s2.y;
    part_ch[slot * slot_stride + p.n] = q2.x + q2.y;
  }
}

// ------------------------------------------------------------------------------------------------ host side
// L2 promotion of the TMA loads.  Measured on the stack kernel: none / 64 B / 128 B 302.8 us, 256 B 305.5 us — every box row is
// one 128-byte line, 256 B promotion fetches a neighbour line another CTA may not want yet.  Debug builds: XVEC_L2PROMO = 0
// none, 1 64 B, 2 128 B, 3 256 B (developer A/B switch; the product library reads no environment).
inline CUtensorMapL2promotion l2_promotion() {
#ifdef XVEC_DEBUG
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("XVEC_L2PROMO");
    v = (e && e[0] >= '0' && e[0] <= '3') ? e[0] - '0' : 2;
  }
  return v == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE : v == 1 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
       : v == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
#else
  return CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
#endif
}
// 2-D row-major tensor map; the inner box is one swizzle-width chunk (128 bytes unless stated).
inline int make_tmap_2d(CUtensorMap* map, const void* ptr, int dtype, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                        uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return set_error(XVEC_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  const uint64_t es = elem_bytes(dtype);
  if ((reinterpret_cast<uintptr_t>(ptr) & 15u) != 0) return set_error(XVEC_E_ARG, "matrix base pointer must be 16-byte aligned");
  if ((ld_elems * es) % 16 != 0) return set_error(XVEC_E_ARG, "row stride must be a multiple of 16 bytes");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * es};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType type = dtype == XVEC_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                 : dtype == XVEC_F16  ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  CUresult r = enc(map, type, 2,
                   const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle, l2_promotion(), CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(XVEC_E_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", static_cast<int>(r));
  return XVEC_OK;
}

// Rows of an input matrix its tensor map covers.  Window form (x_ld < cin: overlapping rows): only rows whose whole window lies
// inside the matrix exist, the rest read as zero.  Returns XVEC_E_ARG (negative) when there is not even one window.
inline int64_t window_rows(int64_t x_rows, int cin, int64_t x_ld) {
  const int64_t rows = x_ld < cin ? x_rows - (cin + x_ld - 1) / x_ld + 1 : x_rows;
  return rows > 0 ? rows : set_error(XVEC_E_ARG, "window form: fewer rows than one window");
}

// Packed weights of layer `l` are chunk-major (xvec_pack_weight): a (kblocks * n_pad) x chunk matrix, so the box a CTA loads per
// K chunk (half of the 256-row weight tile x 128 bytes) is one contiguous 16 KiB run.
inline int make_weight_tmap(CUtensorMap* map, const XvecLayerDesc& l) {
  const int bke = chunk_elems(l.dtype);
  const uint64_t kblocks = static_cast<uint64_t>(l.taps) * ((l.cin + bke - 1) / bke);
  const uint64_t n_pad = static_cast<uint64_t>((l.n + BN - 1) / BN) * BN;
  return make_tmap_2d(map, l.w_packed_dev, l.dtype, bke, kblocks * n_pad, bke, bke, BN_CTA);
}

// Launches kKernel as clusters of 2 CTAs (one tcgen05 CTA pair each).  The first launch on a device raises the kernel's dynamic
// shared-memory limit (once per kernel) and binds the watchdog word of the kernel's translation unit (bind_watchdog).
template <auto kKernel, class... Args>
inline int launch_pair(const char* name, int threads, int smem, int grid, int (*bind_watchdog)(), cudaStream_t st, const Args&... args) {
  static PerDeviceInit configured;  // per kernel
  int rc = once_per_device(configured, [smem] {
    cudaError_t e = cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return set_error(XVEC_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return static_cast<int>(XVEC_OK);
  });
  if (rc) return rc;
  rc = bind_watchdog();
  if (rc) return rc;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kKernel, args...);
  if (e != cudaSuccess) return set_error(XVEC_E_CUDA, "%s launch: %s", name, cudaGetErrorString(e));
  return XVEC_OK;
}

// L2 eviction hints of the TMA traffic: activations in (evict-first), weights (evict-last), activations out (evict-last).
// Debug builds: XVEC_L2HINT = three digits (0 normal, 1 evict-first, 2 evict-last) overrides the default.
inline void l2_policies(unsigned long long* pol_a, unsigned long long* pol_b, unsigned long long* pol_y) {
#ifdef XVEC_DEBUG
  static const unsigned long long pol_tab[3] = {L2_EVICT_NORMAL, L2_EVICT_FIRST, L2_EVICT_LAST};
  static int hint[3] = {-1, 0, 0};
  if (hint[0] < 0) {
    const char* h = getenv("XVEC_L2HINT");
    const char* def = "122";
    if (!h || strlen(h) != 3) h = def;
    int v[3];
    for (int i = 0; i < 3; ++i) v[i] = (h[i] >= '0' && h[i] <= '2') ? h[i] - '0' : 0;
    hint[2] = v[2];
    hint[1] = v[1];
    hint[0] = v[0];
  }
  *pol_a = pol_tab[hint[0]];
  *pol_b = pol_tab[hint[1]];
  *pol_y = pol_tab[hint[2]];
#else
  *pol_a = L2_EVICT_FIRST;
  *pol_b = L2_EVICT_LAST;
  *pol_y = L2_EVICT_LAST;
#endif
}

}  // namespace xvec
