// Small-footprint linear layer for the segment layers (segment_layer6 / segment_layer7, main.py:45-46, 87-90) — sm_100a build,
// legacy mma.sync tensor path on purpose.
//
//   y[m, n] = act( sum_k x[m, k] * W[n, k] + bias[n] ),   x (M, K) and W (N, K) row-major (nn.Linear layout), both bf16, both
//   f16 or both float32 (TF32 math), fp32 accumulate; y float32, bf16 or f16
//
// Why not the tcgen05 kernel: the segment GEMM of a batch (256 x 3000 x 512, 0.8 GFLOP) is tiny, but tdnn_gemm_kernel needs a
// whole SM (227 KiB of shared memory, all of TMEM).  The persistent tdnn_stack_kernel of the NEXT batch already owns every SM, so
// that GEMM (and the split-K reduce behind it) could only run in the gaps between two stack kernels — measured: ~24 us of a
// 325 us step.  This kernel fits NEXT TO a resident stack CTA (128 threads, 5 KiB of shared memory, < 64 registers, no TMEM),
// so the tail of batch i runs concurrently with the stack kernel of batch i+1.  Fixed summation order, no split-K, no atomics.
//
// CTA tile 32 x 32, K step of 64 bytes per row (32 bf16 or f16 / 16 float32; six steps of operands in flight in registers, the
// loop is bound by L2 latency), 4 warps x (16 x 16) via ldmatrix + mma.sync.m16n8k16.bf16 / .f16 / m16n8k8.tf32 (ldmatrix on 32-bit data
// hands thread (g, t) the element (row g, column t) of each 8 x 4 block, which is the tf32 fragment layout).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "xvec_internal.h"

namespace xvec {

constexpr int FS_TILE = 32;         // rows and columns of a CTA tile
constexpr int FS_ROW_BYTES = 64;    // K bytes per row and step
constexpr int FS_PITCH_BYTES = 80;  // shared-memory row pitch: ldmatrix rows land in distinct 16-byte bank groups
constexpr int FS_DEPTH = 6;         // K steps of operands in flight per thread (registers)

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem) {
  const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
// One 16 x 8 x (32 bytes of K) tensor-core step of operand dtype kIn: bf16 or f16 m16n8k16, tf32 m16n8k8 (same register counts,
// same ldmatrix addressing).
template <int kIn>
__device__ __forceinline__ void mma_16x8(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (kIn == XVEC_F32)
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  else if constexpr (kIn == XVEC_BF16)
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  else
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// kIn: operand dtype, kOut: output dtype (XVEC_F32 / XVEC_BF16 / XVEC_F16).
template <int kIn, int kOut>
__global__ void __launch_bounds__(128)
fc_small_kernel(const uint8_t* __restrict__ x, long long ldx_bytes, const uint8_t* __restrict__ w, long long ldw_bytes,
                const float* __restrict__ bias, int M, int N, int k_bytes, int relu, void* __restrict__ y, long long ldy) {
  __shared__ __align__(16) uint8_t xs[FS_TILE * FS_PITCH_BYTES], ws[FS_TILE * FS_PITCH_BYTES];
  const int m0 = blockIdx.y * FS_TILE, n0 = blockIdx.x * FS_TILE;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lrow = tid >> 2, lchunk = tid & 3;  // this thread stages 16 bytes of one row of each operand tile
  const int wm = warp & 1, wn = warp >> 1;      // the warp's 16 x 16 sub-tile
  const bool x_ok = m0 + lrow < M, w_ok = n0 + lrow < N;
  const uint4* xp = reinterpret_cast<const uint4*>(x + static_cast<long long>(x_ok ? m0 + lrow : 0) * ldx_bytes) + lchunk;
  const uint4* wp = reinterpret_cast<const uint4*>(w + static_cast<long long>(w_ok ? n0 + lrow : 0) * ldw_bytes) + lchunk;
  const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
  const int steps = (k_bytes + FS_ROW_BYTES - 1) / FS_ROW_BYTES;
  auto fetch = [&](int s, uint4& rx, uint4& rw) {  // K bytes are a multiple of 16: a 16-byte piece is either whole or past the end
    const bool k_ok = s * FS_ROW_BYTES + lchunk * 16 < k_bytes;
    rx = (x_ok && k_ok) ? __ldg(xp + s * 4) : zero;
    rw = (w_ok && k_ok) ? __ldg(wp + s * 4) : zero;
  };
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  // FS_DEPTH steps of operands in flight in registers: the loop is bound by the L2 latency of these loads, not by the math
  uint4 rx[FS_DEPTH], rw[FS_DEPTH];
#pragma unroll
  for (int j = 0; j < FS_DEPTH; ++j) fetch(j, rx[j], rw[j]);
  for (int s0 = 0; s0 < steps; s0 += FS_DEPTH) {
#pragma unroll
    for (int j = 0; j < FS_DEPTH; ++j) {
      const int s = s0 + j;
      if (s >= steps) break;
      *reinterpret_cast<uint4*>(&xs[lrow * FS_PITCH_BYTES + lchunk * 16]) = rx[j];
      *reinterpret_cast<uint4*>(&ws[lrow * FS_PITCH_BYTES + lchunk * 16]) = rw[j];
      __syncthreads();
      fetch(s + FS_DEPTH, rx[j], rw[j]);  // past the end: zero, no access
#pragma unroll
      for (int kk = 0; kk < 2; ++kk) {  // two 32-byte K blocks per step
        uint32_t a[4], b[4];
        ldmatrix_x4(a, &xs[(16 * wm + (lane & 7) + 8 * ((lane >> 3) & 1)) * FS_PITCH_BYTES + 32 * kk + 16 * (lane >> 4)]);
        ldmatrix_x4(b, &ws[(16 * wn + (lane & 7) + 8 * (lane >> 4)) * FS_PITCH_BYTES + 32 * kk + 16 * ((lane >> 3) & 1)]);
        mma_16x8<kIn>(acc[0], a, b[0], b[1]);
        mma_16x8<kIn>(acc[1], a, b[2], b[3]);
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int col = n0 + 16 * wn + 8 * t + 2 * (lane & 3);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int row = m0 + 16 * wm + (lane >> 2) + 8 * h;
      if (row >= M) continue;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        if (col + e >= N) continue;
        float v = acc[t][2 * h + e] + (bias ? bias[col + e] : 0.f);
        if (relu) v = v < 0.f ? 0.f : v;  // keeps NaN like torch.relu (fmaxf would turn it into 0)
        if constexpr (kOut == XVEC_BF16) reinterpret_cast<__nv_bfloat16*>(y)[static_cast<long long>(row) * ldy + col + e] = __float2bfloat16_rn(v);
        else if constexpr (kOut == XVEC_F16) reinterpret_cast<__half*>(y)[static_cast<long long>(row) * ldy + col + e] = __float2half_rn(v);
        else reinterpret_cast<float*>(y)[static_cast<long long>(row) * ldy + col + e] = v;
      }
    }
  }
}

bool fc_small_supported(int64_t rows, int k, int n, int64_t x_ld, int64_t w_ld, const void* x, const void* w, int dtype) {
  const int per16 = 16 / elem_bytes(dtype);  // elements per 16 bytes
  return rows > 0 && k > 0 && n > 0 && k % per16 == 0 && x_ld % per16 == 0 && w_ld % per16 == 0 &&
         (reinterpret_cast<uintptr_t>(x) & 15u) == 0 && (reinterpret_cast<uintptr_t>(w) & 15u) == 0 && rows <= 0x7fffffffLL / FS_TILE;
}

int fc_small_dispatch(const void* x, int dtype, int64_t rows, int k, int64_t x_ld, const void* w, int n, int64_t w_ld, const float* bias,
                      int relu, void* y, int y_dtype, int64_t y_ld, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!x || !w || !y) return set_error(XVEC_E_ARG, "null pointer argument");
  if (!valid_dtype(dtype)) return set_error(XVEC_E_ARG, "bad dtype %d", dtype);
  if (!fc_small_supported(rows, k, n, x_ld, w_ld, x, w, dtype))
    return set_error(XVEC_E_ARG, "xvec_linear_small needs K and the row strides to be multiples of 16 bytes and 16-byte aligned operands");
  if (!valid_dtype(y_dtype)) return set_error(XVEC_E_ARG, "bad y_dtype %d", y_dtype);
  if (y_ld < n || x_ld < k || w_ld < k) return set_error(XVEC_E_ARG, "row stride smaller than the row");
  const dim3 grid((n + FS_TILE - 1) / FS_TILE, static_cast<unsigned>((rows + FS_TILE - 1) / FS_TILE));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int es = elem_bytes(dtype);
  const uint8_t* xb = static_cast<const uint8_t*>(x);
  const uint8_t* wb = static_cast<const uint8_t*>(w);
  const int m = static_cast<int>(rows);
#define XVEC_FS_LAUNCH(IN, OUT) \
  fc_small_kernel<IN, OUT><<<grid, 128, 0, st>>>(xb, x_ld * es, wb, w_ld * es, bias, m, n, k * es, relu, y, y_ld)
#define XVEC_FS_LAUNCH_OUT(IN)                                 \
  if (y_dtype == XVEC_BF16) XVEC_FS_LAUNCH(IN, XVEC_BF16);     \
  else if (y_dtype == XVEC_F16) XVEC_FS_LAUNCH(IN, XVEC_F16);  \
  else XVEC_FS_LAUNCH(IN, XVEC_F32)
  if (dtype == XVEC_BF16) {
    XVEC_FS_LAUNCH_OUT(XVEC_BF16);
  } else if (dtype == XVEC_F16) {
    XVEC_FS_LAUNCH_OUT(XVEC_F16);
  } else {
    XVEC_FS_LAUNCH_OUT(XVEC_F32);
  }
#undef XVEC_FS_LAUNCH_OUT
#undef XVEC_FS_LAUNCH
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(XVEC_E_CUDA, "fc_small_kernel launch: %s", cudaGetErrorString(e));
  return XVEC_OK;
}

}  // namespace xvec
