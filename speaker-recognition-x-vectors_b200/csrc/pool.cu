// Bandwidth-bound kernels of the extraction path: standalone statistics pooling (partial + finalize), the
// float32 -> bf16 / f16 cast, weight packing and per-trial cosine scoring.  sm_100a build; plain coalesced streaming code —
// these are HBM/L2-bound reductions, not tensor-core work.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "xvec_internal.h"

namespace xvec {

// ------------------------------------------------------------------------------------------------ stats pooling
// grid = (n_utts, max_chunks, ceil(p / 512)), block = 128: thread owns 4 adjacent columns, the CTA streams
// XVEC_POOL_CHUNK rows of one utterance; every row read is one contiguous <= 2 KiB segment per CTA.
// The sums are taken of x - pivot, pivot = the utterance's FIRST row (per column; written to pivot_out by chunk 0): a one-pass
// sum of squares in float32 loses the variance when |mean| >> std (mean 100, std 1: 1e4 * 2^-24 per term), the shifted sums
// do not, and mean / variance are shift-invariant — torch.std (main.py:61) is two-pass and has no such limit either.
template <bool kBf16>
__global__ void __launch_bounds__(128)
stats_pool_partial_kernel(const void* __restrict__ x, long long ld, int p, const long long* __restrict__ row_start,
                          const int* __restrict__ n_rows, const int* __restrict__ slot_start, float* __restrict__ part,
                          float* __restrict__ pivot_out) {
  const int u = blockIdx.x;
  const int nr = n_rows[u];
  const int r0 = blockIdx.y * XVEC_POOL_CHUNK;
  if (r0 >= nr) return;
  const int r1 = min(nr, r0 + XVEC_POOL_CHUNK);
  const int c = (blockIdx.z * 128 + threadIdx.x) * 4;
  if (c >= p) return;
  const long long first = row_start[u] + r0;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
  float4 pv = make_float4(0.f, 0.f, 0.f, 0.f);  // pivot: the utterance's first row (same for all of its chunks)
  auto acc = [&](float a, float b, float cc, float d) {
    a -= pv.x; b -= pv.y; cc -= pv.z; d -= pv.w;
    s0 += a; s1 += b; s2 += cc; s3 += d;
    q0 = fmaf(a, a, q0); q1 = fmaf(b, b, q1); q2 = fmaf(cc, cc, q2); q3 = fmaf(d, d, q3);
  };
  constexpr int U = 8;  // independent row loads in flight per thread
  int r = r0;
  if constexpr (kBf16) {
    const uint2* src = reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(x) + first * ld + c);
    const long long step = ld / 4;  // uint2 = 4 bf16
    if (pivot_out) {
      const uint2 w = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(x) + row_start[u] * ld + c));
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.x));
      const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.y));
      pv = make_float4(a.x, a.y, b.x, b.y);
    }
    for (; r + U <= r1; r += U) {
      uint2 v[U];
#pragma unroll
      for (int i = 0; i < U; ++i) v[i] = __ldcs(src + static_cast<long long>(r - r0 + i) * step);
#pragma unroll
      for (int i = 0; i < U; ++i) {
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[i].x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[i].y));
        acc(a.x, a.y, b.x, b.y);
      }
    }
    for (; r < r1; ++r) {
      const uint2 w = __ldcs(src + static_cast<long long>(r - r0) * step);
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.x));
      const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.y));
      acc(a.x, a.y, b.x, b.y);
    }
  } else {
    const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + first * ld + c);
    const long long step = ld / 4;
    if (pivot_out) pv = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + row_start[u] * ld + c));
    for (; r + U <= r1; r += U) {
      float4 v[U];
#pragma unroll
      for (int i = 0; i < U; ++i) v[i] = __ldcs(src + static_cast<long long>(r - r0 + i) * step);
#pragma unroll
      for (int i = 0; i < U; ++i) acc(v[i].x, v[i].y, v[i].z, v[i].w);
    }
    for (; r < r1; ++r) {
      const float4 w = __ldcs(src + static_cast<long long>(r - r0) * step);
      acc(w.x, w.y, w.z, w.w);
    }
  }
  if (pivot_out && blockIdx.y == 0) *reinterpret_cast<float4*>(pivot_out + static_cast<size_t>(u) * p + c) = pv;
  float* dst = part + static_cast<size_t>(slot_start[u] + blockIdx.y) * 2 * p + c;
  *reinterpret_cast<float4*>(dst) = make_float4(s0, s1, s2, s3);
  *reinterpret_cast<float4*>(dst + p) = make_float4(q0, q1, q2, q3);
}

// grid = (n_utts, ceil(p/128)), block = 128: fixed-order float64 reduction of an utterance's partial slots.
__global__ void __launch_bounds__(128)
pool_finalize_kernel(const float* __restrict__ part, const int* __restrict__ slot_start, const int* __restrict__ n_rows, int p,
                     const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ pivot,
                     float* __restrict__ out, void* __restrict__ out_lp, int lp_dtype, long long lp_ld) {
  const int u = blockIdx.x;
  const int col = blockIdx.y * 128 + threadIdx.x;
  __shared__ double inv_n[2];
  if (threadIdx.x == 0) {
    const int n0 = n_rows[u];
    inv_n[0] = n0 > 0 ? 1.0 / n0 : 0.0;
    inv_n[1] = n0 > 1 ? 1.0 / (n0 - 1) : 0.0;
  }
  __syncthreads();
  if (col >= p) return;
  const int sl0 = slot_start[u], sl1 = slot_start[u + 1];
  double S = 0.0, Q = 0.0;
  int sl = sl0;
  for (; sl + 4 <= sl1; sl += 4) {  // 8 independent loads in flight, summed in slot order
    float a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float* src = part + static_cast<size_t>(sl + i) * 2 * p + col;
      a[i] = src[0];
      b[i] = src[p];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      S += static_cast<double>(a[i]);
      Q += static_cast<double>(b[i]);
    }
  }
  for (; sl < sl1; ++sl) {  // a 3 s utterance has 3-4 slots of 128 frames
    const float* src = part + static_cast<size_t>(sl) * 2 * p + col;
    S += static_cast<double>(src[0]);
    Q += static_cast<double>(src[p]);
  }
  // 1/n and 1/(n-1) once per block (float64 division is a long software sequence; per thread it dominated this kernel)
  const int n = n_rows[u];
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  // the partial sums are of x - pivot (standalone pooling; the fused epilogue passes no pivot): the variance is unchanged
  const double mean = n > 0 ? S * inv_n[0] + (pivot ? static_cast<double>(pivot[static_cast<size_t>(u) * p + col]) : 0.0) : nan;
  double var = n > 1 ? (Q - S * S * inv_n[0]) * inv_n[1] : nan;  // torch.std: unbiased; a single frame gives NaN
  if (var < 0.0) var = 0.0;
  const float sc = scale ? scale[col] : 1.f;
  const float sh = shift ? shift[col] : 0.f;
  const float m = static_cast<float>(mean * sc + sh);
  const float sd = fabsf(sc) * sqrtf(static_cast<float>(var));  // the cancellation is resolved in float64, the root in float32
  out[static_cast<size_t>(u) * 2 * p + col] = m;
  out[static_cast<size_t>(u) * 2 * p + p + col] = sd;
  if (out_lp) {
    if (lp_dtype == XVEC_BF16) {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out_lp) + static_cast<size_t>(u) * lp_ld;
      o[col] = __float2bfloat16_rn(m);
      o[p + col] = __float2bfloat16_rn(sd);
    } else if (lp_dtype == XVEC_F16) {  // round to nearest, NaN stays NaN (a single-frame utterance, like torch.std)
      __half* o = reinterpret_cast<__half*>(out_lp) + static_cast<size_t>(u) * lp_ld;
      o[col] = __float2half_rn(m);
      o[p + col] = __float2half_rn(sd);
    } else {
      float* o = reinterpret_cast<float*>(out_lp) + static_cast<size_t>(u) * lp_ld;
      o[col] = m;
      o[p + col] = sd;
    }
  }
}

// ------------------------------------------------------------------------------------------------ layout expansion
// Expands per-utterance arrays into the per-row / per-128-row-block bookkeeping of the fused pooling epilogue, on the device
// (a ragged batch then only uploads 3 small per-utterance arrays instead of 4 bytes per frame).
//   row_utt[r]        = u if row r is one of the first n_pool[u] rows of utterance u, else -1
//   blk_slot_base[b]  = partial slot of the first utterance with a pooled row in 128-row block b
__global__ void __launch_bounds__(256)
build_layout_kernel(const int* __restrict__ starts, const int* __restrict__ n_pool, const int* __restrict__ slot_start, int n_utts,
                    int rows, int n_blocks, int* __restrict__ row_utt, int* __restrict__ blk_slot_base) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows) {
    int lo = 0, hi = n_utts - 1;  // last utterance with starts[u] <= i
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (starts[mid] <= i) lo = mid; else hi = mid - 1;
    }
    row_utt[i] = (i - starts[lo] < n_pool[lo]) ? lo : -1;
  }
  if (i < n_blocks) {
    const int first_row = i * XVEC_POOL_BLOCK;
    int lo = 0, hi = n_utts;  // first utterance whose last pooled row is >= first_row
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (starts[mid] + n_pool[mid] - 1 >= first_row) hi = mid; else lo = mid + 1;
    }
    int base = 0;
    if (lo < n_utts) {
      const int b0 = starts[lo] / XVEC_POOL_BLOCK;
      base = slot_start[lo] + (i > b0 ? i - b0 : 0);
    }
    blk_slot_base[i] = base;
  }
}

// ------------------------------------------------------------------------------------------------ cast / pack
__global__ void cast_kernel(const float* __restrict__ src, long long src_ld, void* __restrict__ dst, int dst_dtype, long long dst_ld,
                            long long rows, int cols) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols;
    const int c = static_cast<int>(i - r * cols);
    const float v = src[r * src_ld + c];
    if (dst_dtype == XVEC_BF16)
      reinterpret_cast<__nv_bfloat16*>(dst)[r * dst_ld + c] = __float2bfloat16_rn(v);
    else if (dst_dtype == XVEC_F16)
      reinterpret_cast<__half*>(dst)[r * dst_ld + c] = __float2half_rn(v);
    else
      reinterpret_cast<float*>(dst)[r * dst_ld + c] = v;
  }
}

__global__ void pack_weight_kernel(const float* __restrict__ w, int n, int taps, int cin, int tap_k, long long n_pad, long long k_pad,
                                   int dtype, void* __restrict__ out) {
  const long long total = n_pad * k_pad;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / k_pad;
    const int kk = static_cast<int>(i - row * k_pad);
    const int tap = kk / tap_k;
    const int ch = kk - tap * tap_k;
    const float v = (row < n && ch < cin) ? w[row * (static_cast<long long>(taps) * cin) + tap * cin + ch] : 0.f;
    // chunk-major: [K chunk of 128 bytes][row][element in chunk] — the 128-row x 128-byte box the GEMM producers load per
    // K chunk is then one contiguous 16 KiB run of global memory instead of 128 pieces k_pad*elsize bytes apart
    const int bke = dtype == XVEC_F32 ? 32 : 64;
    const long long o = (static_cast<long long>(kk / bke) * n_pad + row) * bke + kk % bke;
    if (dtype == XVEC_BF16)
      reinterpret_cast<__nv_bfloat16*>(out)[o] = __float2bfloat16_rn(v);
    else if (dtype == XVEC_F16)
      reinterpret_cast<__half*>(out)[o] = __float2half_rn(v);
    else
      reinterpret_cast<float*>(out)[o] = v;
  }
}

// ------------------------------------------------------------------------------------------------ cosine trials
// one warp per trial
__global__ void __launch_bounds__(256)
cosine_trials_kernel(const float* __restrict__ xv, long long ld, int dim, const float* __restrict__ mean, const int* __restrict__ enrol,
                     const int* __restrict__ test, long long n_trials, float* __restrict__ out) {
  const long long t = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (t >= n_trials) return;
  const float* a = xv + static_cast<long long>(enrol[t]) * ld;
  const float* b = xv + static_cast<long long>(test[t]) * ld;
  float ab = 0.f, aa = 0.f, bb = 0.f;
  for (int i = lane; i < dim; i += 32) {
    const float mu = mean ? mean[i] : 0.f;
    const float x = a[i] - mu, y = b[i] - mu;
    ab = fmaf(x, y, ab);
    aa = fmaf(x, x, aa);
    bb = fmaf(y, y, bb);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ab += __shfl_xor_sync(0xffffffffu, ab, o);
    aa += __shfl_xor_sync(0xffffffffu, aa, o);
    bb += __shfl_xor_sync(0xffffffffu, bb, o);
  }
  if (lane == 0) out[t] = ab * rsqrtf(aa) * rsqrtf(bb);
}

// ------------------------------------------------------------------------------------------------ PLDA trials
// out[r] = [hi(x_r) | x_r - hi(x_r) | hi(x_r)], hi = x with the 13 low mantissa bits cleared (exactly representable in TF32).
// With weights [W_hi ; W_hi ; W_lo] one TF32 GEMM over K = 3*cols computes x_hi W_hi + x_lo W_hi + x_hi W_lo, i.e. x W to ~2^-21.
__global__ void split_tf32_kernel(const float* __restrict__ x, long long ld, long long rows, int cols, float* __restrict__ out, long long out_ld) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols;
    const int c = static_cast<int>(i - r * cols);
    const float v = x[r * ld + c];
    const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    float* o = out + r * out_ld + c;
    o[0] = hi;
    o[cols] = v - hi;
    o[2 * cols] = hi;
  }
}
// q[i] = 1/2 <x_i - mean, y_i>   (y = (x - mean) Phi from the GEMM kernel): one warp per row
__global__ void __launch_bounds__(256)
plda_rowterm_kernel(const float* __restrict__ x, long long ld, int dim, const float* __restrict__ mean, const float* __restrict__ y,
                    long long y_ld, long long n, float* __restrict__ q) {
  const long long r = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n) return;
  float acc = 0.f;
  for (int i = lane; i < dim; i += 32) acc = fmaf(x[r * ld + i] - mean[i], y[r * y_ld + i], acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) q[r] = 0.5f * acc;
}
// score[t] = scale * (q[e] + q[s] + <p_e, x_s - mean> + cst)   (p = (x - mean) Psi): one warp per trial
__global__ void __launch_bounds__(256)
plda_trials_kernel(const float* __restrict__ x, long long ld, int dim, const float* __restrict__ mean, const float* __restrict__ p,
                   long long p_ld, const float* __restrict__ q, const int* __restrict__ enrol, const int* __restrict__ test,
                   long long n_trials, float cst, float scale, float* __restrict__ out) {
  const long long t = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (t >= n_trials) return;
  const int e = enrol[t], s = test[t];
  const float* pe = p + static_cast<long long>(e) * p_ld;
  const float* xs = x + static_cast<long long>(s) * ld;
  float acc = 0.f;
  for (int i = lane; i < dim; i += 32) acc = fmaf(pe[i], xs[i] - mean[i], acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[t] = scale * (q[e] + q[s] + acc + cst);
}

static int grid_for(long long total) {
  const long long want = (total + 255) / 256;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  return static_cast<int>(want < cap ? want : cap);
}

static int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(XVEC_E_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
  return XVEC_OK;
}

}  // namespace xvec

using namespace xvec;

extern "C" {

int xvec_build_layout(const int32_t* starts_dev, const int32_t* n_pool_dev, const int32_t* slot_start_dev, int n_utts, int64_t rows,
                      int32_t* row_utt_dev, int32_t* blk_slot_base_dev, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!starts_dev || !n_pool_dev || !slot_start_dev || !row_utt_dev || !blk_slot_base_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (n_utts <= 0 || rows <= 0 || rows > 0x7fffff00LL) return set_error(XVEC_E_ARG, "bad n_utts / rows");
  const int n_blocks = static_cast<int>((rows + 255) / 256) * (256 / XVEC_POOL_BLOCK);
  const long long n = rows > n_blocks ? rows : n_blocks;
  build_layout_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      starts_dev, n_pool_dev, slot_start_dev, n_utts, static_cast<int>(rows), n_blocks, row_utt_dev, blk_slot_base_dev);
  return check_launch("build_layout_kernel");
}

int xvec_stats_pool_partial(const void* x_dev, int x_dtype, int64_t x_ld, int p, const int64_t* row_start_dev,
                            const int32_t* n_rows_dev, const int32_t* slot_start_dev, int n_utts, int max_chunks, float* part_dev,
                            float* pivot_dev, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!x_dev || !row_start_dev || !n_rows_dev || !slot_start_dev || !part_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (x_dtype != XVEC_F32 && x_dtype != XVEC_BF16) return set_error(XVEC_E_ARG, "bad x_dtype %d", x_dtype);
  if (p <= 0 || p % 4 != 0 || x_ld % 4 != 0 || x_ld < p) return set_error(XVEC_E_ARG, "p and x_ld must be positive multiples of 4, x_ld >= p");
  const int align = x_dtype == XVEC_BF16 ? 8 : 16;
  if ((reinterpret_cast<uintptr_t>(x_dev) % align) != 0 || (reinterpret_cast<uintptr_t>(part_dev) & 15u) != 0 ||
      (reinterpret_cast<uintptr_t>(pivot_dev) & 15u) != 0)
    return set_error(XVEC_E_ARG, "x_dev / part_dev / pivot_dev are not sufficiently aligned");
  if (n_utts <= 0 || max_chunks <= 0 || max_chunks > 65535) return set_error(XVEC_E_ARG, "bad n_utts / max_chunks");
  dim3 grid(n_utts, max_chunks, (p + 511) / 512);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_dtype == XVEC_BF16)
    stats_pool_partial_kernel<true><<<grid, 128, 0, st>>>(x_dev, x_ld, p, reinterpret_cast<const long long*>(row_start_dev), n_rows_dev,
                                                         slot_start_dev, part_dev, pivot_dev);
  else
    stats_pool_partial_kernel<false><<<grid, 128, 0, st>>>(x_dev, x_ld, p, reinterpret_cast<const long long*>(row_start_dev), n_rows_dev,
                                                          slot_start_dev, part_dev, pivot_dev);
  return check_launch("stats_pool_partial_kernel");
}

int xvec_pool_finalize(const float* part_dev, const int32_t* slot_start_dev, const int32_t* n_rows_dev, int n_utts, int p,
                       const float* bn_scale_dev, const float* bn_shift_dev, const float* pivot_dev, float* out_f32_dev, void* out_lp_dev,
                       int out_lp_dtype, int64_t out_lp_ld, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!part_dev || !slot_start_dev || !n_rows_dev || !out_f32_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (n_utts <= 0 || p <= 0) return set_error(XVEC_E_ARG, "non-positive size");
  if ((bn_scale_dev == nullptr) != (bn_shift_dev == nullptr)) return set_error(XVEC_E_ARG, "bn_scale and bn_shift must be given together");
  if (out_lp_dev && !valid_dtype(out_lp_dtype)) return set_error(XVEC_E_ARG, "bad out_lp_dtype");
  if (out_lp_dev && out_lp_ld < 2 * p) return set_error(XVEC_E_ARG, "out_lp_ld < 2p");
  dim3 grid(n_utts, (p + 127) / 128);
  pool_finalize_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(part_dev, slot_start_dev, n_rows_dev, p, bn_scale_dev,
                                                                            bn_shift_dev, pivot_dev, out_f32_dev, out_lp_dev, out_lp_dtype,
                                                                            out_lp_ld);
  return check_launch("pool_finalize_kernel");
}

int xvec_cast(const float* src_dev, int64_t src_ld, void* dst_dev, int dst_dtype, int64_t dst_ld, int64_t rows, int cols, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!src_dev || !dst_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (rows <= 0 || cols <= 0 || src_ld < cols || dst_ld < cols) return set_error(XVEC_E_ARG, "bad shape");
  if (!valid_dtype(dst_dtype)) return set_error(XVEC_E_ARG, "bad dst_dtype");
  const long long total = rows * cols;
  const int blocks = grid_for(total);
  cast_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(src_dev, src_ld, dst_dev, dst_dtype, dst_ld, rows, cols);
  return check_launch("cast_kernel");
}

int xvec_pack_weight(const float* w_dev, int n, int taps, int cin, int dtype, void* out_dev, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!w_dev || !out_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (n <= 0 || cin <= 0 || taps < 1 || taps > XVEC_MAX_TAPS) return set_error(XVEC_E_ARG, "bad shape");
  if (!valid_dtype(dtype)) return set_error(XVEC_E_ARG, "bad dtype");
  const long long k_pad = xvec_packed_k(cin, taps, dtype);
  const long long n_pad = xvec_packed_n(n);
  const long long total = n_pad * k_pad;
  const int blocks = grid_for(total);
  pack_weight_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(w_dev, n, taps, cin, static_cast<int>(k_pad / taps), n_pad,
                                                                           k_pad, dtype, out_dev);
  return check_launch("pack_weight_kernel");
}

int xvec_cosine_trials(const float* xvec_dev, int64_t ld, int dim, const float* mean_dev, const int32_t* enrol_dev,
                       const int32_t* test_dev, int64_t n_trials, float* out_dev, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!xvec_dev || !enrol_dev || !test_dev || !out_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (dim <= 0 || ld < dim || n_trials <= 0) return set_error(XVEC_E_ARG, "bad shape");
  const long long blocks = (n_trials * 32 + 255) / 256;
  cosine_trials_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(xvec_dev, ld, dim, mean_dev, enrol_dev,
                                                                                                   test_dev, n_trials, out_dev);
  return check_launch("cosine_trials_kernel");
}

int xvec_split_tf32(const float* x_dev, int64_t ld, int64_t rows, int cols, float* out_dev, int64_t out_ld, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!x_dev || !out_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (rows <= 0 || cols <= 0 || ld < cols || out_ld < 3 * static_cast<int64_t>(cols)) return set_error(XVEC_E_ARG, "bad shape");
  split_tf32_kernel<<<grid_for(rows * cols), 256, 0, static_cast<cudaStream_t>(stream)>>>(x_dev, ld, rows, cols, out_dev, out_ld);
  return check_launch("split_tf32_kernel");
}

int xvec_plda_rowterm(const float* x_dev, int64_t ld, int dim, const float* mean_dev, const float* y_dev, int64_t y_ld, int64_t n,
                      float* q_dev, void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!x_dev || !mean_dev || !y_dev || !q_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (dim <= 0 || ld < dim || y_ld < dim || n <= 0) return set_error(XVEC_E_ARG, "bad shape");
  const long long blocks = (n * 32 + 255) / 256;
  plda_rowterm_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(x_dev, ld, dim, mean_dev, y_dev, y_ld, n, q_dev);
  return check_launch("plda_rowterm_kernel");
}

int xvec_plda_trials(const float* x_dev, int64_t ld, int dim, const float* mean_dev, const float* p_dev, int64_t p_ld, const float* q_dev,
                     const int32_t* enrol_dev, const int32_t* test_dev, int64_t n_trials, float cst, float scale, float* out_dev,
                     void* stream) {
  int rc = device_check();
  if (rc) return rc;
  if (!x_dev || !mean_dev || !p_dev || !q_dev || !enrol_dev || !test_dev || !out_dev) return set_error(XVEC_E_ARG, "null pointer argument");
  if (dim <= 0 || ld < dim || p_ld < dim || n_trials <= 0) return set_error(XVEC_E_ARG, "bad shape");
  const long long blocks = (n_trials * 32 + 255) / 256;
  plda_trials_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(x_dev, ld, dim, mean_dev, p_dev, p_ld, q_dev,
                                                                                                 enrol_dev, test_dev, n_trials, cst, scale, out_dev);
  return check_launch("plda_trials_kernel");
}

}  // extern "C"
