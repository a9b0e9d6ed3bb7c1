// Host-side helpers shared by the translation units of libxvec_b200.so (not part of the public ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <mutex>

#include "../../include/xvec_b200.h"

namespace xvec {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Records a message for xvec_last_error() (thread local) and returns `code`.
int set_error(int code, const char* fmt, ...);
// XVEC_OK when the current device is compute capability 10.x.
int device_check();
int num_sms();
// Driver entry point for tensor-map creation, resolved through the runtime (no link-time libcuda dependency).
PFN_encodeTiled get_encode_tiled();

// Elements of `dtype` in one 128-byte K chunk of a packed operand: 32 float32 (TF32 math) or 64 bfloat16 / float16.
inline int chunk_elems(int dtype) { return dtype == XVEC_F32 ? 32 : 64; }
// Bytes per element of XVEC_F32 / XVEC_BF16 / XVEC_F16.
inline int elem_bytes(int dtype) { return dtype == XVEC_F32 ? 4 : 2; }
// The element types of activations and packed weights.
inline bool valid_dtype(int dtype) { return dtype == XVEC_F32 || dtype == XVEC_BF16 || dtype == XVEC_F16; }

// `l` with the given operands and zeros everywhere else (tap slots past `taps`, w_plain_dev); XVEC_E_ARG for bad taps.
int layer_desc(XvecLayerDesc* l, const void* w_packed, const float* bias, int n, int cin, int taps, int dtype, const int32_t* tap_offsets);
// tdnn_gemm.cu: layer `l` as a tcgen05 GEMM over output rows [0, rows) of x ((x_rows, l.cin) of l.dtype, row stride x_ld).
// gemm_store: as xvec_tdnn_layer (split-K over `ws` when that helps and ws is large enough); gemm_pool: as xvec_tdnn_pool_fused.
int gemm_store(const XvecLayerDesc& l, const void* x, int64_t x_rows, int64_t x_ld, int64_t rows, const float* bn_scale,
               const float* bn_shift, int relu, void* y, int y_dtype, int64_t y_ld, void* ws, int64_t ws_bytes, void* stream);
int gemm_pool(const XvecLayerDesc& l, const void* x, int64_t x_rows, int64_t x_ld, int64_t rows, const int32_t* row_utt,
              const int32_t* blk_slot_base, float* part, void* stream);
// tdnn_stack.cu: all TDNN layers (the last one fused with the pooling partials) as one persistent kernel.
bool stack_supported(const XvecLayerDesc* tdnn, int n_tdnn, int64_t rows);
int64_t stack_ctrl_bytes(int64_t rows, int n_layers);
int64_t stack_plan(int64_t rows, int n_layers, const int32_t* n_tiles_per_layer, int band, uint32_t* items_out, int64_t capacity);
int stack_dispatch(const XvecLayerDesc* tdnn, int n_tdnn, const void* x, int64_t rows, int64_t x_ld, void* act0, void* act1,
                   int64_t act_ld, const int32_t* row_utt, const int32_t* blk_slot_base, float* part, void* ctrl, int64_t ctrl_bytes,
                   int band, void* stream);
// fc_small.cu: small-footprint linear layer (mma.sync) that co-resides with the persistent stack kernel.
bool fc_small_supported(int64_t rows, int k, int n, int64_t x_ld, int64_t w_ld, const void* x, const void* w, int dtype);
int fc_small_dispatch(const void* x, int dtype, int64_t rows, int k, int64_t x_ld, const void* w, int n, int64_t w_ld, const float* bias,
                      int relu, void* y, int y_dtype, int64_t y_ld, void* stream);
int64_t splitk_workspace_bytes(int64_t rows, int cin, int taps, int n, int dtype);

// Per-device one-time initialisation (cudaFuncSetAttribute, binding the watchdog word) that is safe when several host threads
// — one per device or several per device — make their first call at the same time.
struct PerDeviceInit {
  std::mutex mu;
  std::atomic<bool> done[64];
  PerDeviceInit() {
    for (auto& d : done) d.store(false, std::memory_order_relaxed);
  }
};
template <class F>
inline int once_per_device(PerDeviceInit& s, F&& f) {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return f();
  if (s.done[dev].load(std::memory_order_acquire)) return XVEC_OK;
  std::lock_guard<std::mutex> lock(s.mu);
  if (!s.done[dev].load(std::memory_order_relaxed)) {
    const int rc = f();
    if (rc) return rc;
    s.done[dev].store(true, std::memory_order_release);
  }
  return XVEC_OK;
}

// The watchdog word: ONE unsigned int of mapped, pinned, portable host memory (it outlives a trapped context).  Kernels
// write it through their TU's g_watchdog_ptr (ptx.cuh), which XVEC_DEFINE_WATCHDOG_BINDER's function binds once per device.
unsigned int* watchdog_host_word();
int read_watchdog();
int bind_watchdog_gemm();   // tdnn_gemm.cu
int bind_watchdog_stack();  // tdnn_stack.cu
#define XVEC_DEFINE_WATCHDOG_BINDER(fn)                                                                               \
  int fn() {                                                                                                          \
    static PerDeviceInit once;                                                                                        \
    return once_per_device(once, [] {                                                                                 \
      unsigned int* w = watchdog_host_word();                                                                         \
      if (!w) return set_error(XVEC_E_CUDA, "cudaHostAlloc(watchdog word) failed");                                   \
      cudaError_t e = cudaMemcpyToSymbol(g_watchdog_ptr, &w, sizeof(w));                                              \
      if (e != cudaSuccess) return set_error(XVEC_E_CUDA, "cudaMemcpyToSymbol(watchdog): %s", cudaGetErrorString(e)); \
      return static_cast<int>(XVEC_OK);                                                                               \
    });                                                                                                               \
  }
int read_trace(long long* out_host, int n);

}  // namespace xvec
