// extern "C" surface of libxvec_b200.so (declared in include/xvec_b200.h) + small host utilities.
#include <stdarg.h>
#include <stdio.h>

#include "xvec_internal.h"

namespace xvec {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

namespace {
struct DevInfo {
  int checked = 0;  // 0 unknown, 1 ok, -1 unsupported
  int sms = 0;
  int major = 0, minor = 0;
};
DevInfo g_dev[64];

DevInfo* cur_dev() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return nullptr;
  DevInfo* di = &g_dev[d];
  if (!di->checked) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, d) != cudaSuccess) return nullptr;
    di->sms = prop.multiProcessorCount;
    di->major = prop.major;
    di->minor = prop.minor;
    di->checked = (prop.major == 10) ? 1 : -1;
  }
  return di;
}
}  // namespace

int device_check() {
  DevInfo* di = cur_dev();
  if (!di) return set_error(XVEC_E_CUDA, "no usable CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
  if (di->checked < 0)
    return set_error(XVEC_E_DEVICE, "device is sm_%d%d; these kernels are built for sm_100a only (no fallback)", di->major, di->minor);
  return XVEC_OK;
}

int num_sms() {
  DevInfo* di = cur_dev();
  return di ? di->sms : 1;
}

PFN_encodeTiled get_encode_tiled() {
  static const PFN_encodeTiled fn = [] {  // initialised once, thread-safe (C++11 local static)
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      return reinterpret_cast<PFN_encodeTiled>(p);
    return static_cast<PFN_encodeTiled>(nullptr);
  }();
  return fn;
}

unsigned int* watchdog_host_word() {
  static std::mutex mu;
  static unsigned int* word = nullptr;
  std::lock_guard<std::mutex> lock(mu);
  if (!word) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return nullptr;
    word = static_cast<unsigned int*>(p);
    *word = 0u;
  }
  return word;
}

int read_watchdog() {
  unsigned int* w = watchdog_host_word();
  return w ? static_cast<int>(*reinterpret_cast<volatile unsigned int*>(w)) : 0;
}

int layer_desc(XvecLayerDesc* l, const void* w_packed, const float* bias, int n, int cin, int taps, int dtype, const int32_t* tap_offsets) {
  if (!tap_offsets) return set_error(XVEC_E_ARG, "tap_offsets_host is NULL");
  if (taps < 1 || taps > XVEC_MAX_TAPS) return set_error(XVEC_E_ARG, "taps must be in [1,%d]", XVEC_MAX_TAPS);
  *l = XvecLayerDesc{};
  l->w_packed_dev = w_packed;
  l->bias_dev = bias;
  l->n = n;
  l->cin = cin;
  l->taps = taps;
  l->dtype = dtype;
  for (int j = 0; j < taps; ++j) l->tap_offsets[j] = tap_offsets[j];
  return XVEC_OK;
}

}  // namespace xvec

using namespace xvec;

extern "C" {

int xvec_abi_version(void) { return XVEC_ABI_VERSION; }
const char* xvec_last_error(void) { return g_err; }
int xvec_device_check(void) { return device_check(); }
int xvec_watchdog_code(void) {
  cudaDeviceSynchronize();  // after a trap this reports the sticky launch failure; the word lives in host memory
  return read_watchdog();
}
void xvec_watchdog_reset(void) {
  if (unsigned int* w = watchdog_host_word()) *reinterpret_cast<volatile unsigned int*>(w) = 0u;
}

int xvec_debug_trace(long long* out_host, int n) { return read_trace(out_host, n); }

int64_t xvec_packed_k(int cin, int taps, int dtype) {
  const int kc = chunk_elems(dtype);
  return static_cast<int64_t>(taps) * ((cin + kc - 1) / kc) * kc;
}
int64_t xvec_splitk_workspace_bytes(int64_t rows, int cin, int taps, int n, int dtype) {
  if (rows <= 0 || cin <= 0 || taps < 1 || n <= 0) return 0;
  return splitk_workspace_bytes(rows, cin, taps, n, dtype);
}
int64_t xvec_packed_n(int n) { return static_cast<int64_t>((n + XVEC_TILE_N - 1) / XVEC_TILE_N) * XVEC_TILE_N; }

int xvec_tdnn_layer(const void* x_dev, int x_dtype, int64_t x_rows, int cin, int64_t x_ld, const void* w_packed_dev, int n,
                    const int32_t* tap_offsets_host, int taps, const float* bias_dev, const float* bn_scale_dev,
                    const float* bn_shift_dev, int relu, void* y_dev, int y_dtype, int64_t y_ld, int64_t rows, void* splitk_ws_dev,
                    int64_t splitk_ws_bytes, void* stream) {
  XvecLayerDesc l;
  const int rc = layer_desc(&l, w_packed_dev, bias_dev, n, cin, taps, x_dtype, tap_offsets_host);
  if (rc) return rc;
  return gemm_store(l, x_dev, x_rows, x_ld, rows, bn_scale_dev, bn_shift_dev, relu, y_dev, y_dtype, y_ld, splitk_ws_dev, splitk_ws_bytes,
                    stream);
}

int xvec_tdnn_pool_fused(const void* x_dev, int x_dtype, int64_t x_rows, int cin, int64_t x_ld, const void* w_packed_dev, int n,
                         const int32_t* tap_offsets_host, int taps, const float* bias_dev, const int32_t* row_utt_dev,
                         const int32_t* blk_slot_base_dev, float* part_dev, int64_t rows, void* stream) {
  XvecLayerDesc l;
  const int rc = layer_desc(&l, w_packed_dev, bias_dev, n, cin, taps, x_dtype, tap_offsets_host);
  if (rc) return rc;
  return gemm_pool(l, x_dev, x_rows, x_ld, rows, row_utt_dev, blk_slot_base_dev, part_dev, stream);
}

int64_t xvec_stack_ctrl_bytes(int64_t rows, int n_tdnn) { return stack_ctrl_bytes(rows, n_tdnn); }
int64_t xvec_stack_plan(int64_t rows, int n_layers, const int32_t* n_tiles_per_layer_host, int band, uint32_t* items_out_host,
                        int64_t capacity) {
  return stack_plan(rows, n_layers, n_tiles_per_layer_host, band, items_out_host, capacity);
}

int xvec_linear_small(const void* x_dev, int dtype, int64_t rows, int k, int64_t x_ld, const void* w_dev, int n, int64_t w_ld,
                      const float* bias_dev, int relu, void* y_dev, int y_dtype, int64_t y_ld, void* stream) {
  return fc_small_dispatch(x_dev, dtype, rows, k, x_ld, w_dev, n, w_ld, bias_dev, relu, y_dev, y_dtype, y_ld, stream);
}

int xvec_tdnn_stack(const XvecLayerDesc* tdnn, int n_tdnn, const void* x_dev, int64_t rows, int64_t x_ld, void* act0_dev, void* act1_dev,
                    int64_t act_ld, const int32_t* row_utt_dev, const int32_t* blk_slot_base_dev, float* part_dev, void* ctrl_dev,
                    int64_t ctrl_bytes, int band, void* stream) {
  if (!tdnn) return set_error(XVEC_E_ARG, "tdnn_host is NULL");
  return stack_dispatch(tdnn, n_tdnn, x_dev, rows, x_ld, act0_dev, act1_dev, act_ld, row_utt_dev, blk_slot_base_dev, part_dev, ctrl_dev,
                        ctrl_bytes, band, stream);
}

// Frame-level stack of xvec_extract_forward: the persistent stack kernel when given its scratch and the stack fits it, else one
// launch per layer.
static int frame_stack(const XvecLayerDesc* tdnn, int n_tdnn, const void* x, int64_t rows, int64_t x_ld, void* act0, void* act1,
                       int64_t act_ld, const int32_t* row_utt, const int32_t* blk_slot_base, float* part, void* ctrl, int64_t ctrl_bytes,
                       void* stream) {
  if (ctrl && stack_supported(tdnn, n_tdnn, rows))
    return stack_dispatch(tdnn, n_tdnn, x, rows, x_ld, act0, act1, act_ld, row_utt, blk_slot_base, part, ctrl, ctrl_bytes, 0, stream);
  void* act[2] = {act0, act1};
  const void* h = x;
  int64_t h_ld = x_ld;
  for (int i = 0; i + 1 < n_tdnn; ++i) {
    const int rc = gemm_store(tdnn[i], h, rows, h_ld, rows, nullptr, nullptr, 1, act[i & 1], tdnn[i + 1].dtype, act_ld, nullptr, 0, stream);
    if (rc) return rc;
    h = act[i & 1];
    h_ld = act_ld;
  }
  return gemm_pool(tdnn[n_tdnn - 1], h, rows, h_ld, rows, row_utt, blk_slot_base, part, stream);
}

// Segment head of xvec_extract_forward: n_fc layers on the pooled statistics `a`, ReLU between them, none after the last.
static int segment_head(const XvecLayerDesc* fc, int n_fc, const void* a, int64_t a_ld, int n_utts, void* fc_tmp, void* splitk_ws,
                        int64_t splitk_ws_bytes, float* out, int64_t out_ld, void* stream) {
  for (int i = 0; i < n_fc; ++i) {
    const XvecLayerDesc& l = fc[i];
    const bool final_layer = i == n_fc - 1;
    void* y = final_layer ? static_cast<void*>(out) : fc_tmp;
    const int y_dtype = final_layer ? XVEC_F32 : fc[i + 1].dtype;
    const int64_t y_ld = final_layer ? out_ld : l.n;
    const int relu = final_layer ? 0 : 1;
    int rc;
    if (l.w_plain_dev && fc_small_supported(n_utts, l.cin, l.n, a_ld, l.cin, a, l.w_plain_dev, l.dtype))
      // small-footprint kernel: runs next to the resident stack CTAs of the next batch instead of waiting for free SMs
      rc = fc_small_dispatch(a, l.dtype, n_utts, l.cin, a_ld, l.w_plain_dev, l.n, l.cin, l.bias_dev, relu, y, y_dtype, y_ld, stream);
    else
      rc = gemm_store(l, a, n_utts, a_ld, n_utts, nullptr, nullptr, relu, y, y_dtype, y_ld, splitk_ws, splitk_ws_bytes, stream);
    if (rc) return rc;
    a = y;
    a_ld = y_ld;
  }
  return XVEC_OK;
}

int xvec_extract_forward(const XvecLayerDesc* tdnn, int n_tdnn, const void* x_dev, int64_t rows, int64_t x_ld, void* act0_dev,
                         void* act1_dev, int64_t act_ld, const int32_t* row_utt_dev, const int32_t* blk_slot_base_dev,
                         const int32_t* utt_slot_start_dev, const int32_t* n_pool_dev, int n_utts, float* part_dev,
                         const float* bn_last_scale_dev, const float* bn_last_shift_dev, float* pooled_dev, void* pooled_lp_dev,
                         const XvecLayerDesc* fc, int n_fc, void* fc_tmp_dev, void* splitk_ws_dev, int64_t splitk_ws_bytes,
                         float* out_dev, int64_t out_ld, void* ctrl_dev, int64_t ctrl_bytes, void* stream) {
  if (!tdnn || n_tdnn < 2 || n_fc < 0 || n_fc > 2 || (n_fc > 0 && !fc))
    return set_error(XVEC_E_ARG, "need >= 2 TDNN layers and 0 to 2 segment layers");
  if (!x_dev || !act0_dev || !act1_dev || !pooled_dev || (n_fc > 0 && !out_dev)) return set_error(XVEC_E_ARG, "null pointer argument");
  if (n_fc == 2 && !fc_tmp_dev) return set_error(XVEC_E_ARG, "fc_tmp_dev is NULL");
  // lp_head: the first segment layer is 16-bit and reads the pooled statistics in its own dtype
  const bool lp_head = n_fc > 0 && (fc[0].dtype == XVEC_BF16 || fc[0].dtype == XVEC_F16);
  if (lp_head && !pooled_lp_dev) return set_error(XVEC_E_ARG, "pooled_lp_dev is required for 16-bit segment layers");
  // the 16-bit copy: in the first segment layer's dtype when that reads it, else (n_fc == 0: the caller runs the head itself) in
  // float16 for a float16 frame stack, else in bfloat16
  const int lp_dtype = lp_head ? fc[0].dtype : tdnn[n_tdnn - 1].dtype == XVEC_F16 ? XVEC_F16 : XVEC_BF16;
  int rc = frame_stack(tdnn, n_tdnn, x_dev, rows, x_ld, act0_dev, act1_dev, act_ld, row_utt_dev, blk_slot_base_dev, part_dev, ctrl_dev,
                       ctrl_bytes, stream);
  if (rc) return rc;
  const int64_t pooled_ld = 2 * static_cast<int64_t>(tdnn[n_tdnn - 1].n);
  rc = xvec_pool_finalize(part_dev, utt_slot_start_dev, n_pool_dev, n_utts, tdnn[n_tdnn - 1].n, bn_last_scale_dev, bn_last_shift_dev, nullptr,
                          pooled_dev, pooled_lp_dev, lp_dtype, pooled_ld, stream);
  if (rc) return rc;
  return segment_head(fc, n_fc, lp_head ? pooled_lp_dev : static_cast<const void*>(pooled_dev), pooled_ld, n_utts, fc_tmp_dev, splitk_ws_dev,
                      splitk_ws_bytes, out_dev, out_ld, stream);
}

}  // extern "C"
