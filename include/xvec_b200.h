/* xvec_b200.h — C ABI of the B200-native x-vector extraction path (libxvec_b200.so).
 *
 * The reference (TorbenHellriegel/Speaker-Recognition-x-vectors) has no FFI / plugin registry: its boundary
 * is the PyTorch nn.Module surface (tdnn_layer.py:5-41 TdnnLayer, main.py:23-94 XVectorModel).  These entry
 * points are what a binding for that surface calls; each names the reference code it replaces.  The Python
 * mirror of the module surface lives in speaker-recognition-x-vectors_b200/{tdnn_layer,xvector}.py and
 * reaches this library through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every `*_dev` pointer is DEVICE memory owned by the caller, `*_host` is host memory
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns without synchronising
 *   - return 0 on success, a negative XVEC_E_* code otherwise; xvec_last_error() describes the last failure of
 *     the calling thread.  Nothing throws across the ABI.  There is no CPU fallback: a device that is not
 *     sm_100 yields XVEC_E_DEVICE.
 *   - frames are laid out as ONE flat row-major frame matrix (total_frames x channels): utterance u occupies
 *     rows [start_u, start_u + T_u).  A TDNN layer computes output row r from input rows r + offset_j, so
 *     every layer keeps the same row indexing; the last (c_last - c_0) rows of each utterance become
 *     don't-care rows that pooling masks out.  No unfolded (time-context) tensor is ever written to memory.
 */
#ifndef XVEC_B200_H_
#define XVEC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XVEC_ABI_VERSION 8

#if defined(__GNUC__)
#define XVEC_API __attribute__((visibility("default")))
#else
#define XVEC_API
#endif

/* element types of activations / packed weights */
#define XVEC_F32 0  /* float32 storage, tensor-core math in TF32 (kind::tf32), fp32 accumulate */
#define XVEC_BF16 1 /* bfloat16 storage, kind::f16 bf16 math, fp32 accumulate */
#define XVEC_F16 2  /* float16 storage, kind::f16 f16 math, fp32 accumulate: the 10-bit mantissa of TF32 operands at the rate and
                       bytes of bf16, range |x| < 65504 (a larger activation becomes +inf, see DESIGN.md section 4) */

#define XVEC_OK 0
#define XVEC_E_ARG (-1)    /* bad shape / alignment / null pointer */
#define XVEC_E_CUDA (-2)   /* a CUDA runtime or driver call failed */
#define XVEC_E_DEVICE (-3) /* current device is not compute capability 10.x */

#define XVEC_MAX_TAPS 8
#define XVEC_TILE_N 256     /* output-channel tile; packed weights are padded to a multiple of this many rows */
#define XVEC_POOL_BLOCK 128 /* rows per pooling partial block of the fused TDNN5+pool epilogue */
#define XVEC_POOL_CHUNK 128 /* rows per partial of the standalone statistics-pooling kernel */
#define XVEC_MAX_STACK 6           /* TDNN layers xvec_tdnn_stack can chain in one launch */
#define XVEC_STACK_MAX_BANDS 512   /* scheduling bands of xvec_tdnn_stack (internal table size) */
#define XVEC_STACK_MAX_TAP_OFFSET 8 /* largest c_j - c_0 xvec_tdnn_stack takes (one activation slab holds 128 + 8 frame rows) */

XVEC_API int xvec_abi_version(void);
XVEC_API const char* xvec_last_error(void);
/* 0 if the current CUDA device can run these kernels (compute capability 10.x), else XVEC_E_DEVICE. */
XVEC_API int xvec_device_check(void);
/* Value left by the device-side pipeline watchdog (0 = never fired): every mbarrier wait / flag spin of the tcgen05 kernels
 * traps after a bounded number of polls and first writes which wait it was (1-8) into a word of mapped HOST memory, so the code
 * survives the failed launch (a trap destroys the context).  Synchronises the device.  xvec_watchdog_reset() clears it. */
XVEC_API int xvec_watchdog_code(void);
XVEC_API void xvec_watchdog_reset(void);

/* Developer aid: with XVEC_TRACE=1 in the environment the GEMM kernel records per-tile clock64 stamps of CTA 0;
 * copies up to n of them to out_host and returns the count (0 when tracing is off). */
XVEC_API int xvec_debug_trace(long long* out_host, int n);

/* Number of K elements one packed weight row holds: taps * ceil(cin / kc) * kc, kc = 32 (F32) or 64 (BF16, F16). */
XVEC_API int64_t xvec_packed_k(int cin, int taps, int dtype);
/* Rows of a packed weight matrix: n rounded up to XVEC_TILE_N. */
XVEC_API int64_t xvec_packed_n(int n);

/* Pack a Linear weight for xvec_tdnn_layer.
 * replaces: the layout nn.Linear(input_size*len(context), output_size) stores (tdnn_layer.py:19): W (n, taps*cin)
 * row-major, column index = tap*cin + channel (context-major, because of torch.cat(..., 2) at tdnn_layer.py:29).
 * w_dev: float32 (n, taps*cin); dtype XVEC_F32, XVEC_BF16 or XVEC_F16 (round to nearest).  out_dev: xvec_packed_n(n) * xvec_packed_k(cin,taps,dtype) elements of `dtype`, zero padded,
 * stored K-chunk-major ([128-byte K chunk][row][element]: every 128-row x 128-byte TMA box is one contiguous 16 KiB run);
 * the layout is private to this library — treat the buffer as opaque. */
XVEC_API int xvec_pack_weight(const float* w_dev, int n, int taps, int cin, int dtype, void* out_dev, void* stream);

/* One TDNN layer on the flat frame matrix, no unfold in memory:
 *   y[r, :] = bn( relu( sum_j W_j . x[r + tap_offsets[j], :] + bias ) ),  r in [0, rows)
 * replaces: TdnnLayer.forward (tdnn_layer.py:26-41) = get_time_context (tdnn_layer.py:43-60) + torch.cat +
 * nn.Linear + ReLU + eval-mode BatchNorm1d; with taps == 1 and relu/bn optional it is also nn.Linear
 * (segment_layer6/7, output: main.py:45-47, 87-90, 71-74).
 *   x_dev      (x_rows, cin) of x_dtype (XVEC_F32 / XVEC_BF16 / XVEC_F16), row stride x_ld elements (x_ld*elsize multiple of 16 bytes, base 16-byte aligned)
 *   w_packed   from xvec_pack_weight with the same taps/cin/dtype
 *   tap_offsets_host  taps non-negative row offsets c_j - c_0 (HOST array)
 *   bias_dev   float32 or NULL;  bn_scale_dev/bn_shift_dev float32 or both NULL:
 *              scale = gamma/sqrt(running_var+eps), shift = beta - running_mean*scale.
 *              These vectors are read 32 columns at a time: each must be 16-byte aligned and hold ceil(n/32)*32 floats.
 *   y_dev      (rows, n) of y_dtype (XVEC_F32 / XVEC_BF16 / XVEC_F16), row stride y_ld elements.  Input rows beyond x_rows read as zero.
 *   splitk_ws_dev / splitk_ws_bytes  optional scratch (16-byte aligned) of at least xvec_splitk_workspace_bytes(...)
 *              bytes: when the GEMM has too few output tiles to fill the GPU (segment6: a few hundred rows, K = 3000)
 *              the K loop is split over CTA pairs into this workspace and a fixed-order second pass applies the
 *              epilogue.  NULL / too small = no split (slower, same result up to fp32 summation order).
 */
XVEC_API int xvec_tdnn_layer(const void* x_dev, int x_dtype, int64_t x_rows, int cin, int64_t x_ld,
                    const void* w_packed_dev, int n, const int32_t* tap_offsets_host, int taps,
                    const float* bias_dev, const float* bn_scale_dev, const float* bn_shift_dev, int relu,
                    void* y_dev, int y_dtype, int64_t y_ld, int64_t rows, void* splitk_ws_dev, int64_t splitk_ws_bytes,
                    void* stream);
/* Scratch bytes xvec_tdnn_layer can use for split-K on this shape (0 = it would not split). */
XVEC_API int64_t xvec_splitk_workspace_bytes(int64_t rows, int cin, int taps, int n, int dtype);

/* Last TDNN layer fused with the first half of statistics pooling: the (rows x n) activation
 * r = relu(W.x + bias) is never written; per XVEC_POOL_BLOCK-row block and utterance the kernel emits column sums of
 * r and r*r into part_dev[slot][2][n] (float32).  BatchNorm of this layer is applied by xvec_pool_finalize.
 * replaces: TdnnLayer #5 (main.py:43) + the reads of torch.mean/torch.std in stat_pool (main.py:59-63).
 *   row_utt_dev        int32 (rows): utterance index of a row that takes part in pooling, -1 for don't-care rows
 *   blk_slot_base_dev  int32 (ceil(rows/256)*2): first partial slot of each 128-row block (slots of a block are
 *                      consecutive, one per utterance with a pooled row in it, in row order)
 */
XVEC_API int xvec_tdnn_pool_fused(const void* x_dev, int x_dtype, int64_t x_rows, int cin, int64_t x_ld,
                         const void* w_packed_dev, int n, const int32_t* tap_offsets_host, int taps,
                         const float* bias_dev, const int32_t* row_utt_dev, const int32_t* blk_slot_base_dev,
                         float* part_dev, int64_t rows, void* stream);

/* Expands per-utterance arrays (device, int32: first row, pooled-frame count, exclusive prefix sum of partial slots — see
 * xvec_tdnn_pool_fused) into row_utt_dev (rows) and blk_slot_base_dev (ceil(rows/256)*2) on the device, so a ragged batch
 * uploads 12 bytes per utterance instead of 4 bytes per frame.  The reference has no counterpart (fixed 3 s cuts, dataset.py:204). */
XVEC_API int xvec_build_layout(const int32_t* starts_dev, const int32_t* n_pool_dev, const int32_t* slot_start_dev, int n_utts,
                      int64_t rows, int32_t* row_utt_dev, int32_t* blk_slot_base_dev, void* stream);

/* Standalone statistics pooling, first half (bandwidth-bound streaming reduction): for utterance u and chunk j,
 * column sums of x and x*x over rows [row_start[u] + j*XVEC_POOL_CHUNK, ...) -> part_dev[slot_start[u] + j][2][p].
 * replaces: the reads of torch.mean / torch.std in XVectorModel.stat_pool (main.py:59-63) on a materialised
 * (B, T', p) activation; ragged lengths are an extension (the reference pads/cuts to 3 s, dataset.py:204).
 *   x_dev (.., p) of x_dtype (XVEC_F32 or XVEC_BF16; XVEC_F16 is not taken) with row stride x_ld elements; p multiple of 4
 *   row_start_dev int64 (n_utts), n_rows_dev int32 (n_utts), slot_start_dev int32 (n_utts+1) = exclusive prefix
 *   sum of ceil(n_rows/XVEC_POOL_CHUNK); max_chunks = max over utterances of that count.
 *   pivot_dev float32 (n_utts, p), 16-byte aligned, or NULL: when given, the sums are taken of x - pivot with pivot = the
 *   utterance's first row (written here, passed on to xvec_pool_finalize) — a one-pass float32 sum of squares otherwise loses
 *   the variance of inputs with |mean| >> std, which the reference's two-pass torch.std (main.py:61) does not.
 */
XVEC_API int xvec_stats_pool_partial(const void* x_dev, int x_dtype, int64_t x_ld, int p, const int64_t* row_start_dev,
                            const int32_t* n_rows_dev, const int32_t* slot_start_dev, int n_utts, int max_chunks,
                            float* part_dev, float* pivot_dev, void* stream);

/* Statistics pooling, second half: deterministic fixed-order (float64) reduction of an utterance's partial slots
 * [slot_start[u], slot_start[u+1]) and the final statistics
 *   mean = s*(S/n) + h,   std = |s| * sqrt( (Q - S*S/n) / (n-1) )       (unbiased, torch.std default; n==1 -> NaN)
 * replaces: torch.mean, torch.std, torch.cat in stat_pool (main.py:60-62) (+ the BatchNorm of TDNN5 folded
 * through the statistics when bn_scale/shift are given; both NULL = plain pooling).
 *   pivot_dev float32 (n_utts, p) or NULL: the partial sums are of x - pivot (xvec_stats_pool_partial); the mean gets it back.
 *   out_f32_dev float32 (n_utts, 2p) [mean || std], row stride 2p;  out_lp_dev optional second copy in out_lp_dtype (XVEC_F32,
 *   XVEC_BF16 or XVEC_F16; NaN stays NaN) with row stride out_lp_ld (feeds segment_layer6 directly), or NULL.
 */
XVEC_API int xvec_pool_finalize(const float* part_dev, const int32_t* slot_start_dev, const int32_t* n_rows_dev, int n_utts,
                       int p, const float* bn_scale_dev, const float* bn_shift_dev, const float* pivot_dev, float* out_f32_dev,
                       void* out_lp_dev, int out_lp_dtype, int64_t out_lp_ld, void* stream);

/* One layer of xvec_extract_forward: a TDNN layer (taps >= 1) or a fully connected layer (taps == 1), operands already
 * packed with xvec_pack_weight in `dtype`; bias as for xvec_tdnn_layer (ceil(n/32)*32 floats) or NULL. */
typedef struct XvecLayerDesc {
  const void* w_packed_dev;
  const float* bias_dev;
  int32_t n;      /* output channels */
  int32_t cin;    /* input channels per tap */
  int32_t taps;
  int32_t dtype;  /* XVEC_F32 / XVEC_BF16 / XVEC_F16: element type of this layer's INPUT activations and packed weights */
  int32_t tap_offsets[XVEC_MAX_TAPS];
  const void* w_plain_dev; /* segment layers only, optional: the nn.Linear weight itself in `dtype`, (n, cin) row-major, row
                              stride cin — lets xvec_extract_forward run the layer with xvec_linear_small; NULL otherwise */
} XvecLayerDesc;

/* The frame-level stack in ONE persistent kernel launch: TDNN layers 0..n_tdnn-2 (bias + ReLU, activations ping-ponged through
 * act0/act1) and the last TDNN layer fused with the pooling partials (as xvec_tdnn_pool_fused).  Every (layer, 256-frame tile,
 * 256-channel tile) is a work item drawn in order from a global counter by the CTA pairs; a tile of layer l+1 starts as soon as
 * the tiles of layer l it reads are complete (per-tile flags in ctrl_dev), so the layers overlap inside the launch.
 * replaces: time_context_layers (main.py:38-44) applied by extract_x_vec (main.py:82) + the reads of stat_pool (main.py:59-63).
 *   x_dev is of tdnn_host[0].dtype; layers 1.. share one dtype (the activation dtype: XVEC_F32, XVEC_BF16 or XVEC_F16); layer 0
 *   is XVEC_F32 (TF32 math) or the activation dtype (a float32 layer 0 with XVEC_BF16 activations may also be XVEC_BF16); layers 0..n-2 need n % XVEC_TILE_N == 0
 *   and a bias; eval-mode BatchNorm folded forward as for xvec_extract_forward.
 *   Window form of a layer with consecutive taps (context [-2..2] of TDNN1, tdnn_layer.py:43-60): when its input rows are
 *   dense (x_ld == channels) the taps*channels window of output row r is ONE contiguous run starting at row r, so the layer
 *   may be described as taps = 1, cin = taps*channels with the real row stride x_ld = channels (rows overlap; the natural
 *   nn.Linear weight is already in window order).  Rows whose window would run past the end of x (the last taps - 1 rows, which
 *   are don't-care rows of the last utterance anyway) read as zero; nothing past the end of x_dev is touched.
 *   xvec_tdnn_layer / xvec_tdnn_pool_fused accept the same form.
 *   ctrl_dev: 128-byte aligned scratch of xvec_stack_ctrl_bytes(rows, n_tdnn) bytes, private to this call until it completes
 *   (the call zeroes it on `stream`).  band: m-tiles per scheduling band, 0 = the library's choice (any value gives the same
 *   bits; tests sweep it).  Tap offsets up to XVEC_STACK_MAX_TAP_OFFSET.  Returns XVEC_E_ARG for stacks outside these limits
 *   (use the per-layer calls).  The encoded tensor maps of the last 64 distinct argument sets are cached inside the library. */
XVEC_API int64_t xvec_stack_ctrl_bytes(int64_t rows, int n_tdnn);
/* Host-side replay of xvec_tdnn_stack's work-item order (needs no GPU; used by the CPU tests): items_out_host[i] =
 * layer | n_tile << 3 | m_tile << 8 of the i-th item the CTA pairs draw, for n_layers layers with n_tiles_per_layer_host[]
 * 256-channel tiles over `rows` frame rows; band = m-tiles per scheduling band, 0 = the library's default.  Returns the
 * number of items (writes at most `capacity` of them; items_out_host may be NULL) or a negative XVEC_E_* code.
 * The order must list every (layer, m_tile, n_tile) once and every tile after the tiles (layer-1, m_tile-1 .. m_tile+1) it
 * depends on: with in-order drawing that is what makes the dependency waits deadlock-free. */
XVEC_API int64_t xvec_stack_plan(int64_t rows, int n_layers, const int32_t* n_tiles_per_layer_host, int band, uint32_t* items_out_host,
                        int64_t capacity);
XVEC_API int xvec_tdnn_stack(const struct XvecLayerDesc* tdnn_host, int n_tdnn, const void* x_dev, int64_t rows, int64_t x_ld,
                    void* act0_dev, void* act1_dev, int64_t act_ld, const int32_t* row_utt_dev, const int32_t* blk_slot_base_dev,
                    float* part_dev, void* ctrl_dev, int64_t ctrl_bytes, int band, void* stream);

/* Small-footprint linear layer: y = act(x W' + bias), x (rows, k) and W (n, k) row-major (the nn.Linear layout, NOT packed) of
 * `dtype` (XVEC_BF16, XVEC_F16, or XVEC_F32 = TF32 math), float32 accumulation, y float32, bfloat16 or float16 (y_dtype).  128 threads, 5 KiB of shared
 * memory, no tensor memory: its CTAs fit next to a resident CTA of the persistent xvec_tdnn_stack kernel, so the segment layers
 * of one batch run concurrently with the frame-level stack of the next one instead of waiting for free SMs.
 * replaces: segment_layer6 / segment_layer7 (main.py:45-46, 87-90) on the pooled statistics.
 * k, x_ld, w_ld multiples of 16 bytes of elements; x_dev / w_dev 16-byte aligned; bias_dev float32 (n) or NULL. */
XVEC_API int xvec_linear_small(const void* x_dev, int dtype, int64_t rows, int k, int64_t x_ld, const void* w_dev, int n, int64_t w_ld,
                      const float* bias_dev, int relu, void* y_dev, int y_dtype, int64_t y_ld, void* stream);

/* The whole extraction path for one flat batch in ONE call (3 kernel launches + one small memset enqueued on `stream`; the tensor
 * maps of recurring argument sets are cached): xvec_tdnn_stack, xvec_pool_finalize, then the n_fc segment layers (ReLU between
 * them, none after the last; xvec_linear_small when the layer carries w_plain_dev, else xvec_tdnn_layer with split-K).
 * Without ctrl_dev (NULL) or for a stack xvec_tdnn_stack does not take, the TDNN layers run as one launch each
 * (xvec_tdnn_layer / xvec_tdnn_pool_fused) — same results.
 * replaces: XVectorModel.extract_x_vec (main.py:81-94) = time_context_layers (main.py:38-44) + stat_pool (:59-63) +
 * segment_layer6 [+ relu + segment_layer7]; eval-mode BatchNorm of layers 0..n-2 must already be folded into the next
 * layer's packed weights, the last TDNN layer's BatchNorm is passed as bn_last_scale/shift (or NULL).
 *   x_dev (rows, tdnn[0].cin) of tdnn[0].dtype, row stride x_ld (window form: see xvec_tdnn_stack);  act0/act1: ping-pong activation buffers (rows, act_ld) of the
 *   dtype of tdnn[1];  layout arrays as for xvec_tdnn_pool_fused / xvec_pool_finalize;  part_dev (n_slots, 2, n_last);
 *   pooled_dev float32 (n_utts, 2 n_last);  pooled_lp_dev NULL or a 16-bit copy of it (n_utts, 2 n_last): in fc[0].dtype when that
 *   is XVEC_BF16 or XVEC_F16 (the first segment layer reads it; required then), else in float16 when the TDNN layers are
 *   XVEC_F16, else in bfloat16;  fc: n_fc segment layers (taps == 1);
 *   fc_tmp_dev (n_utts, fc[0].n) of fc[1].dtype when n_fc == 2;  out_dev float32 (n_utts, fc[n_fc-1].n), row stride out_ld;
 *   splitk_ws_dev: scratch for the segment layers (see xvec_splitk_workspace_bytes) or NULL;
 *   ctrl_dev / ctrl_bytes: scratch of xvec_tdnn_stack or NULL / 0.
 *   n_fc == 0 ends the call after xvec_pool_finalize; fc_host, fc_tmp_dev, splitk_ws_dev and out_dev may then be NULL. */
XVEC_API int xvec_extract_forward(const XvecLayerDesc* tdnn_host, int n_tdnn, const void* x_dev, int64_t rows, int64_t x_ld,
                         void* act0_dev, void* act1_dev, int64_t act_ld, const int32_t* row_utt_dev,
                         const int32_t* blk_slot_base_dev, const int32_t* utt_slot_start_dev, const int32_t* n_pool_dev,
                         int n_utts, float* part_dev, const float* bn_last_scale_dev, const float* bn_last_shift_dev,
                         float* pooled_dev, void* pooled_lp_dev, const XvecLayerDesc* fc_host, int n_fc, void* fc_tmp_dev,
                         void* splitk_ws_dev, int64_t splitk_ws_bytes, float* out_dev, int64_t out_ld, void* ctrl_dev,
                         int64_t ctrl_bytes, void* stream);

/* MFCC front end (the step BEFORE the path; SURVEY §8 row f4): waveform -> (frames, 24) float32 rows of the flat frame
 * matrix, with the reference's fixed parameters: 16 kHz, pre-emphasis 0.97, 400-sample frames every 160 samples (zero padded,
 * rectangular window), 512-point power spectrum / 512, 26 triangular mel filters on integer bins, log, orthonormal DCT-II
 * (first 24), lifter 22, coefficient 0 = log frame energy.
 * replaces: python_speech_features.mfcc(sample, 16000, numcep=24, nfilt=26, nfft=512) (dataset.py:130); that package is not
 * available offline, so parity for this entry point is UNPINNED (checked against oracle/mfcc_oracle.py only).
 *   wav_dev        float32 or int16 samples of all utterances; utterance u = wav[wav_start[u] .. + wav_len[u])
 *   row_start_dev  int64 first output row of utterance u; n_frames_dev int32 = xvec_mfcc_num_frames(wav_len[u])
 *   norm_offset_dev / norm_scale_dev  optional per-utterance affine applied to the samples first, x' = (x + offset) * scale
 *                  (from xvec_wav_minmax = the reference's min-max normalisation, dataset.py:217-218), or both NULL
 *   out_dev        (total_frames, >= 24) float32 with row stride out_ld */
XVEC_API int64_t xvec_mfcc_num_frames(int64_t n_samples);
XVEC_API int xvec_mfcc(const void* wav_dev, int wav_is_int16, const int64_t* wav_start_dev, const int32_t* wav_len_dev,
              const int64_t* row_start_dev, const int32_t* n_frames_dev, int n_utts, int max_frames,
              const float* norm_offset_dev, const float* norm_scale_dev, float* out_dev, int64_t out_ld, void* stream);
/* Per-utterance (offset, scale) = (-min, 1/(max-min)) of the raw samples: x -= min(x); x /= max(x) (dataset.py:217-218). */
XVEC_API int xvec_wav_minmax(const void* wav_dev, int wav_is_int16, const int64_t* wav_start_dev, const int32_t* wav_len_dev,
                    int n_utts, float* norm_offset_dev, float* norm_scale_dev, void* stream);

/* float32 -> dtype copy of a (rows, cols) matrix (row strides in elements); XVEC_F32 is a strided copy, XVEC_BF16 / XVEC_F16 round
 * to nearest (NaN stays NaN).
 * replaces: samples.float() (main.py:137) for the 16-bit pipelines. */
XVEC_API int xvec_cast(const float* src_dev, int64_t src_ld, void* dst_dev, int dst_dtype, int64_t dst_ld, int64_t rows,
              int cols, void* stream);

/* Cosine score of each trial: out[i] = <a,b>/(|a||b|) with a = xvec[enrol[i]] - mean, b = xvec[test[i]] - mean
 * (float32 in, float32 out, float32 accumulation; mean_dev float32 (dim) or NULL for no centring).
 * BASELINE.json config 5; the reference scores with PLDA on the full NxN matrix and picks trial entries afterwards
 * (plda_score_stat.py:59-87). */
XVEC_API int xvec_cosine_trials(const float* xvec_dev, int64_t ld, int dim, const float* mean_dev, const int32_t* enrol_dev,
                       const int32_t* test_dev, int64_t n_trials, float* out_dev, void* stream);

/* PLDA log-likelihood-ratio scoring of trials (two-covariance model mean / F / Sigma), without the N x N score matrix:
 *   score[t] = scale * ( q[e] + q[s] + <p_e, x_s - mean> + cst ),   q_i = 1/2 <x_i - mean, (x_i - mean) Phi>,   p = (x - mean) Psi
 * replaces: plda_classifier.plda_scores (plda_classifier.py:81-87, speechbrain.processing.PLDA_LDA.fast_PLDA_scoring) + the
 * per-trial lookup loop plda_score_stat.py:59-87.  Phi, Psi, cst come from the model on the host (float64, once per model);
 * y = (x - mean) Phi and p = (x - mean) Psi are two xvec_tdnn_layer GEMMs (taps = 1, bias = -mean Phi / -mean Psi) run as
 * split-TF32: xvec_split_tf32 writes [hi(x) | x - hi(x) | hi(x)] (hi = TF32-exact part) and the weights are packed as
 * [W_hi | W_hi | W_lo], so one TF32 GEMM over K = 3 dim gives x W to ~2^-21 relative (plain TF32 would move scores by 1e-3 of
 * their magnitude — more than the gap between neighbouring trial scores at the decision threshold).
 * SpeechBrain is not vendored with the reference: parity for these two entry points is UNPINNED (checked against
 * oracle/plda_oracle.py, which is itself checked against the model's Gaussian definition). */
XVEC_API int xvec_split_tf32(const float* x_dev, int64_t ld, int64_t rows, int cols, float* out_dev, int64_t out_ld, void* stream);
XVEC_API int xvec_plda_rowterm(const float* x_dev, int64_t ld, int dim, const float* mean_dev, const float* y_dev, int64_t y_ld,
                      int64_t n, float* q_dev, void* stream);
XVEC_API int xvec_plda_trials(const float* x_dev, int64_t ld, int dim, const float* mean_dev, const float* p_dev, int64_t p_ld,
                     const float* q_dev, const int32_t* enrol_dev, const int32_t* test_dev, int64_t n_trials, float cst, float scale,
                     float* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* XVEC_B200_H_ */
