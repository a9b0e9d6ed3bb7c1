"""Functional wrappers: torch CUDA tensors in, C-ABI calls on the current CUDA stream, torch CUDA tensors out.

torch is plumbing here (device memory, streams); every FLOP and every reduction happens in libxvec_b200.so.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._lib import BF16, F32, check, dtype_code, ptr, stream_ptr, taps_array


_POOL_LAYOUTS = {}


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise ValueError("xvec_b200 has no CPU path: tensors must live on a CUDA device")


def _rowmajor_2d(t: torch.Tensor, what: str):
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError(f"{what} must be a 2-D tensor with unit stride in the last dimension")
    return t.stride(0)


def pad32(vec: torch.Tensor | None) -> torch.Tensor | None:
    """Column-parameter vectors are read 32 floats at a time by the epilogue: float32, contiguous, padded with zeros."""
    if vec is None:
        return None
    v = vec.detach().to(torch.float32).contiguous()
    n = v.numel()
    m = (n + 31) // 32 * 32
    if m == n:
        return v
    out = torch.zeros(m, dtype=torch.float32, device=v.device)
    out[:n] = v
    return out


def pack_weight(weight: torch.Tensor, taps: int, cin: int, dtype: torch.dtype) -> torch.Tensor:
    """nn.Linear weight (n, taps*cin) float32 -> packed (n_pad, k_pad) operand for xvec_tdnn_layer, in float32, bfloat16 or
    float16 (round to nearest)."""
    _require_cuda(weight)
    lib = _lib.load()
    w = weight.detach().to(torch.float32).contiguous()
    n = w.shape[0]
    if w.shape[1] != taps * cin:
        raise ValueError(f"weight has {w.shape[1]} columns, expected taps*cin = {taps * cin}")
    code = dtype_code(dtype)
    out = torch.empty((lib.xvec_packed_n(n), lib.xvec_packed_k(cin, taps, code)), dtype=dtype, device=w.device)
    with _lib.on_device(w.device):
        check(lib.xvec_pack_weight(ptr(w), n, taps, cin, code, ptr(out), stream_ptr()))
    return out


def tdnn_layer_flat(x: torch.Tensor, w_packed: torch.Tensor, n: int, offsets, bias=None, bn_scale=None, bn_shift=None,
                    relu: bool = True, out: torch.Tensor | None = None, out_dtype: torch.dtype | None = None, cin: int | None = None,
                    workspace: torch.Tensor | None = None):
    """y[r] = bn(relu(sum_j W_j x[r + offsets[j]] + bias)) over a flat (rows, cin) frame matrix; returns (rows, n).
    x and w_packed: float32 (TF32 math), bfloat16 or float16; the output dtype is any of the three."""
    _require_cuda(x, w_packed, bias, bn_scale, bn_shift, out)
    lib = _lib.load()
    x_ld = _rowmajor_2d(x, "x")
    rows = x.shape[0]
    cin = x.shape[1] if cin is None else cin
    if out is None:
        out = torch.empty((rows, n), dtype=out_dtype or x.dtype, device=x.device)
    y_ld = _rowmajor_2d(out, "out")
    if out.shape[0] != rows or out.shape[1] != n:
        raise ValueError("out must be (rows, n)")
    if w_packed.dtype != x.dtype:
        raise ValueError("packed weights and activations must share a dtype")
    need = (n + 31) // 32 * 32
    bias, bn_scale, bn_shift = [v if v is None or (v.numel() >= need and v.dtype == torch.float32) else pad32(v)
                                for v in (bias, bn_scale, bn_shift)]
    offs = taps_array(offsets)
    ws_bytes = 0 if workspace is None else workspace.numel() * workspace.element_size()
    with _lib.on_device(x.device):
        check(lib.xvec_tdnn_layer(ptr(x), dtype_code(x.dtype), rows, cin, x_ld, ptr(w_packed), n, offs, len(offsets),
                                  ptr(bias), ptr(bn_scale), ptr(bn_shift), int(bool(relu)), ptr(out), dtype_code(out.dtype),
                                  y_ld, rows, ptr(workspace), ws_bytes, stream_ptr()))
    return out


def splitk_workspace(rows: int, cin: int, taps: int, n: int, dtype: torch.dtype, device) -> torch.Tensor | None:
    """Scratch for split-K on this GEMM shape, or None when the shape fills the GPU without it."""
    nbytes = _lib.load().xvec_splitk_workspace_bytes(rows, cin, taps, n, dtype_code(dtype))
    return torch.empty(nbytes, dtype=torch.uint8, device=device) if nbytes > 0 else None


def tdnn_pool_fused(x: torch.Tensor, w_packed: torch.Tensor, n: int, offsets, bias, row_utt: torch.Tensor,
                    blk_slot_base: torch.Tensor, part: torch.Tensor):
    """Last TDNN layer with the pooling sums fused into its epilogue; fills part (n_slots, 2, n) float32."""
    _require_cuda(x, w_packed, bias, row_utt, blk_slot_base, part)
    lib = _lib.load()
    x_ld = _rowmajor_2d(x, "x")
    rows = x.shape[0]
    if row_utt.dtype != torch.int32 or blk_slot_base.dtype != torch.int32 or part.dtype != torch.float32:
        raise ValueError("row_utt / blk_slot_base must be int32, part float32")
    if row_utt.numel() < rows or blk_slot_base.numel() < ((rows + 255) // 256) * (256 // _lib.POOL_BLOCK) or not part.is_contiguous():
        raise ValueError("pooling bookkeeping arrays are too small for this frame matrix")
    offs = taps_array(offsets)
    with _lib.on_device(x.device):
        check(lib.xvec_tdnn_pool_fused(ptr(x), dtype_code(x.dtype), rows, x.shape[1], x_ld, ptr(w_packed), n, offs, len(offsets),
                                       ptr(bias), ptr(row_utt), ptr(blk_slot_base), ptr(part), rows, stream_ptr()))
    return part


def tdnn_stack(layer_descs, n_layers: int, x: torch.Tensor, act0: torch.Tensor, act1: torch.Tensor, row_utt: torch.Tensor,
               blk_slot_base: torch.Tensor, part: torch.Tensor, ctrl: torch.Tensor, band: int = 0):
    """All TDNN layers of the stack in one persistent launch (xvec_tdnn_stack): layers 0..n-2 ping-pong through act0/act1,
    the last one fills the pooling partials `part`.  layer_descs: ctypes array of _lib.LayerDesc (packed operands);
    band: m-tiles per scheduling band (0 = the library's choice; every value gives the same bits)."""
    _require_cuda(x, act0, act1, row_utt, blk_slot_base, part, ctrl)
    lib = _lib.load()
    x_ld = _rowmajor_2d(x, "x")
    act_ld = _rowmajor_2d(act0, "act0")
    rows = x.shape[0]
    if dtype_code(x.dtype) != layer_descs[0].dtype or act0.dtype != act1.dtype or _rowmajor_2d(act1, "act1") != act_ld:
        raise ValueError("x must have the dtype of layer 0; act0 / act1 must share dtype and row stride")
    if act0.shape[0] < rows or act1.shape[0] < rows:
        raise ValueError("activation buffers are too small for this frame matrix")
    if row_utt.numel() < rows or blk_slot_base.numel() < ((rows + 255) // 256) * (256 // _lib.POOL_BLOCK) or not part.is_contiguous():
        raise ValueError("pooling bookkeeping arrays are too small for this frame matrix")
    with _lib.on_device(x.device):
        check(lib.xvec_tdnn_stack(layer_descs, n_layers, ptr(x), rows, x_ld, ptr(act0), ptr(act1), act_ld, ptr(row_utt), ptr(blk_slot_base),
                                  ptr(part), ptr(ctrl), ctrl.numel(), int(band), stream_ptr()))
    return part


def pool_finalize(part: torch.Tensor, slot_start: torch.Tensor, n_rows: torch.Tensor, p: int, bn_scale=None, bn_shift=None,
                  out: torch.Tensor | None = None, out_lp: torch.Tensor | None = None, pivot: torch.Tensor | None = None):
    """[mean || unbiased std] per utterance from partial sums; returns float32 (n_utts, 2p).  pivot: float32 (n_utts, p) when
    the partial sums were taken of x - pivot (stats_pool_ragged)."""
    _require_cuda(part, slot_start, n_rows, bn_scale, bn_shift, out, out_lp, pivot)
    if pivot is not None and (pivot.dtype != torch.float32 or not pivot.is_contiguous() or pivot.shape != (n_rows.numel(), p)):
        raise ValueError("pivot must be contiguous float32 (n_utts, p)")
    lib = _lib.load()
    n_utts = n_rows.numel()
    if out is None:
        out = torch.empty((n_utts, 2 * p), dtype=torch.float32, device=part.device)
    if not out.is_contiguous() or out.shape != (n_utts, 2 * p) or out.dtype != torch.float32:
        raise ValueError("out must be contiguous float32 (n_utts, 2p)")
    lp_code, lp_ld = F32, 0
    if out_lp is not None:
        lp_ld = _rowmajor_2d(out_lp, "out_lp")
        lp_code = dtype_code(out_lp.dtype)
    with _lib.on_device(part.device):
        check(lib.xvec_pool_finalize(ptr(part), ptr(slot_start), ptr(n_rows), n_utts, p, ptr(bn_scale), ptr(bn_shift), ptr(pivot), ptr(out),
                                     ptr(out_lp), lp_code, lp_ld, stream_ptr()))
    return out


def build_layout_device(starts: torch.Tensor, n_pool: torch.Tensor, slot_start: torch.Tensor, rows: int, row_utt: torch.Tensor,
                        blk_slot_base: torch.Tensor) -> None:
    """Expand per-utterance int32 device arrays into row_utt (rows) / blk_slot_base (ceil(rows/256)*8) on the device."""
    _require_cuda(starts, n_pool, slot_start, row_utt, blk_slot_base)
    lib = _lib.load()
    if any(t.dtype != torch.int32 or not t.is_contiguous() for t in (starts, n_pool, slot_start, row_utt, blk_slot_base)):
        raise ValueError("layout arrays must be contiguous int32")
    if row_utt.numel() < rows or blk_slot_base.numel() < ((rows + 255) // 256) * (256 // _lib.POOL_BLOCK) or slot_start.numel() < starts.numel() + 1:
        raise ValueError("layout output arrays are too small")
    with _lib.on_device(starts.device):
        check(lib.xvec_build_layout(ptr(starts), ptr(n_pool), ptr(slot_start), starts.numel(), rows, ptr(row_utt), ptr(blk_slot_base),
                                    stream_ptr()))


def stats_pool_ragged(x: torch.Tensor, row_start: np.ndarray, n_rows: np.ndarray, out_lp: torch.Tensor | None = None):
    """Standalone statistics pooling over row ranges of a flat (rows, p) matrix -> float32 (n_utts, 2p)."""
    _require_cuda(x)
    lib = _lib.load()
    ld = _rowmajor_2d(x, "x")
    p = x.shape[1]
    row_start = np.asarray(row_start, dtype=np.int64)
    n_rows = np.asarray(n_rows, dtype=np.int32)
    if (n_rows < 1).any():
        raise ValueError("every utterance needs at least one frame to pool")
    if (row_start < 0).any() or ((row_start + n_rows) > x.shape[0]).any():
        raise ValueError("row range outside of x")
    dev = x.device
    key = (row_start.tobytes(), n_rows.tobytes(), str(dev))
    hit = _POOL_LAYOUTS.get(key)
    if hit is None:  # small index arrays: uploaded once per distinct (row_start, n_rows) and cached
        chunks = (n_rows.astype(np.int64) + _lib.POOL_CHUNK - 1) // _lib.POOL_CHUNK
        slot_start = np.concatenate(([0], np.cumsum(chunks))).astype(np.int32)
        hit = (torch.from_numpy(row_start).to(dev), torch.from_numpy(n_rows).to(dev), torch.from_numpy(slot_start).to(dev),
               int(slot_start[-1]), int(chunks.max()))
        if len(_POOL_LAYOUTS) >= 8:
            _POOL_LAYOUTS.pop(next(iter(_POOL_LAYOUTS)))
        _POOL_LAYOUTS[key] = hit
    rs_d, nr_d, ss_d, n_slots, max_chunks = hit
    part = torch.empty((n_slots, 2, p), dtype=torch.float32, device=dev)
    pivot = torch.empty((len(n_rows), p), dtype=torch.float32, device=dev)  # each utterance's first row: the sums are shifted by it
    with _lib.on_device(dev):
        check(lib.xvec_stats_pool_partial(ptr(x), dtype_code(x.dtype), ld, p, ptr(rs_d), ptr(nr_d), ptr(ss_d), len(n_rows),
                                          max_chunks, ptr(part), ptr(pivot), stream_ptr()))
    return pool_finalize(part, ss_d, nr_d, p, out_lp=out_lp, pivot=pivot)


def mfcc(wav: torch.Tensor, wav_lengths, normalize: bool = True, out: torch.Tensor | None = None):
    """Waveforms -> flat MFCC frame matrix on the GPU.  `wav` is a 1-D CUDA tensor (float32 or int16) holding all utterances
    back to back, `wav_lengths` their sample counts.  normalize=True applies the reference's per-utterance min-max
    normalisation first.  Returns (flat (sum frames, 24) float32, frame counts int64 numpy) — exactly what
    XVectorModel.extract_x_vec_flat takes."""
    _require_cuda(wav, out)
    lib = _lib.load()
    if wav.dim() != 1 or wav.dtype not in (torch.float32, torch.int16) or not wav.is_contiguous():
        raise ValueError("wav must be a contiguous 1-D float32 or int16 tensor")
    wl = np.asarray(wav_lengths, dtype=np.int64).reshape(-1)
    if wl.size == 0 or (wl <= 0).any() or int(wl.sum()) != wav.numel() or wl.max() >= 2**31:
        raise ValueError("wav_lengths must be positive and sum to wav.numel()")
    if wl.size > 65535:
        raise ValueError("at most 65535 utterances per call")
    nf = np.asarray([lib.xvec_mfcc_num_frames(int(v)) for v in wl], dtype=np.int64)
    wstart = np.concatenate(([0], np.cumsum(wl)[:-1]))
    rstart = np.concatenate(([0], np.cumsum(nf)[:-1]))
    dev = wav.device
    meta64 = torch.from_numpy(np.stack([wstart, rstart])).to(dev)
    meta32 = torch.from_numpy(np.stack([wl, nf]).astype(np.int32)).to(dev)
    total = int(nf.sum())
    if out is None:
        out = torch.empty((total, 24), dtype=torch.float32, device=dev)
    if out.dim() != 2 or out.shape[0] != total or out.shape[1] < 24 or out.stride(1) != 1 or out.dtype != torch.float32:
        raise ValueError("out must be float32 (sum frames, >=24) with unit column stride")
    is16 = int(wav.dtype == torch.int16)
    with _lib.on_device(dev):
        off = scl = None
        if normalize:
            off = torch.empty(wl.size, dtype=torch.float32, device=dev)
            scl = torch.empty(wl.size, dtype=torch.float32, device=dev)
            check(lib.xvec_wav_minmax(ptr(wav), is16, ptr(meta64[0]), ptr(meta32[0]), wl.size, ptr(off), ptr(scl), stream_ptr()))
        check(lib.xvec_mfcc(ptr(wav), is16, ptr(meta64[0]), ptr(meta32[0]), ptr(meta64[1]), ptr(meta32[1]), wl.size, int(nf.max()),
                            ptr(off), ptr(scl), ptr(out), out.stride(0), stream_ptr()))
    return out, nf


def cast(src: torch.Tensor, dtype: torch.dtype, out: torch.Tensor | None = None) -> torch.Tensor:
    """float32 -> float32 / bfloat16 / float16 copy (round to nearest; NaN stays NaN)."""
    _require_cuda(src, out)
    lib = _lib.load()
    if src.dtype != torch.float32:
        raise ValueError("cast source must be float32")
    s_ld = _rowmajor_2d(src, "src")
    if out is None:
        out = torch.empty(src.shape, dtype=dtype, device=src.device)
    d_ld = _rowmajor_2d(out, "out")
    with _lib.on_device(src.device):
        check(lib.xvec_cast(ptr(src), s_ld, ptr(out), dtype_code(out.dtype), d_ld, src.shape[0], src.shape[1], stream_ptr()))
    return out


def cosine_trials(xvecs: torch.Tensor, enrol: torch.Tensor, test: torch.Tensor, center: bool = False) -> torch.Tensor:
    """Cosine score of every (enrol, test) index pair; float32 (n_trials).  center=True subtracts the mean x-vector of
    the set first (computed by the statistics-pooling kernel over the (N, dim) matrix)."""
    _require_cuda(xvecs, enrol, test)
    lib = _lib.load()
    if xvecs.dtype != torch.float32 or enrol.dtype != torch.int32 or test.dtype != torch.int32:
        raise ValueError("xvecs must be float32, trial indices int32")
    ld = _rowmajor_2d(xvecs, "xvecs")
    n = enrol.numel()
    if test.numel() != n:
        raise ValueError("enrol and test must have the same length")
    out = torch.empty(n, dtype=torch.float32, device=xvecs.device)
    mean = None
    if center:
        mean = stats_pool_ragged(xvecs, np.zeros(1, np.int64), np.asarray([xvecs.shape[0]], np.int32))[0, : xvecs.shape[1]].contiguous()
    with _lib.on_device(xvecs.device):
        check(lib.xvec_cosine_trials(ptr(xvecs), ld, xvecs.shape[1], ptr(mean), ptr(enrol.contiguous()), ptr(test.contiguous()), n,
                                     ptr(out), stream_ptr()))
    return out


def plda_trials(xvecs: torch.Tensor, mean: torch.Tensor, w_phi: torch.Tensor, b_phi: torch.Tensor, w_psi: torch.Tensor, b_psi: torch.Tensor,
                cst: float, scale: float, enrol: torch.Tensor, test: torch.Tensor) -> torch.Tensor:
    """PLDA log-likelihood-ratio of every (enrol, test) index pair into xvecs (N, D) float32; float32 (n_trials).
    w_phi / w_psi: [W_hi | W_hi | W_lo] of W = Phi' / Psi' packed with pack_weight(…, 1, 3 D, float32) for the split-TF32
    GEMMs (include/xvec_b200.h); b_phi / b_psi: -mean Phi / -mean Psi (pad32)."""
    _require_cuda(xvecs, mean, w_phi, b_phi, w_psi, b_psi, enrol, test)
    lib = _lib.load()
    if xvecs.dtype != torch.float32 or enrol.dtype != torch.int32 or test.dtype != torch.int32:
        raise ValueError("xvecs must be float32, trial indices int32")
    ld = _rowmajor_2d(xvecs, "xvecs")
    n, d = xvecs.shape
    if test.numel() != enrol.numel():
        raise ValueError("enrol and test must have the same length")
    x = xvecs
    x3 = torch.empty((n, 3 * d), dtype=torch.float32, device=x.device)  # [hi | lo | hi]: split-TF32 operand of both GEMMs
    with _lib.on_device(x.device):
        check(lib.xvec_split_tf32(ptr(x), ld, n, d, ptr(x3), x3.stride(0), stream_ptr()))
    y = tdnn_layer_flat(x3, w_phi, d, [0], b_phi, None, None, relu=False, out_dtype=torch.float32, cin=3 * d)  # (x - mean) Phi
    p = tdnn_layer_flat(x3, w_psi, d, [0], b_psi, None, None, relu=False, out_dtype=torch.float32, cin=3 * d)  # (x - mean) Psi
    q = torch.empty(n, dtype=torch.float32, device=x.device)
    out = torch.empty(enrol.numel(), dtype=torch.float32, device=x.device)
    with _lib.on_device(x.device):
        check(lib.xvec_plda_rowterm(ptr(x), x.stride(0), d, ptr(mean), ptr(y), y.stride(0), n, ptr(q), stream_ptr()))
        check(lib.xvec_plda_trials(ptr(x), x.stride(0), d, ptr(mean), ptr(p), p.stride(0), ptr(q), ptr(enrol.contiguous()),
                                   ptr(test.contiguous()), enrol.numel(), float(cst), float(scale), ptr(out), stream_ptr()))
    return out


def linear_small(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor | None = None, relu: bool = False,
                 out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """y = act(x W' + bias) with the small-footprint mma.sync kernel (xvec_linear_small): x (rows, k) and weight (n, k)
    row-major (the nn.Linear layout), both bfloat16, both float16 or both float32 (TF32 math), float32 accumulation; float32,
    bfloat16 or float16 result."""
    _require_cuda(x, weight, bias)
    lib = _lib.load()
    if x.dtype != weight.dtype:
        raise ValueError("x and weight must share a dtype (float32, bfloat16 or float16)")
    x_ld, w_ld = _rowmajor_2d(x, "x"), _rowmajor_2d(weight, "weight")
    if x.shape[1] != weight.shape[1]:
        raise ValueError("x and weight disagree on k")
    out = torch.empty((x.shape[0], weight.shape[0]), dtype=out_dtype, device=x.device)
    b = None if bias is None else bias.detach().float().contiguous()
    with _lib.on_device(x.device):
        check(lib.xvec_linear_small(ptr(x), dtype_code(x.dtype), x.shape[0], x.shape[1], x_ld, ptr(weight), weight.shape[0], w_ld, ptr(b),
                                    int(bool(relu)), ptr(out), dtype_code(out_dtype), out.stride(0), stream_ptr()))
    return out
