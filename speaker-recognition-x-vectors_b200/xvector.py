"""XVectorModel — the extraction surface of the reference's main.XVectorModel (main.py:23-94) on B200.

Same constructor keywords, same sub-module names and state_dict keys (so a reference checkpoint's
``ckpt['state_dict']`` loads with load_state_dict), same ``forward`` / ``extract_x_vec`` / ``stat_pool`` /
``test_step`` semantics in eval mode.  The Lightning trainer, dataset and optimiser are out of scope.

Pipeline of extract_x_vec on one flat frame matrix (rows = sum of utterance lengths):
    TDNN1..5  xvec_tdnn_stack        ONE persistent launch: tcgen05 GEMM tiles of all five layers drawn from a work queue,
                                     TMA-shifted frame windows, bias+ReLU epilogue (BN folded forward); TDNN5's epilogue =
                                     per-utterance column sums (its activation is never stored)
    pooling   xvec_pool_finalize     fixed-order fp64 reduction -> [mean || std], BN5 folded through
    segment6/7  xvec_tdnn_layer (taps = 1)
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops
from .layout import utterance_layout, window_layout
from .tdnn_layer import OperandCache, TdnnLayer, _aligned_rows, pack_checked, param_fingerprint, tap_offsets

# "tf32": float32 storage, tensor-core math in TF32 (10-bit mantissa operands, fp32 accumulate; measured 1e-4 of the row norm
# against the reference's fp32, bound 1e-3).  "fp32" is kept as an alias for callers that name the reference's dtype
# (main.py:137 samples.float()); it is the SAME TF32 arithmetic, not IEEE fp32 products.  "bf16": bfloat16 activations/weights.
# "fp16": float16 activations/weights on the same kind::f16 pipe and bytes as bf16, with the 10-bit mantissa of TF32 operands;
# its range is |x| < 65504: a folded weight or bias outside it is refused when the model is prepared (ValueError), an activation
# outside it becomes inf and reaches the x-vector as a non-finite value (DESIGN.md section 4).
PRECISIONS = {"tf32": torch.float32, "fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


class _Layout:
    """Device copy of a batch's pooling layout (layout.utterance_layout, or layout.window_layout with windows; cached by lengths
    and windows for repeated shapes).  The stack reads the rows [row0, row0 + rows) of the frame matrix, its pooling epilogue sums
    the pooled runs (`starts`, `n_pool`: the utterances, or the windows' pieces) into partial slots, and the finalize writes output
    row u (an utterance, or a window) from the slots [slot_lo[u], slot_hi[u])."""

    def __init__(self, wl, frames, device, staging):
        self.row0, self.rows, self.n_slots, self.n_utts = wl.row0, wl.rows, wl.n_slots, int(wl.starts.shape[0])
        self.frames = frames  # rows of the whole frame matrix
        self.n_out = int(wl.slot_lo.shape[0])
        (self.starts, self.n_pool, self.utt_slot_start, self.slot_lo, self.slot_hi, self.out_n_pool) = _upload(
            (wl.starts, wl.n_pool, wl.slot_start, wl.slot_lo, wl.slot_hi, wl.win_n_pool), device, staging)
        self.row_utt = torch.empty(self.rows, dtype=torch.int32, device=device)
        self.blk_slot_base = torch.empty(((self.rows + 255) // 256) * (256 // _lib.POOL_BLOCK), dtype=torch.int32, device=device)
        ops.build_layout_device(self.starts, self.n_pool, self.utt_slot_start, self.rows, self.row_utt, self.blk_slot_base)


def _upload(arrays, device, staging):
    """Device copies of 1-D int32 host arrays from ONE pinned upload.  An array that is a view of an earlier one (utterance_layout's
    slot_lo / slot_hi are slot_start[:-1] / slot_start[1:], its win_n_pool is n_pool) becomes the same view of that array's device
    copy and adds no bytes."""
    host = staging.get(sum(int(a.shape[0]) for a in arrays))
    addr = lambda a: a.__array_interface__["data"][0]
    place, total = [], 0  # element offset of each array in the upload
    for i, a in enumerate(arrays):
        j = next((j for j in range(i) if a is arrays[j] or a.base is arrays[j]), None)
        if j is None:
            host[total:total + a.shape[0]] = torch.from_numpy(a)
            place.append(total)
            total += a.shape[0]
        else:
            place.append(place[j] + (addr(a) - addr(arrays[j])) // a.itemsize)
    dev = torch.empty(total, dtype=torch.int32, device=device)
    dev.copy_(host[:total], non_blocking=True)
    staging.mark()
    return [dev[o:o + a.shape[0]] for a, o in zip(arrays, place)]


class _PinnedStaging:
    """A small ring of reusable pinned int32 buffers for the per-batch layout uploads; an event per buffer guards reuse, so
    the host only ever waits for a copy issued 16 batches ago."""

    RING = 16

    def __init__(self):
        self.bufs = [None] * self.RING
        self.evs = [None] * self.RING
        self.i = -1

    def get(self, n):
        self.i = (self.i + 1) % self.RING
        if self.evs[self.i] is not None:
            self.evs[self.i].synchronize()
        if self.bufs[self.i] is None or self.bufs[self.i].numel() < n:
            self.bufs[self.i] = torch.empty(max(n, 8192), dtype=torch.int32, pin_memory=True)
        return self.bufs[self.i]

    def mark(self):
        if self.evs[self.i] is None:
            self.evs[self.i] = torch.cuda.Event()
        self.evs[self.i].record()


class _Scratch:
    """Activation ping-pong buffers, pooling partials and pooled statistics of one slot; grown on demand, shared by layouts."""

    def __init__(self, device, act_dtype, widths, pool_dim):
        self.device, self.act_dtype, self.pool_dim = device, act_dtype, pool_dim
        per16 = 16 // torch.empty((), dtype=act_dtype).element_size()
        self.ld = (max(widths) + per16 - 1) // per16 * per16
        self.rows_cap = self.slots_cap = self.utts_cap = 0
        self.act = self.part = self.pooled = self.pooled_lp = self.ctrl = None
        self.fc_tmp = self.ws = self.ws_for = None

    def ensure(self, rows, n_slots, n_utts):
        if rows > self.rows_cap:
            self.rows_cap = max(rows, int(self.rows_cap * 1.25))
            self.act = [torch.empty((self.rows_cap, self.ld), dtype=self.act_dtype, device=self.device) for _ in range(2)]
            # work-item counter + per-tile completion flags of xvec_tdnn_stack (zeroed by the call itself)
            need = _lib.load().xvec_stack_ctrl_bytes(self.rows_cap, _lib.MAX_STACK)
            self.ctrl = torch.empty(need + 128, dtype=torch.uint8, device=self.device)
            off = (-self.ctrl.data_ptr()) % 128
            self.ctrl = self.ctrl[off: off + need]
        if n_slots > self.slots_cap:
            self.slots_cap = max(n_slots, int(self.slots_cap * 1.25))
            self.part = torch.empty((self.slots_cap, 2, self.pool_dim), dtype=torch.float32, device=self.device)
        if n_utts > self.utts_cap:
            self.utts_cap = max(n_utts, int(self.utts_cap * 1.25))
            self.pooled = torch.empty((self.utts_cap, 2 * self.pool_dim), dtype=torch.float32, device=self.device)
            self.pooled_lp = (torch.empty((self.utts_cap, 2 * self.pool_dim), dtype=self.act_dtype, device=self.device)
                              if self.act_dtype != torch.float32 else None)
            self.fc_tmp = None

    def ensure_head(self, n_utts, fc_shapes, width):
        """Scratch of the segment layers: the hidden (n_utts, width) activation and the split-K workspace."""
        if self.fc_tmp is None or self.fc_tmp.shape[0] < n_utts or self.fc_tmp.shape[1] != width:
            self.fc_tmp = torch.empty((max(n_utts, self.utts_cap), width), dtype=self.act_dtype, device=self.device)
        self.splitk_ws(n_utts, fc_shapes)

    def splitk_ws(self, rows, fc_shapes):
        """The slot's one split-K workspace (None until a shape splits), grown to what any (cin, n) segment shape in fc_shapes
        needs at `rows` rows: it only ever grows, so it is sized for the largest need seen."""
        key = (rows, tuple(fc_shapes))
        if self.ws_for != key:
            lib = _lib.load()
            need = max(lib.xvec_splitk_workspace_bytes(rows, cin, 1, n, _lib.dtype_code(self.act_dtype)) for cin, n in fc_shapes)
            if need > 0 and (self.ws is None or self.ws.numel() < need):
                self.ws = torch.empty(need, dtype=torch.uint8, device=self.device)
            self.ws_for = key
        return self.ws


class XVectorModel(nn.Module):
    def __init__(self, input_size=24, hidden_size=512, num_classes=1211, x_vector_size=512, x_vec_extract_layer=6,
                 batch_size=512, learning_rate=0.001, batch_norm=True, dropout_p=0.0, augmentations_per_sample=2,
                 data_folder_path="data", precision="tf32"):
        super().__init__()
        self.time_context_layers = nn.Sequential(
            TdnnLayer(input_size=input_size, output_size=hidden_size, context=[-2, -1, 0, 1, 2], batch_norm=batch_norm, dropout_p=dropout_p),
            TdnnLayer(input_size=hidden_size, output_size=hidden_size, context=[-2, 0, 2], batch_norm=batch_norm, dropout_p=dropout_p),
            TdnnLayer(input_size=hidden_size, output_size=hidden_size, context=[-3, 0, 3], batch_norm=batch_norm, dropout_p=dropout_p),
            TdnnLayer(input_size=hidden_size, output_size=hidden_size, batch_norm=batch_norm, dropout_p=dropout_p),
            TdnnLayer(input_size=hidden_size, output_size=1500, batch_norm=batch_norm, dropout_p=dropout_p),
        )
        self.segment_layer6 = nn.Linear(3000, x_vector_size)
        self.segment_layer7 = nn.Linear(x_vector_size, x_vector_size)
        self.output = nn.Linear(x_vector_size, num_classes)

        self.x_vec_extract_layer = x_vec_extract_layer
        self.batch_size = batch_size
        self.learning_rate = learning_rate
        self.input_size = input_size
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
        self.precision = precision
        self._layouts: "OrderedDict[tuple, _Layout]" = OrderedDict()
        self._scratch = {}
        self._prep = OperandCache()

    # ------------------------------------------------------------------ helpers
    @property
    def act_dtype(self) -> torch.dtype:
        return PRECISIONS[self.precision]

    @property
    def lost_frames(self) -> int:
        return sum(tap_offsets(l.context)[-1] for l in self.time_context_layers)

    def _device(self):
        return self._modules["segment_layer6"]._parameters["weight"].device

    def _check_eval(self):
        if self.training:
            raise RuntimeError("xvec_b200.XVectorModel implements the eval-mode extraction path only; call .eval() first")

    def _layout_for(self, lengths, windows=None) -> _Layout:
        lengths = np.asarray(lengths, dtype=np.int64)
        dev = self._device()
        if windows is not None:
            windows = np.ascontiguousarray(windows)
        key = (lengths.tobytes(), None if windows is None else (windows.shape, windows.dtype.str, windows.tobytes()), dev.index,
               _lib.stream_ptr(dev.index))
        lay = self._layouts.get(key)
        if lay is None:
            st = self._scratch.setdefault(("pin", str(dev)), _PinnedStaging())  # one ring per device: its buffers are event-guarded
            wl = (utterance_layout(lengths, self.lost_frames) if windows is None
                  else window_layout(lengths, windows, self.lost_frames))
            lay = _Layout(wl, int(lengths.sum()), dev, st)
            self._layouts[key] = lay
            while len(self._layouts) > 128:
                self._layouts.popitem(last=False)
        else:
            self._layouts.move_to_end(key)
        return lay

    def _scratch_for(self, slot: int) -> _Scratch:
        dev = self._device()
        key = (dev.index, self.precision, slot)
        sc = self._scratch.get(key)
        if sc is None:
            layers = list(self.time_context_layers)
            sc = _Scratch(dev, self.act_dtype, [l.output_size for l in layers[:-1]], layers[-1].output_size)
            self._scratch[key] = sc
        return sc

    def _stack_kernel_ok(self) -> bool:
        """Limits of xvec_tdnn_stack (include/xvec_b200.h): stored layers are whole 256-channel tiles, chained widths."""
        layers = list(self.time_context_layers)
        return (2 <= len(layers) <= _lib.MAX_STACK
                and all(l.output_size % _lib.TILE_N == 0 for l in layers[:-1])
                and all(a.output_size == b.input_size for a, b in zip(layers[:-1], layers[1:]))
                and all(tap_offsets(l.context)[-1] <= _lib.STACK_MAX_TAP_OFFSET for l in layers))

    def _stack_params(self):
        """Packed operands of the five TDNN layers for the fused pipeline, with every layer's eval-mode BatchNorm folded
        FORWARD into the next layer (BN comes after ReLU, tdnn_layer.py:30-39, so it cannot fold into its own layer):
            W'_i = W_i . diag(s_{i-1} (x) 1_k),   b'_i = b_i + W_i . (h_{i-1} (x) 1_k)
        so each epilogue is just relu(acc + b'); the last layer's BN is folded through the statistics by
        xvec_pool_finalize (mean' = s.mean + h, std' = |s|.std).  Computed once in float64, cached until parameters change.
        Layer 1 reads the float32 MFCCs (TF32 math) in both precisions; the fused pipeline uses its window form (_pipeline)."""
        return self._prep.get(("stack", self.act_dtype), param_fingerprint(self._modules["time_context_layers"]), self._fold_stack)

    def _fold_stack(self):
        layers = list(self.time_context_layers)
        out, prev = [], None
        for i, layer in enumerate(layers):
            layer._check_eval()
            offs = tap_offsets(layer.context)
            W = layer.linear.weight.detach().double()
            b = (layer.linear.bias.detach().double() if layer.linear.bias is not None
                 else torch.zeros(layer.output_size, dtype=torch.float64, device=W.device))
            if prev is not None:
                s, h = prev
                b = b + W @ h.repeat(len(offs))
                W = W * s.repeat(len(offs))[None, :]
            what = f"time_context_layers[{i}] with the BatchNorm of layer {i - 1} folded in"
            out.append((*pack_checked(what, W, b, len(offs), layer.input_size, torch.float32 if i == 0 else self.act_dtype), offs))
            prev = layer.bn_affine64()
        last_bn = (None, None) if prev is None else (prev[0].float().contiguous(), prev[1].float().contiguous())
        return out, last_bn

    def _pipeline(self):
        """XvecLayerDesc arrays for xvec_extract_forward (one C call per batch), rebuilt when parameters change."""
        mods = self._modules
        use7 = self.x_vec_extract_layer == 7
        fp = param_fingerprint(mods["time_context_layers"], mods["segment_layer6"], mods["segment_layer7"] if use7 else None)
        return self._prep.get(("pipeline", self.act_dtype, use7), fp, lambda: self._build_pipeline(use7))

    def _build_pipeline(self, use7):
        layers = list(self.time_context_layers)
        names = ("segment_layer6", "segment_layer7") if use7 else ("segment_layer6",)
        fcs = [self._modules[n] for n in names]
        stack, (scale5, shift5) = self._stack_params()
        code = _lib.dtype_code
        tdnn = (_lib.LayerDesc * len(layers))()
        window = None
        for i, (layer, (w, bias, offs)) in enumerate(zip(layers, stack)):
            d = tdnn[i]
            cin, taps = layer.input_size, len(offs)
            if i == 0 and list(offs) == list(range(taps)) and taps > 1 and (cin * 4) % 16 == 0 and self._stack_kernel_ok():
                # Window form of TDNN1 (include/xvec_b200.h, xvec_tdnn_stack): consecutive taps over dense rows are one
                # contiguous run of taps*cin values, so the layer is a plain K = 120 GEMM over overlapping rows of the float32
                # frames (TF32 math): 4 K chunks per tile instead of 5, no unfold, no copy.  nn.Linear's weight is already in
                # window order.
                w = ops.pack_weight(layer.linear.weight.detach().float(), 1, taps * cin, torch.float32)
                window = {"w": w, "cin": taps * cin}
                cin, offs = taps * cin, [0]
            d.w_packed_dev, d.bias_dev = w.data_ptr(), (bias.data_ptr() if bias is not None else None)
            d.n, d.cin, d.taps, d.dtype = layer.output_size, cin, len(offs), code(w.dtype)
            for j, o in enumerate(offs):
                d.tap_offsets[j] = o
        fc = (_lib.LayerDesc * len(fcs))()
        keep = [stack, window]  # the descriptors hold raw pointers: these own what they point to
        for i, (name, lin) in enumerate(zip(names, fcs)):
            w, b = self._fc(name, self.act_dtype)
            keep.append((w, b))
            d = fc[i]
            d.w_packed_dev, d.bias_dev = w.data_ptr(), (b.data_ptr() if b is not None else None)
            d.n, d.cin, d.taps, d.dtype = lin.out_features, lin.in_features, 1, code(w.dtype)
            d.tap_offsets[0] = 0
            if lin.in_features % 8 == 0:
                # plain copy of the weight in the activation dtype for xvec_linear_small (a small-footprint kernel that runs next to
                # the next batch's resident stack kernel instead of waiting for free SMs)
                w32 = lin.weight.detach().float().contiguous()
                w_plain = w32.clone() if self.act_dtype == torch.float32 else ops.cast(w32, self.act_dtype)
                keep.append(w_plain)
                d.w_plain_dev = w_plain.data_ptr()
        return {"tdnn": tdnn, "n_tdnn": len(layers), "fc": fc, "n_fc": len(fcs), "keep": keep, "window": window,
                "scale5": scale5, "shift5": shift5, "out_dim": fcs[-1].out_features, "hidden": fcs[0].out_features,
                "fc_shapes": [(f.in_features, f.out_features) for f in fcs]}

    def _fc(self, name: str, dtype):
        """(packed weight, padded bias) of the segment layer `name` (an nn.Linear attribute) in `dtype`."""
        lin = self._modules[name]
        return self._prep.get((name, dtype), param_fingerprint(lin),
                              lambda: pack_checked(name, lin.weight, lin.bias, 1, lin.in_features, dtype))

    def _linear(self, name: str, x2d: torch.Tensor, relu: bool, out_dtype) -> torch.Tensor:
        """Segment layer `name` on x2d, split-K through slot 0's workspace (forward() runs in slot 0's scratch)."""
        lin = self._modules[name]
        w, b = self._fc(name, x2d.dtype)
        ws = self._scratch_for(0).splitk_ws(x2d.shape[0], ((lin.in_features, lin.out_features),))
        return ops.tdnn_layer_flat(x2d, w, lin.out_features, [0], b, None, None, relu=relu, out_dtype=out_dtype, cin=lin.in_features,
                                   workspace=ws)

    def _frames_for(self, flat_x: torch.Tensor, pipe) -> torch.Tensor:
        """The frame matrix as layer 1 reads it: 16-byte aligned rows, and DENSE rows (stride == input_size) when layer 1 is in
        window form — its taps*cin window is one contiguous run only then (include/xvec_b200.h, xvec_tdnn_stack).  A (rows, 24)
        view of a wider buffer (ops.mfcc(out=...) allows one) is copied once instead of silently mixing padding columns into the
        taps."""
        x = _aligned_rows(flat_x)
        if pipe["window"] is not None and x.stride(0) != self.input_size:
            x = _aligned_rows(x.contiguous())
        return x

    # ------------------------------------------------------------------ the hot path
    def _extract_forward(self, flat_x: torch.Tensor, lengths, slot: int, head: bool, out: torch.Tensor | None = None, windows=None):
        """ONE C-ABI call (xvec_extract_forward) that enqueues the path on the current
        stream: the TDNN stack (the persistent stack kernel, or one launch per layer for stacks it does not take) with the pooling
        partials, the pooling finalize into the slot's scratch and, when `head`, the segment layer(s) into `out` (allocated when
        None).  Returns (layout, scratch, out)."""
        self._check_eval()
        if not flat_x.is_cuda:
            raise ValueError("xvec_b200 has no CPU path: move the input (and the model) to a CUDA device")
        if flat_x.dim() != 2 or flat_x.shape[1] != self.input_size:
            raise ValueError(f"expected a flat (rows, {self.input_size}) frame matrix")
        lay = self._layout_for(lengths, windows)
        if lay.frames != flat_x.shape[0]:
            raise ValueError("sum(lengths) does not match the number of rows")
        pipe = self._pipeline()
        sc = self._scratch_for(slot)
        sc.ensure(lay.rows, lay.n_slots, lay.n_out)
        if flat_x.dtype != torch.float32:
            flat_x = flat_x.float()
        if lay.rows != lay.frames:  # windows: the stack reads the rows from the first window's first frame to the last one's end
            flat_x = flat_x[lay.row0: lay.row0 + lay.rows]
        x = self._frames_for(flat_x, pipe)  # layer 1 always reads the float32 frames (TF32 math): no cast pass over the input
        fc, n_fc, fc_tmp, ws = None, 0, None, None
        if head:
            sc.ensure_head(lay.n_out, pipe["fc_shapes"], pipe["hidden"])
            fc, n_fc, fc_tmp, ws = pipe["fc"], pipe["n_fc"], sc.fc_tmp, sc.ws
            if out is None:
                out = torch.empty((lay.n_out, pipe["out_dim"]), dtype=torch.float32, device=flat_x.device)
            elif (out.dtype != torch.float32 or out.device != flat_x.device or out.shape != (lay.n_out, pipe["out_dim"]) or out.stride(1) != 1):
                raise ValueError(f"out must be a float32 ({lay.n_out}, {pipe['out_dim']}) tensor on the input's device with unit column stride")
        p = _lib.ptr
        with _lib.on_device(flat_x.device):
            _lib.check(_lib.load().xvec_extract_forward(
                pipe["tdnn"], pipe["n_tdnn"], p(x), lay.rows, x.stride(0), p(sc.act[0]), p(sc.act[1]), sc.ld, p(lay.row_utt),
                p(lay.blk_slot_base), p(lay.slot_lo), p(lay.slot_hi), p(lay.out_n_pool), lay.n_out, p(sc.part), p(pipe["scale5"]), p(pipe["shift5"]),
                p(sc.pooled), p(sc.pooled_lp), fc, n_fc, p(fc_tmp), p(ws), 0 if ws is None else ws.numel(),
                p(out), 0 if out is None else out.stride(0), p(sc.ctrl), sc.ctrl.numel(), _lib.stream_ptr()))
        return lay, sc, out

    def pooled_stats_flat(self, flat_x: torch.Tensor, lengths, slot: int = 0) -> "tuple[torch.Tensor, torch.Tensor | None]":
        """TDNN stack + statistics pooling over a flat (rows, input_size) float32 frame matrix.
        Returns (pooled float32 (U, 3000), same in the activation dtype or None).  The returned tensors are scratch of
        the (lengths, slot) plan: they are overwritten by the next call with the same lengths and slot."""
        lay, sc, _ = self._extract_forward(flat_x, lengths, slot, head=False)
        return sc.pooled[: lay.n_out], None if sc.pooled_lp is None else sc.pooled_lp[: lay.n_out]

    def _head(self, pooled, pooled_lp, layer) -> torch.Tensor:
        a = pooled if pooled_lp is None else pooled_lp
        if layer == 7:  # main.py:88-90
            h6 = self._linear("segment_layer6", a, relu=True, out_dtype=a.dtype)
            return self._linear("segment_layer7", h6, relu=False, out_dtype=torch.float32)
        return self._linear("segment_layer6", a, relu=False, out_dtype=torch.float32)  # 6 and "anything else" (main.py:86-87,91-92)

    def extract_x_vec_flat(self, flat_x: torch.Tensor, lengths, slot: int = 0, out: torch.Tensor | None = None) -> torch.Tensor:
        """Ragged extraction: flat (sum(lengths), input_size) frames -> float32 (len(lengths), x_vector_size).
        `slot` selects an independent scratch set so that calls on different CUDA streams can overlap; `out` (float32 CUDA,
        (len(lengths), x_vector_size), unit column stride) receives the x-vectors in place, e.g. a row range of a whole set's matrix.
        The whole path is ONE C-ABI call (xvec_extract_forward) that enqueues its kernels on the current stream: the
        persistent TDNN-stack kernel (all five layers + pooling partials), the pooling finalize and the segment layer(s)."""
        return self._extract_forward(flat_x, lengths, slot, head=True, out=out)[2]

    def extract_x_vec_windows(self, flat_x: torch.Tensor, lengths, windows, slot: int = 0, out: torch.Tensor | None = None) -> torch.Tensor:
        """x-vectors of windows of recordings: flat (sum(lengths), input_size) frames of the recordings -> float32
        (W, x_vector_size).  windows: int (W, 3) array of (recording, first_frame, n_frames); row w is what extract_x_vec
        (main.py:81-94) gives for frames [first_frame, first_frame + n_frames) of that recording alone, layer 6 / 7 / other
        alike.  Windows may come in any order, repeat and nest; n_frames must exceed the model's lost_frames (a window of
        lost_frames + 1 frames pools one frame: NaN, like torch.std).  layout.sliding_windows makes the usual fixed-length,
        fixed-shift windows.
        The frame-level stack runs ONCE over the recordings (from the first window's first frame to the last window's last
        frame) instead of once per window; only the pooling finalize and the segment layer(s) are per window.  One C-ABI call
        (xvec_extract_forward) on the current stream; `slot` and `out` as for extract_x_vec_flat."""
        return self._extract_forward(flat_x, lengths, slot, head=True, out=out, windows=windows)[2]

    # ------------------------------------------------------------------ reference surface
    def extract_x_vec(self, x: torch.Tensor) -> torch.Tensor:
        """main.py:81-94.  x: (B, T, input_size) CUDA tensor -> (B, x_vector_size) float32, the pre-ReLU affine
        output of segment_layer6 (x_vec_extract_layer 6 / other) or segment_layer7 (7)."""
        if x.dim() != 3:
            raise ValueError(f"expected (B, T, {self.input_size}), got {tuple(x.shape)}")
        B, T, C = x.shape
        return self.extract_x_vec_flat(x.reshape(B * T, C), [T] * B)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """main.py:66-75 in eval mode: logits (B, num_classes)."""
        if x.dim() != 3:
            raise ValueError(f"expected (B, T, {self.input_size}), got {tuple(x.shape)}")
        B, T, C = x.shape
        pooled, pooled_lp = self.pooled_stats_flat(x.reshape(B * T, C), [T] * B)
        a = pooled if pooled_lp is None else pooled_lp
        h = self._linear("segment_layer6", a, relu=True, out_dtype=a.dtype)
        h = self._linear("segment_layer7", h, relu=True, out_dtype=a.dtype)
        return self._linear("output", h, relu=False, out_dtype=torch.float32)

    def stat_pool(self, x: torch.Tensor) -> torch.Tensor:
        """main.py:59-63: (B, T', P) -> (B, 2P) = [mean over time || unbiased std over time] (standalone HBM-bound kernel)."""
        if x.dim() != 3:
            raise ValueError("expected (B, T', P)")
        if not x.is_cuda:
            raise ValueError("xvec_b200 has no CPU path: move the input to a CUDA device")
        B, T, P = x.shape
        if x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        if x.stride(2) != 1 or x.stride(0) != T * x.stride(1) or P % 4 or x.stride(1) % 4 or x.data_ptr() % 16:
            x = x.contiguous()
            if P % 4:
                raise ValueError("stat_pool needs a channel count that is a multiple of 4")
        ld = x.stride(1)
        flat = torch.as_strided(x, (B * T, P), (ld, 1))
        return ops.stats_pool_ragged(flat, np.arange(B, dtype=np.int64) * T, np.full(B, T, dtype=np.int32))

    def test_step(self, batch, batch_index=0):
        """main.py:135-138 — the extraction step: (samples, labels, ids) -> [(x_vecs, labels, ids)]."""
        samples, labels, ids = batch
        x_vecs = self.extract_x_vec(samples.float())
        return [(x_vecs, labels, ids)]

    def load_reference_checkpoint(self, path: str, map_location="cpu", trust_pickle: bool = False):
        """Load the 'state_dict' of a Lightning checkpoint written by the reference (main.py:198,213).
        The file is read with torch.load(weights_only=True); a checkpoint that also pickles Lightning objects (callback state,
        hyper-parameter containers) needs the full unpickler, which executes code from the file — that is only done on
        explicit opt-in (trust_pickle=True, for files you wrote yourself).  Keys this model does not have (the reference's
        metric modules) are ignored; a key this model HAS and the checkpoint lacks is an error, not a silent random init."""
        try:
            ckpt = torch.load(path, map_location=map_location, weights_only=True)
        except Exception as e:
            if not trust_pickle:
                raise RuntimeError(f"{path} cannot be read with weights_only=True ({type(e).__name__}: {e}); pass trust_pickle=True "
                                   "only for a checkpoint from a trusted source") from e
            ckpt = torch.load(path, map_location=map_location, weights_only=False)
        sd = ckpt.get("state_dict", ckpt) if isinstance(ckpt, dict) else ckpt
        own = self.state_dict()
        missing = [k for k in own if k not in sd and not k.endswith("num_batches_tracked")]
        if missing:
            raise KeyError(f"checkpoint lacks {len(missing)} parameter(s) of the x-vector model, e.g. {missing[:3]}")
        return self.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=False)
