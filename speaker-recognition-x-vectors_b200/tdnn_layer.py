"""TdnnLayer — same module surface as the reference's tdnn_layer.TdnnLayer (tdnn_layer.py:5-41), computed by
the sm_100a tcgen05 kernel in csrc/tdnn_gemm.cu.  Eval-mode only (BatchNorm running statistics, Dropout off):
this package accelerates extraction, not training.
"""
from __future__ import annotations

from operator import attrgetter

import torch
import torch.nn as nn

from . import ops

BN_EPS_DEFAULT = 1e-5


def tap_offsets(context):
    """Row offsets c_j - c_0 of a context (tdnn_layer.py:43-60).  Like the reference, only symmetric contexts are
    meaningful: its slicing makes torch.cat fail otherwise, which is reported here as ValueError."""
    c = [int(v) for v in context]
    if not c:
        raise ValueError("empty context")
    if any(b <= a for a, b in zip(c, c[1:])):
        raise ValueError(f"context {c} must be strictly increasing")
    if len(c) > 1 and c[-1] != -c[0]:
        raise ValueError(f"context {c} is not symmetric (c[-1] != -c[0]); the reference cannot concatenate its views")
    return [v - c[0] for v in c]


class TdnnLayer(nn.Module):
    def __init__(self, input_size=24, output_size=512, context=[0], batch_norm=True, dropout_p=0.0):
        super().__init__()
        self.input_size = input_size
        self.output_size = output_size
        self.context = context
        self.batch_norm = batch_norm
        self.dropout_p = dropout_p

        self.linear = nn.Linear(input_size * len(context), output_size)
        self.relu = nn.ReLU()
        if self.batch_norm:
            self.norm = nn.BatchNorm1d(output_size)
        if self.dropout_p:
            self.drop = nn.Dropout(p=self.dropout_p)
        self._prep = OperandCache()

    # ------------------------------------------------------------------ parameter preparation (cached)
    def prepared(self, dtype: torch.dtype, fold_bn: bool = True):
        """(w_packed, bias, bn_scale, bn_shift) on the parameters' device; re-packed when parameters change."""
        def build():
            w, bias = pack_checked("TdnnLayer", self.linear.weight, self.linear.bias, len(tap_offsets(self.context)), self.input_size,
                                   dtype)
            affine = self.bn_affine64()
            return (w, bias) + ((None, None) if affine is None else (ops.pad32(affine[0]), ops.pad32(affine[1])))

        return self._prep.get(dtype, param_fingerprint(self), build)

    def bn_affine64(self):
        """(scale, shift) of this layer's eval-mode BatchNorm in float64, or None."""
        if not self.batch_norm:
            return None
        n = self.norm
        gamma = n.weight.detach().double() if n.weight is not None else torch.ones_like(n.running_var, dtype=torch.float64)
        beta = n.bias.detach().double() if n.bias is not None else torch.zeros_like(n.running_var, dtype=torch.float64)
        s = gamma / torch.sqrt(n.running_var.detach().double() + n.eps)
        return s, beta - n.running_mean.detach().double() * s

    def _check_eval(self):
        if self.training and (self.batch_norm or self.dropout_p):
            raise RuntimeError("xvec_b200.TdnnLayer implements eval-mode semantics only (BatchNorm running statistics, "
                               "Dropout off); call .eval() first")

    # ------------------------------------------------------------------ flat (rows, Cin) -> (rows, N)
    def forward_flat(self, x2d: torch.Tensor, out: torch.Tensor | None = None, out_dtype: torch.dtype | None = None):
        self._check_eval()
        w, bias, scale, shift = self.prepared(x2d.dtype)
        return ops.tdnn_layer_flat(x2d, w, self.output_size, tap_offsets(self.context), bias, scale, shift, relu=True, out=out,
                                   out_dtype=out_dtype, cin=self.input_size)

    # ------------------------------------------------------------------ reference surface
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: (B, T, input_size) CUDA float32 (TF32 tensor-core math), bfloat16 or float16 -> (B, T - (c[-1]-c[0]), output_size)."""
        if x.dim() != 3 or x.shape[2] != self.input_size:
            raise ValueError(f"expected (B, T, {self.input_size}), got {tuple(x.shape)}")
        if not x.is_cuda:
            raise ValueError("xvec_b200 has no CPU path: move the input (and the module) to a CUDA device")
        offs = tap_offsets(self.context)
        B, T, C = x.shape
        t_out = T - offs[-1]
        if t_out <= 0:
            raise ValueError(f"input of {T} frames is shorter than the context span {offs[-1]}+1")
        if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            x = x.float()
        flat = _aligned_rows(x.reshape(B * T, C))
        y = self.forward_flat(flat)
        return y.view(B, T, self.output_size)[:, :t_out, :]


FP16_MAX = 65504.0


def check_fp16_range(what: str, weight: torch.Tensor, bias: torch.Tensor | None = None) -> None:
    """float16 holds magnitudes below 65504: a weight or bias at or beyond that would be stored as inf.  Raise instead of
    computing with it (float16 has no range scaling here; the "tf32" precision has the float32 range)."""
    for name, t in (("weight", weight), ("bias", bias)):
        if t is not None and t.numel() and float(t.detach().abs().max()) >= FP16_MAX:
            raise ValueError(f"{what}: a {name} of magnitude {float(t.detach().abs().max()):.6g} does not fit float16 (max 65504); "
                             "use precision \"tf32\"")


def pack_checked(what: str, weight: torch.Tensor, bias: torch.Tensor | None, taps: int, cin: int, dtype: torch.dtype):
    """(packed weight, padded float32 bias) of one layer; float16 operands are range-checked first (check_fp16_range)."""
    if dtype == torch.float16:
        check_fp16_range(what, weight, bias)
    return ops.pack_weight(weight, taps, cin, dtype), ops.pad32(bias)


_version = attrgetter("_version")


def param_fingerprint(*modules):
    """(key, tensors) of every parameter and buffer of `modules` and their sub-modules.  The key holds the identity and in-place
    version of each tensor: .to()/.cuda() and replacing a sub-module create new tensors, load_state_dict and optimiser steps bump
    the version.  Ids are only unique among live tensors, so whoever keeps the key keeps the tensors too.  Reads the module dicts
    directly: this runs once per batch, and nn.Module.__getattr__ costs more than the comparison."""
    tensors, todo = [], list(modules)
    for m in todo:  # sub-modules are appended while the list is walked
        if m is None:
            continue
        if params := m._parameters:
            tensors += params.values()
        if buffers := m._buffers:
            tensors += buffers.values()
        if children := m._modules:
            todo += children.values()
    tensors = [t for t in tensors if t is not None]
    return tuple(map(id, tensors)) + tuple(map(_version, tensors)), tensors


class OperandCache:
    """Kernel operands prepared from module parameters (packed weights, folded BatchNorm), each rebuilt when the parameters it
    was built from change.  Preparation is enqueued on the current stream, and its results are then read by kernels on other
    streams (one per pipeline slot) with no event in between; so a build blocks the host until the current stream is done, and
    stale operands are dropped only once every stream of their device is idle, as kernels in flight may still read them.  Both
    happen once per parameter change, never per batch."""

    def __init__(self):
        self._entries = {}

    def get(self, key, fingerprint, build):
        """The value cached under `key` if it was built at `fingerprint` (param_fingerprint), else build() stored in its place."""
        fp, tensors = fingerprint
        old = self._entries.get(key)
        if old is not None:
            if old[0] == fp:
                return old[2]
            for dev in {t.device for t in old[1] if t.is_cuda}:  # where the parameters the old operands came from live
                torch.cuda.synchronize(dev)
        value = build()
        for dev in {t.device for t in tensors if t.is_cuda}:
            torch.cuda.current_stream(dev).synchronize()
        self._entries[key] = (fp, tensors, value)
        return value


def _aligned_rows(x2d: torch.Tensor) -> torch.Tensor:
    """TMA needs a 16-byte aligned base and row pitch; copy into a padded buffer only when the input is not."""
    es = x2d.element_size()
    ok = x2d.stride(1) == 1 and (x2d.stride(0) * es) % 16 == 0 and x2d.data_ptr() % 16 == 0
    if ok:
        return x2d
    per16 = 16 // es
    ld = (x2d.shape[1] + per16 - 1) // per16 * per16
    buf = torch.zeros((x2d.shape[0], ld), dtype=x2d.dtype, device=x2d.device)
    buf[:, : x2d.shape[1]].copy_(x2d)
    return buf[:, : x2d.shape[1]]


def get_time_context(x, c=[0]):
    """Kept for surface parity with tdnn_layer.get_time_context (tdnn_layer.py:43-60): returns the k shifted views.
    The kernels never call this — they read the shifted windows with TMA instead of materialising them."""
    offs = tap_offsets(c)
    t_out = x.shape[1] - offs[-1]
    return [x[:, o:o + t_out, :] for o in offs]
