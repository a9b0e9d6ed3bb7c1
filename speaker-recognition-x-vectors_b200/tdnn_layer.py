"""TdnnLayer — same module surface as the reference's tdnn_layer.TdnnLayer (tdnn_layer.py:5-41), computed by
the sm_100a tcgen05 kernel in csrc/tdnn_gemm.cu.  Eval-mode only (BatchNorm running statistics, Dropout off):
this package accelerates extraction, not training.
"""
from __future__ import annotations

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
        self._prep = {}

    # ------------------------------------------------------------------ parameter preparation (cached)
    def _fingerprint(self):
        """(identity, in-place version) per parameter / buffer: .to()/.cuda() create new tensors (new identity), load_state_dict
        and optimiser steps bump the version, replacing a sub-module changes the dicts.  Read straight from the modules'
        parameter dicts — this runs once per batch and layer, and nn.Module.__getattr__ costs more than the comparison."""
        mods = self._modules
        lin = mods["linear"]
        out = [id(lin)]
        for t in lin._parameters.values():
            if t is not None:
                out.append(id(t))
                out.append(t._version)
        if self.batch_norm:
            norm = mods["norm"]
            out.append(id(norm))
            for d in (norm._parameters, norm._buffers):
                for t in d.values():
                    if t is not None:
                        out.append(id(t))
                        out.append(t._version)
        return tuple(out)

    def prepared(self, dtype: torch.dtype, fold_bn: bool = True):
        """(w_packed, bias, bn_scale, bn_shift) on the parameters' device; re-packed when parameters change."""
        fp = self._fingerprint()
        hit = self._prep.get(dtype)
        if hit is not None and hit[0] == fp:
            return hit[1]
        if hit is not None and hit[1][0].is_cuda:  # operands about to be dropped may still be read by kernels in flight
            with torch.cuda.device(hit[1][0].device):
                torch.cuda.synchronize()
        offs = tap_offsets(self.context)
        if dtype == torch.float16:
            check_fp16_range("TdnnLayer", self.linear.weight.detach(), self.linear.bias)
        w = ops.pack_weight(self.linear.weight, len(offs), self.input_size, dtype)
        bias = ops.pad32(self.linear.bias)
        scale = shift = None
        if self.batch_norm:
            n = self.norm
            gamma = n.weight.detach().double() if n.weight is not None else torch.ones_like(n.running_var, dtype=torch.float64)
            beta = n.bias.detach().double() if n.bias is not None else torch.zeros_like(n.running_var, dtype=torch.float64)
            s = gamma / torch.sqrt(n.running_var.detach().double() + n.eps)
            scale = ops.pad32(s.float())
            shift = ops.pad32((beta - n.running_mean.detach().double() * s).float())
        out = (w, bias, scale, shift)
        self._prep[dtype] = (fp, out)
        if w.is_cuda:  # the cached operands may be used from any stream from here on (see xvector._prep_fence)
            with torch.cuda.device(w.device):
                torch.cuda.current_stream().synchronize()
        return out

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
