"""Host-facing extraction: pinned host MFCC buffers in, host x-vectors out — the call a user of the reference's
test_step/test_epoch_end (main.py:135-146) makes, minus the per-utterance .cpu() round trips.

Each of the `n_slots` slots owns a CUDA stream, a device staging buffer, model scratch and a pinned result buffer, so
the host->device copy of batch i+1 overlaps the kernels of batch i and the device->host copy of batch i-1.  The persistent
TDNN-stack kernel of the next batch takes over the SMs as the current one drains, so the small finalize / segment kernels of a
batch finish about one step late: six slots (measured on B200: 3 / 4 / 6 slots = 623 k / 678 k / 700 k utt/s) keep the GPU fed
while the host is blocked reading a result.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .layout import check_windows, window_layout



@dataclass
class _Slot:
    stream: torch.cuda.Stream
    done: torch.cuda.Event
    x_dev: torch.Tensor | None = None
    out_host: torch.Tensor | None = None
    n_out: int = 0
    busy: bool = False


class HostExtractor:
    def __init__(self, model, n_slots: int = 6):
        self.model = model
        self.device = model._device()
        if self.device.type != "cuda":
            raise ValueError("xvec_b200 has no CPU path: move the model to a CUDA device first")
        with torch.cuda.device(self.device):
            self.slots = [_Slot(torch.cuda.Stream(), torch.cuda.Event()) for _ in range(n_slots)]
        self._next = 0
        self._flat = None
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    @property
    def _dim(self) -> int:
        """Width of an x-vector: the output of segment_layer7 (x_vec_extract_layer 7) or segment_layer6."""
        return (self.model.segment_layer7 if self.model.x_vec_extract_layer == 7 else self.model.segment_layer6).out_features

    def reserve(self, max_rows: int, max_utts: int, channels: int, max_slots: int | None = None) -> None:
        """Size the staging buffer, the pinned result buffer and the model scratch of every slot for batches of up to
        max_rows frames / max_utts utterances (or windows) / max_slots pooling partial slots (default: the most max_utts
        utterances in max_rows frames can have); allocation synchronises the device, so do it before the pipeline runs."""
        dim = self._dim
        # partial slots: an utterance of n pooled frames touches <= n/128 + 2 groups
        pooled_slots = max_rows // 128 + 2 * max_utts + 2 if max_slots is None else max_slots
        with torch.cuda.device(self.device):
            for i, sl in enumerate(self.slots):
                if sl.x_dev is None or sl.x_dev.shape[0] < max_rows or sl.x_dev.shape[1] != channels:
                    sl.x_dev = torch.empty((max_rows, channels), dtype=torch.float32, device=self.device)
                if sl.out_host is None or sl.out_host.shape[0] < max_utts or sl.out_host.shape[1] != dim:
                    sl.out_host = torch.empty((max_utts, dim), dtype=torch.float32, pin_memory=True)
                self.model._scratch_for(i).ensure(max_rows, pooled_slots, max_utts)

    def submit(self, x_host: torch.Tensor, lengths, out_dev: torch.Tensor | None = None, windows=None) -> int:
        """Enqueue one batch: x_host is a float32 host tensor (rows, C) or (B, T, C), ideally pinned.  Returns a ticket.
        out_dev: float32 (len(lengths), dim) CUDA tensor that receives the x-vectors ON THE DEVICE instead of the slot's pinned
        host buffer (no device->host copy; result(ticket) then only waits) — for consumers that stay on the GPU (the sharded
        gather over NCCL, trial scoring).  windows: (W, 3) (recording, first_frame, n_frames) of the batch's recordings: one
        x-vector per window (XVectorModel.extract_x_vec_windows) instead of one per recording; out_dev is then (W, dim)."""
        if x_host.is_cuda:
            raise ValueError("HostExtractor.submit takes host tensors; call model.extract_x_vec for device tensors")
        if x_host.dim() == 3:
            x_host = x_host.reshape(-1, x_host.shape[-1])
        if x_host.dtype != torch.float32:
            x_host = x_host.float()  # main.py:137 samples.float()
        i = self._next
        self._next = (self._next + 1) % len(self.slots)
        sl = self.slots[i]
        if sl.busy:
            sl.done.synchronize()
        rows, c = x_host.shape
        n_utts = len(lengths) if windows is None else len(windows)
        dim = self._dim
        with _lib.on_device(self.device), torch.cuda.stream(sl.stream):
            if sl.x_dev is None or sl.x_dev.shape[0] < rows or sl.x_dev.shape[1] != c:
                sl.x_dev = torch.empty((rows, c), dtype=torch.float32, device=self.device)
            if out_dev is None and (sl.out_host is None or sl.out_host.shape[0] < n_utts or sl.out_host.shape[1] != dim):
                sl.out_host = torch.empty((n_utts, dim), dtype=torch.float32, pin_memory=True)
            xd = sl.x_dev[:rows]
            xd.copy_(x_host, non_blocking=True)
            if windows is None:
                xv = self.model.extract_x_vec_flat(xd, lengths, slot=i, out=out_dev)
            else:
                xv = self.model.extract_x_vec_windows(xd, lengths, windows, slot=i, out=out_dev)
            if out_dev is None:
                sl.out_host[:n_utts].copy_(xv, non_blocking=True)
                self.d2h_bytes += n_utts * dim * 4
            sl.done.record(sl.stream)
        sl.n_out = n_utts if out_dev is None else 0
        sl.busy = True
        self.h2d_bytes += rows * c * 4
        return i

    def result(self, ticket: int) -> torch.Tensor:
        """Host float32 (n_utts, dim) view of the slot's pinned result buffer (valid until the slot is reused); None for a batch
        submitted with out_dev (its x-vectors are in that device tensor once this returns)."""
        sl = self.slots[ticket]
        sl.done.synchronize()
        sl.busy = False
        return None if sl.out_host is None or sl.n_out == 0 else sl.out_host[: sl.n_out]

    def extract_flat(self, flat_host: torch.Tensor, lengths, max_frames: int = 1 << 17, max_utts: int = 1 << 30,
                     to_host: bool = True, batch_sizes=None, out_dev: torch.Tensor | None = None):
        """Extract a whole (ragged) set given as ONE flat host tensor (sum(lengths), C) float32 (pinned for full speed) plus
        the utterance lengths.  Batches are runs of CONSECUTIVE utterances of at most max_frames frames: the flat frame
        layout has no padding, so there is nothing to gain from length bucketing and no per-batch gather is needed.
        Returns float64 numpy (N, dim) in the original order, the dtype test_epoch_end stores (main.py:145) — or, with
        to_host=False, a float32 CUDA tensor (N, dim) that every batch wrote its rows into on the device (no device->host copy;
        all batches are complete when the call returns).  batch_sizes: explicit utterance counts of the consecutive batches
        (sharding.shard_batches: batch boundaries that do not depend on the number of GPUs) instead of the greedy cut;
        out_dev: with to_host=False, the (N, dim) float32 CUDA tensor to fill (e.g. the send buffer of the NCCL gather)."""
        lengths = np.asarray(lengths, dtype=np.int64)
        n = len(lengths)
        if to_host:
            out_dev = None
        elif out_dev is not None and (out_dev.shape != (n, self._dim) or out_dev.dtype != torch.float32 or out_dev.device != self.device):
            raise ValueError(f"out_dev must be a float32 ({n}, {self._dim}) tensor on {self.device}")
        if batch_sizes is not None:
            if int(np.sum(batch_sizes)) != n or min(int(b) for b in batch_sizes) < 1:
                raise ValueError("batch_sizes must be positive and sum to the number of utterances")
            cuts = np.concatenate(([0], np.cumsum(batch_sizes))).tolist()
            runs = list(zip(cuts[:-1], cuts[1:]))
        else:
            runs = _runs(lengths, max_frames, max_utts)
        # an utterance of n pooled frames touches <= n/128 + 2 partial slots
        batches = [(lo, hi, None, lo, hi, int(lengths[lo:hi].sum()) // 128 + 2 * (hi - lo) + 2) for lo, hi in runs]
        return self._extract(flat_host, lengths, batches, n, to_host, out_dev)

    def extract_windows(self, flat_host: torch.Tensor, lengths, windows, max_frames: int = 1 << 17, to_host: bool = True):
        """x-vectors of windows (recording, first_frame, n_frames) of recordings given as ONE flat host tensor (sum(lengths), C)
        float32 (pinned for full speed): one pass of the frame-level stack over each recording (XVectorModel.extract_x_vec_windows).
        Batches are runs of consecutive WHOLE recordings of at most max_frames frames; a longer recording is a batch of its own.
        Returns float64 numpy (W, dim) in the order of `windows` — or, with to_host=False, a float32 CUDA tensor (W, dim)."""
        lengths, windows = check_windows(lengths, windows, self.model.lost_frames)
        order = np.argsort(windows[:, 0], kind="stable")  # the windows of a batch are then one run of `order`
        sorted_w = windows[order]
        batches = []
        for lo, hi in _runs(lengths, max_frames):
            w0, w1 = (int(i) for i in np.searchsorted(sorted_w[:, 0], [lo, hi], side="left"))
            if w1 > w0:  # recordings without a window are not read at all
                wins = sorted_w[w0:w1] - np.asarray([lo, 0, 0])
                batches.append((lo, hi, wins, w0, w1, window_layout(lengths[lo:hi], wins, self.model.lost_frames).n_slots))
        return self._extract(flat_host, lengths, batches, len(windows), to_host, None, order)

    def _extract(self, flat_host, lengths, batches, n_out, to_host, out_dev, order=None):
        """Run `batches` (first and one-past-last recording, windows relative to the batch or None, first and one-past-last output
        row, partial slots) through the slots and gather the (n_out, dim) result: float64 numpy, or with to_host=False a float32
        CUDA tensor (out_dev when given).  order: the output row of each batch output row (windows, batched by recording), None
        for the identity."""
        if flat_host.dim() != 2 or flat_host.shape[0] != int(lengths.sum()):
            raise ValueError("flat_host must be (sum(lengths), C)")
        ends = np.concatenate(([0], np.cumsum(lengths))).tolist()
        # size every slot's buffers once for the largest batch: growing a slot's scratch in the middle of the run costs a
        # cudaFree + cudaMalloc (device-wide synchronisation) per growth
        self.reserve(max(ends[hi] - ends[lo] for lo, hi, *_ in batches), max(o1 - o0 for _, _, _, o0, o1, _ in batches),
                     flat_host.shape[1], max_slots=max(b[5] for b in batches))
        out = np.empty((n_out, self._dim), dtype=np.float64) if to_host else None
        if not to_host and out_dev is None:
            out_dev = torch.empty((n_out, self._dim), dtype=torch.float32, device=self.device)
        pending = []

        def drain(k):
            while len(pending) > k:
                ticket, o0, o1 = pending.pop(0)
                r = self.result(ticket)
                if to_host:
                    out[slice(o0, o1) if order is None else order[o0:o1]] = r.numpy()

        for lo, hi, wins, o0, o1, _ in batches:
            drain(len(self.slots) - 1)
            dst = None if to_host else out_dev[o0:o1]
            pending.append((self.submit(flat_host[ends[lo]:ends[hi]], lengths[lo:hi], dst, windows=wins), o0, o1))
        drain(0)
        if to_host:
            return out
        if order is None:
            return out_dev
        res = torch.empty_like(out_dev)
        res[torch.from_numpy(order).to(self.device)] = out_dev
        return res

    def extract_all(self, utts, max_frames: int = 1 << 17, max_utts: int = 1 << 30) -> np.ndarray:
        """Extract a list of host (T_i, C) float32 tensors: concatenated once into a pinned flat buffer, then extract_flat."""
        rows = sum(int(u.shape[0]) for u in utts)
        if self._flat is None or self._flat.shape[0] < rows or self._flat.shape[1] != utts[0].shape[1]:
            self._flat = torch.empty((rows, utts[0].shape[1]), dtype=torch.float32, pin_memory=True)
        torch.cat([u.float() if u.dtype != torch.float32 else u for u in utts], out=self._flat[:rows])
        return self.extract_flat(self._flat[:rows], [int(u.shape[0]) for u in utts], max_frames, max_utts)


def _runs(lengths, max_frames: int, max_utts: int = 1 << 30):
    """Batches of consecutive whole recordings (or utterances): [(first, one past last)], each of at most max_frames frames (a
    longer recording alone) and max_utts recordings."""
    ends = np.cumsum(lengths)
    runs, lo, n = [], 0, len(lengths)
    while lo < n:
        row0 = int(ends[lo - 1]) if lo else 0
        hi = max(lo + 1, min(int(np.searchsorted(ends, row0 + max_frames, side="right")), lo + max_utts, n))
        runs.append((lo, hi))
        lo = hi
    return runs
