"""Flat frame-matrix layout of a (possibly ragged) batch of utterances and the pooling bookkeeping derived from it.

All utterances of a batch are concatenated into one (total_frames x channels) matrix: utterance u owns rows
[start[u], start[u] + length[u]).  Every TDNN layer keeps this row indexing (output row r reads input rows
r + offset_j), so after the five layers only the first length[u] - 14 rows of each utterance are meaningful —
exactly the frames the reference's stack produces for that utterance alone (tdnn_layer.py:43-60, main.py:38-44).
The remaining rows are don't-care and are masked out of statistics pooling.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import _lib

TOTAL_CONTEXT = 14  # frames lost over the five layers: 4 + 4 + 6 + 0 + 0 (main.py:39-43)


@dataclass
class FrameLayout:
    lengths: np.ndarray          # int64 (U) input frames per utterance
    starts: np.ndarray           # int64 (U) first row of each utterance
    n_pool: np.ndarray           # int32 (U) pooled frames per utterance
    rows: int                    # total rows
    row_utt: np.ndarray          # int32 (rows) utterance of a pooled row, -1 for don't-care rows
    blk_slot_base: np.ndarray    # int32 (ceil(rows/256)*2) first partial slot of each 128-row block
    utt_slot_start: np.ndarray   # int32 (U+1) partial slots of utterance u are [utt_slot_start[u], utt_slot_start[u+1])
    n_slots: int

    @property
    def n_utts(self) -> int:
        return int(self.lengths.shape[0])


def build_layout(lengths, lost_frames: int = TOTAL_CONTEXT) -> FrameLayout:
    lengths = np.asarray(lengths, dtype=np.int64).reshape(-1)
    if lengths.size == 0:
        raise ValueError("empty batch")
    if (lengths <= lost_frames).any():
        raise ValueError(f"every utterance needs more than {lost_frames} frames (the TDNN context); got min {int(lengths.min())}")
    starts = np.concatenate(([0], np.cumsum(lengths)[:-1]))
    rows = int(lengths.sum())
    if rows >= 2**31 - 256:
        raise ValueError("batch too large for 32-bit row indices; split it")
    n_pool = (lengths - lost_frames).astype(np.int64)
    utt_of_row = np.repeat(np.arange(lengths.size, dtype=np.int64), lengths)
    pos = np.arange(rows, dtype=np.int64) - starts[utt_of_row]
    row_utt = np.where(pos < n_pool[utt_of_row], utt_of_row, -1).astype(np.int32)
    blk = _lib.POOL_BLOCK
    b0 = starts // blk
    b1 = (starts + n_pool - 1) // blk
    cnt = b1 - b0 + 1
    utt_slot_start = np.concatenate(([0], np.cumsum(cnt))).astype(np.int64)
    n_slots = int(utt_slot_start[-1])
    # block index of every slot, in slot order (non-decreasing)
    slot_utt = np.repeat(np.arange(lengths.size, dtype=np.int64), cnt)
    slot_block = b0[slot_utt] + (np.arange(n_slots, dtype=np.int64) - utt_slot_start[slot_utt])
    n_blocks = ((rows + 255) // 256) * (256 // blk)  # the GEMM tiles 256 rows per CTA pair
    blk_slot_base = np.searchsorted(slot_block, np.arange(n_blocks, dtype=np.int64), side="left").astype(np.int32)
    return FrameLayout(lengths, starts, n_pool.astype(np.int32), rows, row_utt, blk_slot_base, utt_slot_start.astype(np.int32), n_slots)


def utterance_layout(lengths, lost_frames: int = TOTAL_CONTEXT) -> WindowLayout:
    """window_layout of the windows that are the whole utterances, in order, in O(#utterances) host work: the pieces are the
    utterances and output row u reduces the slots [slot_start[u], slot_start[u+1]), so slot_lo / slot_hi are views of slot_start
    and win_n_pool is n_pool.  The per-row / per-block arrays are expanded from it on the device (xvec_build_layout)."""
    lengths = np.asarray(lengths, dtype=np.int64).reshape(-1)
    if lengths.size == 0:
        raise ValueError("empty batch")
    if (lengths <= lost_frames).any():
        raise ValueError(f"every utterance needs more than {lost_frames} frames (the TDNN context); got min {int(lengths.min())}")
    starts = np.concatenate(([0], np.cumsum(lengths)[:-1]))
    rows = int(lengths.sum())
    if rows >= 2**31 - 256:
        raise ValueError("batch too large for 32-bit row indices; split it")
    n_pool = (lengths - lost_frames).astype(np.int32)
    slot_start = _slot_prefix(starts, n_pool).astype(np.int32)
    return WindowLayout(0, rows, starts.astype(np.int32), n_pool, slot_start, slot_start[:-1], slot_start[1:], n_pool,
                        int(slot_start[-1]))


def _slot_prefix(starts, n_pool):
    """Exclusive prefix sum of the partial slots of runs of pooled rows [starts[i], starts[i] + n_pool[i]) (sorted, disjoint):
    the fused pooling epilogue gives a run one slot per 128-row block it has a row in."""
    blk = _lib.POOL_BLOCK
    cnt = (starts + n_pool - 1) // blk - starts // blk + 1
    return np.concatenate(([0], np.cumsum(cnt))).astype(np.int64)


@dataclass
class WindowLayout:
    """Pooling bookkeeping of windows of recordings (window_layout), utterances being the windows that cover whole recordings
    (utterance_layout).  Rows are relative to `row0`, the first input row the frame-level stack has to read: rows before the
    first window's first frame are not passed to it at all."""
    row0: int                    # first row of the flat recordings matrix that the stack reads
    rows: int                    # rows the stack reads: [row0, row0 + rows)
    starts: np.ndarray           # int32 (P) first row (relative to row0) of each piece
    n_pool: np.ndarray           # int32 (P) pooled rows of each piece
    slot_start: np.ndarray       # int32 (P+1) partial slots of piece i are [slot_start[i], slot_start[i+1])
    slot_lo: np.ndarray          # int32 (W) window w reduces the partial slots [slot_lo[w], slot_hi[w])
    slot_hi: np.ndarray          # int32 (W)
    win_n_pool: np.ndarray       # int32 (W) pooled frames of each window, n - lost_frames
    n_slots: int


def check_windows(lengths, windows, lost_frames: int = TOTAL_CONTEXT):
    """(lengths int64 (R), windows int64 (W, 3)) after the checks of window_layout; ValueError for a bad window."""
    lengths = np.asarray(lengths, dtype=np.int64).reshape(-1)
    w = np.asarray(windows)
    if w.ndim != 2 or w.shape[1] != 3 or w.shape[0] < 1:
        raise ValueError("windows must be a (W >= 1, 3) integer array of (recording, first_frame, n_frames)")
    if w.dtype.kind not in "iu":
        raise ValueError("windows must be integers")
    w = w.astype(np.int64)
    rec, a, n = w[:, 0], w[:, 1], w[:, 2]
    if ((rec < 0) | (rec >= lengths.size)).any():
        raise ValueError(f"window recording index out of range [0, {lengths.size})")
    if (a < 0).any():
        raise ValueError("window first_frame must be >= 0")
    if (n <= lost_frames).any():
        raise ValueError(f"every window needs more than {lost_frames} frames (the TDNN context); got min {int(n.min())}")
    if (a + n > lengths[rec]).any():
        raise ValueError("a window runs past the end of its recording (first_frame + n_frames > length)")
    return lengths, w


def window_layout(lengths, windows, lost_frames: int = TOTAL_CONTEXT) -> WindowLayout:
    """Pooling layout of windows (recording, first_frame, n_frames) of the recordings of a flat matrix (recording k owns rows
    [sum(lengths[:k]), sum(lengths[:k+1]))), computed in O(W log W).

    Window [a, a+n) of a recording pools the stack's output rows a .. a+n-1-lost_frames, and output row r reads input rows
    r .. r+lost_frames only, so ONE pass over the recording yields them.  The pooled rows are cut at every window's first and
    one-past-last pooled row; the intervals between consecutive cuts that some window covers are the PIECES: disjoint, sorted by
    row, so the fused pooling epilogue sums each into its own slots exactly as it does utterances (xvec_build_layout takes them as
    they are).  A window then covers a run of consecutive pieces and with it the contiguous slot range [slot_lo, slot_hi).
    With windows = the whole recordings in order, the layout is utterance_layout's."""
    lengths, w = check_windows(lengths, windows, lost_frames)
    rec_start = np.concatenate(([0], np.cumsum(lengths)[:-1]))
    lo = rec_start[w[:, 0]] + w[:, 1]              # first pooled row of each window (absolute)
    hi = lo + w[:, 2] - lost_frames                # one past its last pooled row
    row0 = int(lo.min())
    rows = int((lo + w[:, 2]).max()) - row0        # the last input row any window reads, plus one
    if rows >= 2**31 - 256:
        raise ValueError("batch too large for 32-bit row indices; split it")
    cuts, inv = np.unique(np.concatenate((lo, hi)), return_inverse=True)
    cover = np.zeros(cuts.size, dtype=np.int64)    # windows covering [cuts[i], cuts[i+1])
    np.add.at(cover, inv[: lo.size], 1)
    np.add.at(cover, inv[lo.size:], -1)
    cover = np.cumsum(cover)[:-1]
    keep = np.nonzero(cover > 0)[0]                # interval i = [cuts[i], cuts[i+1]) is a piece
    starts = cuts[keep] - row0
    n_pool = cuts[keep + 1] - cuts[keep]
    slot_start = _slot_prefix(starts, n_pool)
    # first piece of a window: the one starting at its first pooled row; one past its last: the first piece starting at or after hi
    p_lo = np.searchsorted(starts, lo - row0, side="left")
    p_hi = np.searchsorted(starts, hi - row0, side="left")
    i32 = lambda v: np.ascontiguousarray(v, dtype=np.int32)
    return WindowLayout(row0, rows, i32(starts), i32(n_pool), i32(slot_start), i32(slot_start[p_lo]), i32(slot_start[p_hi]),
                        i32(w[:, 2] - lost_frames), int(slot_start[-1]))


def sliding_windows(lengths, window: int, shift: int) -> np.ndarray:
    """Windows (recording, first_frame, n_frames) of `window` frames every `shift` frames over each recording, int64 (W, 3), in
    recording order: starts 0, shift, 2 shift, ... while start + window <= T; when the last of them does not end at T, one more
    window [T - window, T) so that the end of the recording is covered; a recording shorter than `window` gets one window over
    all of it."""
    lengths = np.asarray(lengths, dtype=np.int64).reshape(-1)
    window, shift = int(window), int(shift)
    if window < 1 or shift < 1:
        raise ValueError("window and shift must be positive")
    out = []
    for k, t in enumerate(lengths.tolist()):
        if t <= window:
            out.append(np.asarray([[k, 0, t]], dtype=np.int64))
            continue
        a = np.arange(0, t - window + 1, shift, dtype=np.int64)
        if a[-1] + window < t:
            a = np.append(a, t - window)
        out.append(np.stack((np.full_like(a, k), a, np.full_like(a, window)), axis=1))
    return np.concatenate(out) if out else np.zeros((0, 3), dtype=np.int64)


def lpt_partition(lengths, n_parts: int, lost_frames: int = TOTAL_CONTEXT):
    """Longest-processing-time-first partition of utterances over `n_parts` workers by pooled frames.

    Returns a list of int64 index arrays (original utterance indices, each sorted by decreasing length so that a
    worker's batches are length-bucketed).  No data-path collective is needed: utterances are independent.
    """
    lengths = np.asarray(lengths, dtype=np.int64)
    order = np.argsort(-lengths, kind="stable")
    loads = np.zeros(n_parts, dtype=np.int64)
    parts = [[] for _ in range(n_parts)]
    for i in order:
        j = int(np.argmin(loads))
        parts[j].append(int(i))
        loads[j] += max(int(lengths[i]) - lost_frames, 1)
    return [np.asarray(p, dtype=np.int64) for p in parts]


def bucket_batches(lengths, max_frames: int, max_utts: int = 1 << 30):
    """Greedy length-bucketed batching: utterances sorted by decreasing length, cut whenever a batch would exceed
    max_frames total frames or max_utts utterances.  Returns a list of index arrays."""
    lengths = np.asarray(lengths, dtype=np.int64)
    order = np.argsort(-lengths, kind="stable")
    batches, cur, frames = [], [], 0
    for i in order:
        li = int(lengths[i])
        if cur and (frames + li > max_frames or len(cur) >= max_utts):
            batches.append(np.asarray(cur, dtype=np.int64))
            cur, frames = [], 0
        cur.append(int(i))
        frames += li
    if cur:
        batches.append(np.asarray(cur, dtype=np.int64))
    return batches


def balanced_batches(lengths, target_frames: int = 49152, multiple_of: int = 8):
    """Cut the utterance list (in its given order) into n contiguous batches of nearly equal total frames, n a multiple of
    `multiple_of` (so that 1, 2, 4 or 8 workers each get the same number of batches).  Returns a list of int64 index arrays.

    This is the unit of sharding that keeps results BIT-identical for any number of GPUs: a batch's composition — and with it
    the row position of every utterance inside the flat frame matrix, which fixes the fp32 summation order of its pooling — is a
    function of the lengths alone, never of the world size; worker r simply takes batches r, r + world, ...  (lpt_partition
    balances single utterances and is exact to one utterance, but a worker's batches then depend on the world size, and the
    x-vectors agree across world sizes only to fp32 rounding.)  Balance: batches differ by at most one utterance's frames."""
    lengths = np.asarray(lengths, dtype=np.int64).reshape(-1)
    if lengths.size == 0:
        raise ValueError("empty utterance list")
    total = int(lengths.sum())
    n = max(1, int(round(total / max(int(target_frames), 1) / multiple_of))) * multiple_of
    if n > lengths.size:
        n = int(lengths.size)
    ends = np.cumsum(lengths)
    cuts = [0]
    for k in range(1, n):
        want = total * k / n
        j = int(np.searchsorted(ends, want, side="left"))          # utterance boundary nearest to the k-th equal share
        if j > 0 and abs(int(ends[j - 1]) - want) <= abs(int(ends[min(j, ends.size - 1)]) - want):
            j -= 1
        j = min(max(j + 1, cuts[-1] + 1), lengths.size - (n - k))  # at least one utterance per batch, also in the remaining ones
        cuts.append(j)
    cuts.append(int(lengths.size))
    return [np.arange(a, b, dtype=np.int64) for a, b in zip(cuts[:-1], cuts[1:])]
