"""CPU tests of windowed extraction (x-vectors of windows of recordings from one pass of the frame-level stack): the piece layout
of layout.window_layout, a numpy restatement of the fused pooling epilogue + the ranges finalize on it, sliding_windows and the
validation."""
import dataclasses

import numpy as np
import pytest

import xvec_b200
from xvec_b200 import layout as L

B = xvec_b200._lib.POOL_BLOCK


def _random_windows(rng, lengths, lost, n):
    """Arbitrary windows: random starts / sizes, windows touching both recording ends, shifts of 1-3 frames, duplicates."""
    out = []
    for k, t in enumerate(lengths):
        for _ in range(n):
            size = int(rng.integers(lost + 1, t + 1))
            out.append((k, int(rng.integers(0, t - size + 1)), size))
        size = int(rng.integers(lost + 1, t + 1))
        out += [(k, 0, size), (k, t - size, size), (k, 0, t)]
        a = int(rng.integers(0, max(1, t - size - 8)))
        for s in (1, 2, 3):  # several pieces in one 32-row sub-block
            if a + s + size <= t:
                out.append((k, a + s, size))
        out.append(out[-1])
    w = np.asarray(out, dtype=np.int64)
    return w[rng.permutation(len(w))]


def _expand(wl):
    """numpy statement of xvec_build_layout on the pieces: row_utt (piece of a pooled row, -1 elsewhere), blk_slot_base."""
    row_utt = np.full(wl.rows, -1, dtype=np.int64)
    for i, (s, n) in enumerate(zip(wl.starts, wl.n_pool)):
        row_utt[s:s + n] = i
    n_blocks = -(-wl.rows // 256) * (256 // B)
    last = wl.starts.astype(np.int64) + wl.n_pool - 1
    blk_slot_base = np.zeros(n_blocks, dtype=np.int64)
    for b in range(n_blocks):
        p = int(np.searchsorted(last, b * B, side="left"))  # first piece whose last pooled row is in or after block b
        if p < len(wl.starts):
            b0 = wl.starts[p] // B
            blk_slot_base[b] = wl.slot_start[p] + max(b - b0, 0)
    return row_utt, blk_slot_base


def _epilogue(wl, row_utt, blk_slot_base, r):
    """The fused pooling epilogue: per 128-row block, one slot per piece with a row in it, numbered from blk_slot_base."""
    part = np.full((wl.n_slots, 2, r.shape[1]), np.nan)
    for b in range(-(-wl.rows // B)):
        rows = np.arange(b * B, min(wl.rows, b * B + B))
        us = row_utt[rows]
        for j, u in enumerate(sorted(set(us[us >= 0].tolist()))):
            sel = rows[us == u]
            slot = blk_slot_base[b] + j
            assert np.isnan(part[slot]).all(), "slot written twice"
            part[slot, 0] = r[sel].sum(0)
            part[slot, 1] = (r[sel] ** 2).sum(0)
    assert np.isfinite(part).all(), "unused slot"
    return part


def _finalize_ranges(wl, part):
    P = part.shape[2]
    out = np.empty((len(wl.slot_lo), 2 * P))
    for w, (lo, hi, n) in enumerate(zip(wl.slot_lo, wl.slot_hi, wl.win_n_pool)):
        S, Q = part[lo:hi, 0].sum(0), part[lo:hi, 1].sum(0)
        out[w, :P] = S / n
        out[w, P:] = np.sqrt(np.maximum((Q - S * S / n) / (n - 1), 0)) if n > 1 else np.nan
    return out


@pytest.mark.parametrize("lost", [14, 20])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_window_layout_pieces_and_slot_ranges(lost, seed):
    rng = np.random.default_rng(seed)
    lengths = rng.integers(lost + 1, 700, 5).tolist() + [lost + 1, 2000]
    w = _random_windows(rng, lengths, lost, 6)
    wl = xvec_b200.window_layout(lengths, w, lost)
    rec_start = np.concatenate(([0], np.cumsum(lengths)[:-1]))
    lo = rec_start[w[:, 0]] + w[:, 1] - wl.row0
    hi = lo + w[:, 2] - lost
    assert lo.min() == 0 and wl.starts[0] == 0
    assert wl.rows == (lo + w[:, 2]).max() and wl.rows + wl.row0 <= sum(lengths)
    s, n = wl.starts.astype(np.int64), wl.n_pool.astype(np.int64)
    # pieces: non-empty, sorted, disjoint, inside one recording's pooled rows, each covered by some window
    assert (n >= 1).all() and (s[1:] >= s[:-1] + n[:-1]).all()
    k = np.searchsorted(rec_start - wl.row0, s, side="right") - 1
    assert (s + n <= rec_start[k] - wl.row0 + np.asarray(lengths)[k] - lost).all()
    assert all(((lo <= a) & (a + m <= hi)).any() for a, m in zip(s, n))
    assert (wl.slot_start == L._slot_prefix(s, n)).all()
    assert wl.n_slots == wl.slot_start[-1] and (wl.win_n_pool == w[:, 2] - lost).all()
    for i in range(len(w)):
        p = np.nonzero((wl.slot_start[:-1] >= wl.slot_lo[i]) & (wl.slot_start[:-1] < wl.slot_hi[i]))[0]
        # the window's piece run: consecutive pieces that tile exactly its pooled rows
        assert p.size and (np.diff(p) == 1).all()
        assert s[p[0]] == lo[i] and s[p[-1]] + n[p[-1]] == hi[i] and (s[p[1:]] == s[p[:-1]] + n[p[:-1]]).all()
        assert n[p].sum() == w[i, 2] - lost
        assert wl.slot_lo[i] == wl.slot_start[p[0]] and wl.slot_hi[i] == wl.slot_start[p[-1] + 1]
        # its slots: exactly one per (128-row block, piece) pair of its rows
        pairs = {(r // B, j) for j in p for r in range(s[j], s[j] + n[j])}
        assert wl.slot_hi[i] - wl.slot_lo[i] == len(pairs)


@pytest.mark.parametrize("seed,late", [(3, False), (4, False), (5, True)])
def test_epilogue_and_ranges_finalize_equal_direct_window_statistics(seed, late):
    """late: no window reads the first frames, so the stack starts at row0 > 0 (the rows before it are not passed at all)."""
    rng = np.random.default_rng(seed)
    lengths = [300, 40, 777, 15, 1200]
    w = np.concatenate([_random_windows(rng, lengths, 14, 4), L.sliding_windows(lengths, 150, 75), [[3, 0, 15], [1, 5, 16]]])
    if late:
        w = w[(w[:, 0] >= 1) & (w[:, 1] >= 3)]
    wl = xvec_b200.window_layout(lengths, w)
    assert (wl.row0 > 0) == late and wl.starts[0] == 0
    row_utt, blk_slot_base = _expand(wl)
    r = np.abs(rng.standard_normal((wl.rows, 6)))
    got = _finalize_ranges(wl, _epilogue(wl, row_utt, blk_slot_base, r))
    rec_start = np.concatenate(([0], np.cumsum(lengths)[:-1]))
    for i, (k, a, n) in enumerate(w):
        seg = r[rec_start[k] + a - wl.row0: rec_start[k] + a - wl.row0 + n - 14]
        assert np.allclose(got[i, :6], seg.mean(0), rtol=1e-12, atol=1e-12)
        if n - 14 > 1:
            assert np.allclose(got[i, 6:], seg.std(0, ddof=1), rtol=1e-9, atol=1e-12)
        else:
            assert np.isnan(got[i, 6:]).all()  # one pooled frame: NaN, like torch.std


@pytest.mark.parametrize("lengths", [[300, 45, 1000, 15], [15], [128, 129, 256, 257],
                                     [142, 142, 142],    # 128 pooled rows each, starting off block boundaries
                                     [16] * 20,          # two pooled rows each, many utterances per 128-row block
                                     [141, 15, 142],     # 127, 1 and 128 pooled rows: a one-frame utterance between block edges
                                     [5000, 15, 300]])   # one utterance spanning 39 blocks
def test_whole_recording_windows_equal_the_utterance_layout(lengths):
    w = np.stack([np.arange(len(lengths)), np.zeros(len(lengths), dtype=np.int64), lengths], 1)
    wl = xvec_b200.window_layout(lengths, w)
    ul = L.utterance_layout(lengths)
    assert type(ul) is type(wl) and wl.row0 == 0
    for f in dataclasses.fields(wl):
        a, b = getattr(wl, f.name), getattr(ul, f.name)
        if isinstance(a, np.ndarray):
            assert a.dtype == b.dtype == np.int32 and np.array_equal(a, b), f.name
        else:
            assert type(a) is type(b) is int and a == b, f.name
    assert np.array_equal(ul.slot_lo, ul.slot_start[:-1]) and np.array_equal(ul.slot_hi, ul.slot_start[1:])
    lay = xvec_b200.build_layout(lengths)
    row_utt, blk_slot_base = _expand(wl)
    assert np.array_equal(row_utt, lay.row_utt)
    used = [b for b in range(blk_slot_base.size) if (row_utt[b * B:(b + 1) * B] >= 0).any()]  # blocks without a pooled row read none
    assert np.array_equal(blk_slot_base[used], lay.blk_slot_base[used])


def test_sliding_windows_policy():
    w = xvec_b200.sliding_windows([600, 100, 150, 151, 300], 150, 75)
    by = {k: w[w[:, 0] == k, 1:].tolist() for k in range(5)}
    assert by[0] == [[a, 150] for a in (0, 75, 150, 225, 300, 375, 450)]  # ends exactly at T: no extra window
    assert by[1] == [[0, 100]]                                             # shorter than the window: one window over all of it
    assert by[2] == [[0, 150]]
    assert by[3] == [[0, 150], [1, 150]]                                   # the last regular window misses frame 150: [T-150, T)
    assert by[4] == [[0, 150], [75, 150], [150, 150]]
    assert w.dtype == np.int64 and (w[:, 1] + w[:, 2] <= np.asarray([600, 100, 150, 151, 300])[w[:, 0]]).all()
    w = xvec_b200.sliding_windows([1000], 300, 10)
    assert w[-1, 1] == 700 and len(w) == 71 and (np.diff(w[:, 1]) == 10).all()
    for bad in ((0, 10), (10, 0)):
        with pytest.raises(ValueError):
            xvec_b200.sliding_windows([100], *bad)


@pytest.mark.parametrize("windows,match", [
    (np.zeros((0, 3), dtype=np.int64), "W >= 1"),
    (np.asarray([0, 0, 50]), "W >= 1"),
    (np.asarray([[0, 0, 50.0]]), "integers"),
    (np.asarray([[2, 0, 50]]), "recording index"),
    (np.asarray([[-1, 0, 50]]), "recording index"),
    (np.asarray([[0, -1, 50]]), "first_frame"),
    (np.asarray([[0, 0, 14]]), "more than 14"),
    (np.asarray([[1, 10, 91]]), "past the end"),
])
def test_window_validation(windows, match):
    with pytest.raises(ValueError, match=match):
        xvec_b200.window_layout([200, 100], windows)


def test_window_validation_uses_the_models_lost_frames():
    assert xvec_b200.window_layout([100], [[0, 0, 15]]).win_n_pool.tolist() == [1]
    with pytest.raises(ValueError, match="more than 20"):
        xvec_b200.window_layout([100], [[0, 0, 20]], lost_frames=20)
