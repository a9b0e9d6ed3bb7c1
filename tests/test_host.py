"""CPU-side tests: the C-ABI library loads and exports every declared symbol (no compute calls), the flat-layout /
pooling bookkeeping is exact (emulated in numpy), partitioning, and the module surface mirrors the reference."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import xvec_b200
from oracle import xvector_oracle as ox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "xvec_b200.h")).read()
    declared = set(re.findall(r"XVEC_API\s+[\w\s\*]+?\b(xvec_\w+)\s*\(", header))
    assert len(declared) >= 13
    assert declared == set(xvec_b200._lib.EXPORTS)
    lib = ctypes.CDLL(xvec_b200._lib.LIB_PATH) if os.path.exists(xvec_b200._lib.LIB_PATH) else xvec_b200._lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    lib = xvec_b200._lib.load()
    assert lib.xvec_abi_version() == xvec_b200._lib.ABI_VERSION == int(re.search(r"#define XVEC_ABI_VERSION (\d+)", header).group(1))
    assert xvec_b200._lib.STACK_MAX_TAP_OFFSET == int(re.search(r"#define XVEC_STACK_MAX_TAP_OFFSET (\d+)", header).group(1))
    assert lib.xvec_watchdog_code() == 0  # readable without a device: the word lives in host memory
    assert lib.xvec_packed_k(24, 5, xvec_b200._lib.F32) == 160 and lib.xvec_packed_k(512, 3, xvec_b200._lib.BF16) == 1536
    assert lib.xvec_packed_k(3000, 1, xvec_b200._lib.BF16) == 3008 and lib.xvec_packed_n(1500) == 1536


def test_ctypes_signatures_have_the_headers_arity():
    """Every declared entry point takes as many arguments in the ctypes binding as in include/xvec_b200.h (a wrong count would
    shift pointers silently: ctypes does not check)."""
    header = open(os.path.join(ROOT, "include", "xvec_b200.h")).read()
    decls = re.findall(r"XVEC_API\s+[\w\s\*]+?\b(xvec_\w+)\s*\(([^;]*?)\);", header, re.S)
    assert len(decls) == len(xvec_b200._lib.EXPORTS)
    for name, params in decls:
        params = params.strip()
        n = 0 if params in ("void", "") else len([q for q in params.split(",") if q.strip()])
        assert n == len(xvec_b200._lib._SIGNATURES[name][1]), name


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu():
    lib = xvec_b200._lib.load()
    assert lib.xvec_device_check() != 0 and len(lib.xvec_last_error()) > 0
    m = xvec_b200.XVectorModel().eval()
    with pytest.raises(ValueError, match="no CPU path"):
        m.extract_x_vec(torch.randn(2, 40, 24))
    with pytest.raises(ValueError, match="no CPU path"):
        xvec_b200.TdnnLayer().eval()(torch.randn(2, 40, 24))
    with pytest.raises(ValueError, match="no CPU path"):
        m.stat_pool(torch.randn(2, 40, 1500))


def test_extract_forward_segment_layer_count():
    """xvec_extract_forward takes 0 to 2 segment layers.  Its arguments are checked before any CUDA call, so this needs no
    device: 3 layers are rejected; 0 layers with NULL fc_host / out_dev pass the checks and fail only at the missing device."""
    lib = xvec_b200._lib.load()
    tdnn = (xvec_b200._lib.LayerDesc * 2)()
    for d in tdnn:
        d.w_packed_dev, d.bias_dev, d.n, d.cin, d.taps, d.dtype = 256, 256, 256, 256, 1, xvec_b200._lib.F32
    fc = (xvec_b200._lib.LayerDesc * 3)()
    buf = 256  # stands for device pointers; nothing is dereferenced on these paths

    def call(fc_host, n_fc, out):
        return lib.xvec_extract_forward(tdnn, 2, buf, 300, 256, buf, buf, 256, buf, buf, buf, buf, 1, buf, None, None, buf, None,
                                        fc_host, n_fc, buf, None, 0, out, 256, None, 0, None)

    assert call(fc, 3, buf) == xvec_b200._lib.E_ARG
    if lib.xvec_device_check() != 0:  # no usable device: the call gets as far as the first CUDA call and reports its error
        assert call(None, 0, None) == lib.xvec_device_check() != xvec_b200._lib.E_ARG


def _emulate_fused_pool(lay, r):
    """numpy model of the EPI_POOL epilogue + finalize: per 128-row block, per utterance present -> one slot."""
    P = r.shape[1]
    part = np.full((lay.n_slots, 2, P), np.nan)
    B = xvec_b200._lib.POOL_BLOCK
    n_blocks = (lay.rows + B - 1) // B
    for b in range(n_blocks):
        rows = np.arange(b * B, min(lay.rows, b * B + B))
        us = lay.row_utt[rows]
        seg = 0
        for u in sorted(set(us[us >= 0].tolist())):
            sel = rows[us == u]
            assert (np.diff(sel) == 1).all()
            slot = lay.blk_slot_base[b] + seg
            assert np.isnan(part[slot]).all(), "slot written twice"
            part[slot, 0] = r[sel].sum(0)
            part[slot, 1] = (r[sel] ** 2).sum(0)
            seg += 1
    out = np.empty((lay.n_utts, 2 * P))
    for u in range(lay.n_utts):
        sl = part[lay.utt_slot_start[u]: lay.utt_slot_start[u + 1]]
        assert np.isfinite(sl).all()
        n = lay.n_pool[u]
        S, Q = sl[:, 0].sum(0), sl[:, 1].sum(0)
        out[u, :P] = S / n
        out[u, P:] = np.sqrt(np.maximum((Q - S * S / n) / (n - 1), 0)) if n > 1 else np.nan
    assert np.isfinite(part).all(), "unused slot"
    return out


@pytest.mark.parametrize("lens", [[300] * 7, [15, 16, 17, 31, 32, 33, 46, 47, 48, 127, 128, 129, 300, 2000, 15],
                                  list(np.random.default_rng(1).integers(15, 700, 60))])
def test_layout_bookkeeping_is_exact(lens):
    lay = xvec_b200.build_layout(lens)
    assert lay.rows == sum(lens) and lay.n_utts == len(lens)
    assert (lay.n_pool == np.asarray(lens) - 14).all()
    for u, (s, l) in enumerate(zip(lay.starts, lens)):
        assert (lay.row_utt[s:s + l - 14] == u).all() and (lay.row_utt[s + l - 14:s + l] == -1).all()
    assert lay.blk_slot_base.shape[0] == -(-lay.rows // 256) * (256 // xvec_b200._lib.POOL_BLOCK)
    rng = np.random.default_rng(0)
    r = np.abs(rng.standard_normal((lay.rows, 8)))
    got = _emulate_fused_pool(lay, r)
    for u, (s, n) in enumerate(zip(lay.starts, lay.n_pool)):
        seg = r[s:s + n]
        assert np.allclose(got[u, :8], seg.mean(0))
        if n > 1:
            assert np.allclose(got[u, 8:], seg.std(0, ddof=1))


def test_layout_rejects_short_or_empty():
    with pytest.raises(ValueError):
        xvec_b200.build_layout([300, 14])
    with pytest.raises(ValueError):
        xvec_b200.build_layout([])


def test_lpt_partition_and_buckets():
    lens = ox.synth_lengths(4874, 400, 2000, seed=3)
    for n in (1, 2, 4, 8):
        parts = xvec_b200.lpt_partition(lens, n)
        allidx = np.sort(np.concatenate(parts))
        assert np.array_equal(allidx, np.arange(len(lens)))          # a partition: every utterance exactly once
        loads = np.array([(lens[p] - 14).sum() for p in parts])
        assert loads.max() / loads.mean() < 1.001                    # length-balanced
    batches = xvec_b200.bucket_batches(lens, max_frames=200_000)
    assert np.array_equal(np.sort(np.concatenate(batches)), np.arange(len(lens)))
    assert all(lens[b].sum() <= 200_000 for b in batches)
    assert all(lens[b].max() - lens[b].min() <= 700 for b in batches)   # bucketed by length


def test_module_surface_mirrors_reference():
    m = xvec_b200.XVectorModel()
    sd = ox.make_state_dict(seed=0)
    assert set(m.state_dict().keys()) == set(sd.keys())               # reference checkpoint keys (SURVEY §8a)
    assert all(m.state_dict()[k].shape == sd[k].shape for k in sd)
    assert not m.load_state_dict(sd).missing_keys
    lay = m.time_context_layers[1]
    assert (lay.input_size, lay.output_size, lay.context, lay.batch_norm, lay.dropout_p) == (512, 512, [-2, 0, 2], True, 0.0)
    assert hasattr(lay, "linear") and hasattr(lay, "relu") and hasattr(lay, "norm") and not hasattr(lay, "drop")
    assert hasattr(xvec_b200.TdnnLayer(dropout_p=0.1), "drop")
    assert not hasattr(xvec_b200.TdnnLayer(batch_norm=False), "norm")
    assert m.x_vec_extract_layer == 6 and m.lost_frames == 14
    assert xvec_b200.tap_offsets([-2, -1, 0, 1, 2]) == [0, 1, 2, 3, 4] and xvec_b200.tap_offsets([-3, 0, 3]) == [0, 3, 6]
    for bad in ([-1, 0, 2], [0, 1, 2], []):
        with pytest.raises(ValueError):
            xvec_b200.tap_offsets(bad)
    with pytest.raises(RuntimeError, match="eval"):
        xvec_b200.XVectorModel().train().extract_x_vec(torch.randn(1, 30, 24))


def test_get_time_context_matches_reference_kat(kat):
    x = torch.from_numpy(kat["x"])
    for name in ("c5", "c2", "c5d2", "c11"):
        got = torch.cat(xvec_b200.get_time_context(x, kat[name + "_ctx"].tolist()), 2)
        assert torch.equal(got, torch.from_numpy(kat[name]))


def test_state_dict_interchange_with_reference(golden):
    """The reference model's state dict after torch.manual_seed(0) is pinned by its SHA-256 in the golden file (names and
    bytes); the oracle rebuilds it bit for bit, and it loads into ours strictly."""
    ref = ox.make_state_dict(seed=0, randomize_bn=False)
    assert ox.state_dict_digest(ref) == str(golden["default_init_digest"])
    ours = xvec_b200.XVectorModel()
    res = ours.load_state_dict(ref, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert torch.equal(ours.segment_layer6.weight, ref["segment_layer6.weight"])


def test_load_reference_checkpoint_roundtrip(tmp_path):
    """A Lightning checkpoint as the reference writes it (main.py:198,213): torch.save dict with 'state_dict' (+ extras)."""
    sd = ox.make_state_dict(seed=0)
    extra = dict(sd)
    extra["accuracy.tp"] = torch.zeros(1)          # torchmetrics state that the reference's module also saves
    path = str(tmp_path / "last.ckpt")
    torch.save({"state_dict": extra, "hyper_parameters": {"x_vec_extract_layer": 6}, "epoch": 3}, path)
    m = xvec_b200.XVectorModel()
    res = m.load_reference_checkpoint(path)
    assert not res.missing_keys and not res.unexpected_keys
    for k, v in sd.items():
        assert torch.equal(m.state_dict()[k], v), k


class Opaque:  # stands for the Lightning objects (callback state, hyper-parameter containers) a real checkpoint may pickle
    pass


def test_load_reference_checkpoint_rejects_incomplete_and_untrusted(tmp_path):
    sd = ox.make_state_dict(seed=0)
    short = {k: v for k, v in sd.items() if not k.startswith("segment_layer6")}
    path = str(tmp_path / "short.ckpt")
    torch.save({"state_dict": short}, path)
    with pytest.raises(KeyError, match="segment_layer6"):     # a silently random-initialised layer would be worse than an error
        xvec_b200.XVectorModel().load_reference_checkpoint(path)

    path2 = str(tmp_path / "pickled.ckpt")
    torch.save({"state_dict": sd, "callbacks": Opaque()}, path2)
    with pytest.raises(RuntimeError, match="trust_pickle"):   # the code-executing unpickler is opt-in only
        xvec_b200.XVectorModel().load_reference_checkpoint(path2)
    assert not xvec_b200.XVectorModel().load_reference_checkpoint(path2, trust_pickle=True).missing_keys


@pytest.mark.parametrize("rows,band", [(76800, 0), (76800, 5), (76800, 7), (76800, 1000), (300, 0), (257, 3), (131072, 0), (1536000, 0),
                                        (40000, 33)])
def test_stack_schedule_is_a_dependency_respecting_permutation(rows, band):
    """The work-item order of xvec_tdnn_stack (host replay of the device decode): every (layer, m_tile, n_tile) exactly once, and
    every tile after ALL tiles (layer-1, m_tile-1..m_tile+1, any n) it waits for — the precondition that makes in-order
    drawing + dependency flags deadlock-free for any number of resident CTA pairs."""
    import ctypes
    lib = xvec_b200._lib.load()
    n_tiles = [2, 2, 2, 2, 6]  # 512, 512, 512, 512, 1500 channels
    arr = (ctypes.c_int32 * 5)(*n_tiles)
    m_tiles = -(-rows // 256)
    total = lib.xvec_stack_plan(rows, 5, arr, band, None, 0)
    assert total == m_tiles * sum(n_tiles), lib.xvec_last_error()
    items = np.empty(total, dtype=np.uint32)
    assert lib.xvec_stack_plan(rows, 5, arr, band, items.ctypes.data_as(ctypes.c_void_p), total) == total
    layer, nt, mt = items & 7, (items >> 3) & 31, (items >> 8).astype(np.int64)
    assert layer.max() == 4 and (nt < np.asarray(n_tiles)[layer]).all() and mt.max() == m_tiles - 1
    key = (layer.astype(np.int64) * m_tiles + mt) * 8 + nt
    assert np.unique(key).size == total  # a permutation
    # position of the LAST item of every (layer, m_tile): a consumer must come after it
    last = np.full((5, m_tiles), -1, dtype=np.int64)
    np.maximum.at(last, (layer, mt), np.arange(total))
    pos = np.arange(total)
    for d in (-1, 0, 1):
        m_dep = mt + d
        ok = (layer > 0) & (m_dep >= 0) & (m_dep < m_tiles)
        assert (last[layer[ok] - 1, m_dep[ok]] < pos[ok]).all()
