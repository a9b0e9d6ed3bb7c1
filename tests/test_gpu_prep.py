"""Operand preparation on a B200: the private members bench.py times the model through, the prepared-operand cache (no
rebuild while parameters stay put, exactly the stale operands rebuilt when they change) and the one split-K workspace per slot."""
import math

import numpy as np
import pytest
import torch

from oracle import xvector_oracle as ox

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xb():
    import xvec_b200
    assert xvec_b200._lib.load().xvec_device_check() == 0, xvec_b200._lib.load().xvec_last_error()
    return xvec_b200


def _model(xb, sd, precision):
    m = xb.XVectorModel(precision=precision)
    m.load_state_dict(sd)
    return m.cuda().eval()


@pytest.mark.parametrize("precision", ["bf16", "tf32"])
def test_bench_reaches_the_model_internals_it_times(xb, precision):
    """bench.py times the per-layer launches and the stack kernel alone through _layout_for, _scratch_for, _stack_params,
    _pipeline, _frames_for and _head: their names, signatures and return shapes are its interface."""
    import bench
    from xvec_b200 import ops
    m = bench.synthetic_model(xb, precision).cuda().eval()
    lengths = [300] * 8
    x_dev = torch.randn(2, 2400, 24, device="cuda")
    times = bench.instrumented_layer_times(m, x_dev, lengths, n_batches=2, iters=1)
    assert len(times) == 7 and all(math.isfinite(t) and t > 0 for t in times.values()), times
    # the launch() body of bench.Arm.stack_launch_times, against the pooling partials of the whole extraction path
    m.pooled_stats_flat(x_dev[0], lengths)
    lay = m._layout_for(lengths)
    sc = m._scratch_for(0)
    sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
    ref = sc.part[: lay.n_slots].clone()
    pipe = m._pipeline()
    part = torch.zeros_like(ref)
    ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], m._frames_for(x_dev[0], pipe), sc.act[0], sc.act[1], lay.row_utt, lay.blk_slot_base,
                   part, sc.ctrl)
    torch.cuda.synchronize()
    assert torch.equal(part, ref)


@pytest.mark.parametrize("precision", ["bf16", "tf32"])
def test_operands_are_packed_once_and_rebuilt_only_when_stale(xb, state_dict, precision, monkeypatch):
    """Weights are packed on the first call of each kind only, whatever the slot and stream.  An in-place change of one
    BatchNorm statistic repacks exactly the frame-level stack (its five layers plus the window form of layer 0); a replaced
    segment layer takes the place of the old one.  Either way the model then computes what a fresh model with its state does."""
    from xvec_b200 import ops
    packs = []
    pack_weight = ops.pack_weight

    def counting(weight, taps, cin, dtype):
        packs.append((weight.shape[0], taps, cin))
        return pack_weight(weight, taps, cin, dtype)

    def packs_per_call(fn, n):
        counts = []
        for i in range(n):
            before = len(packs)
            fn(i)
            counts.append(len(packs) - before)
        return counts

    monkeypatch.setattr(ops, "pack_weight", counting)
    m = _model(xb, state_dict, precision)
    lens = np.asarray([300] * 6 + [45, 16, 777, 120])
    flat = torch.cat(ox.synth_ragged(lens, seed=3)).cuda()
    x = ox.synth_mfcc(8, 300, seed=4).cuda()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = []

    def extract(i):
        streams[i % 2].wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(streams[i % 2]):
            outs.append(m.extract_x_vec_flat(flat, lens, slot=i % 2))

    assert packs_per_call(extract, 10) == [7] + [0] * 9  # TDNN1-5, TDNN1 in window form, segment6
    torch.cuda.synchronize()
    assert all(torch.equal(o, outs[0]) for o in outs)
    assert packs_per_call(lambda i: m(x), 2) == [2, 0]  # segment7 and output; segment6 is shared with extraction
    n_entries = len(m._prep._entries)

    with torch.no_grad():
        m.time_context_layers[2].norm.running_var.mul_(1.5)
    packs.clear()
    out = m.extract_x_vec_flat(flat, lens)
    stack = [(l.output_size, len(l.context), l.input_size) for l in m.time_context_layers] + [(512, 1, 5 * 24)]
    assert sorted(packs) == sorted(stack)
    assert torch.equal(out, _model(xb, m.state_dict(), precision).extract_x_vec_flat(flat, lens))

    torch.manual_seed(5)
    m.segment_layer6 = torch.nn.Linear(3000, 512).cuda()
    f = _model(xb, m.state_dict(), precision)
    assert torch.equal(m.extract_x_vec(x), f.extract_x_vec(x))
    assert torch.equal(m(x), f(x))
    assert len(m._prep._entries) == n_entries  # the replaced layer's operands took the place of the old ones
    assert xb._lib.load().xvec_watchdog_code() == 0


@pytest.mark.parametrize("precision", ["bf16", "tf32"])
def test_forward_keeps_one_split_k_workspace(xb, state_dict, precision):
    """forward() runs the segment layers with split-K through its slot's one workspace: once the scratch has reached its size,
    more batch sizes add only their layouts (a few KiB each), not a workspace each."""
    m = _model(xb, state_dict, precision)
    x = ox.synth_mfcc(24, 300, seed=8).cuda()
    m(x)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    for b in range(1, 24):
        m(x[:b])
    torch.cuda.synchronize()
    growth = torch.cuda.memory_allocated() - before
    assert growth < 16 << 20, f"{growth / 2**20:.1f} MiB"
