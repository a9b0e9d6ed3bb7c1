#!/usr/bin/env python
"""Experiment: does the tail of a batch (pool_finalize + segment6) cost step time because of stream ORDER (the next stack kernel of
the same slot waits for it) or because of SM occupancy?  Variant A: everything of a slot on one stream (the product path).
Variant B: the stack kernel on the slot's main stream, the tail on a second stream behind an event."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, xvec_b200
from xvec_b200 import ops
from oracle import xvector_oracle as ox

m = xvec_b200.XVectorModel(precision="bf16"); m.load_state_dict(ox.make_state_dict(0)); m = m.cuda().eval()
B, T, NRES, NS = 256, 300, 24, 2
x = torch.randn(NRES, B * T, 24, device="cuda")
lengths = [T] * B
lay = m._layout_for(lengths)
pipe = m._pipeline()
scs = []
for s in range(2 * NS):
    sc = m._scratch_for(s); sc.ensure(lay.rows, lay.n_slots, lay.n_utts); sc.ensure_head(lay.n_utts, pipe["fc_shapes"], pipe["hidden"]); scs.append(sc)
w6, b6 = m._fc("segment_layer6", m.act_dtype)
main = [torch.cuda.Stream() for _ in range(NS)]
tail = [torch.cuda.Stream() for _ in range(NS)]
evs = [[torch.cuda.Event() for _ in range(2)] for _ in range(2 * NS)]

def step(i, split):
    s = i % NS
    k = i % (2 * NS) if split else s       # scratch set: the split variant alternates two sets per slot
    sc = scs[k]
    part = sc.part[: lay.n_slots]; pooled = sc.pooled[: lay.n_utts]; pooled_lp = sc.pooled_lp[: lay.n_utts]
    with torch.cuda.stream(main[s]):
        if split: main[s].wait_event(evs[k][1])      # the tail that last read this scratch set is done
        xs = x[i % NRES]
        ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], xs, sc.act[0], sc.act[1], lay.row_utt, lay.blk_slot_base, part, sc.ctrl)
        if split: evs[k][0].record(main[s])
    with torch.cuda.stream(tail[s] if split else main[s]):
        if split: tail[s].wait_event(evs[k][0])
        ops.pool_finalize(part, lay.utt_slot_start, lay.n_pool, 1500, pipe["scale5"], pipe["shift5"], out=pooled, out_lp=pooled_lp)
        # segment6 split-K through this scratch set's own workspace (model._head uses slot 0's, which both streams would share)
        ops.tdnn_layer_flat(pooled_lp, w6, 512, [0], b6, None, None, relu=False, out_dtype=torch.float32, cin=3000, workspace=sc.ws)
        if split: evs[k][1].record(tail[s])

for split in (False, True, False, True):
    for i in range(12): step(i, split)
    torch.cuda.synchronize()
    n = 300
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for st in main + tail: st.wait_event(e0)
    for i in range(n): step(i, split)
    cur = torch.cuda.current_stream()
    for st in main + tail: cur.wait_stream(st)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    print(f"tail on {'a second stream' if split else 'the same stream'}: {ms * 1e3:.1f} us/step  {B / ms * 1e3:,.0f} utt/s", flush=True)
