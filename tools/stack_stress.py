#!/usr/bin/env python
"""Stress test of the tdnn_stack_kernel dependency protocol: many launches, several band heights, two launches in flight on two
streams (separate scratch), every result compared BITWISE with the per-layer launches (same tiles, same K order)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, xvec_b200
from xvec_b200 import ops
from oracle import xvector_oracle as ox

sd = ox.make_state_dict(0)
bad = 0
for precision in ("bf16", "tf32"):
    m = xvec_b200.XVectorModel(precision=precision); m.load_state_dict(sd); m = m.cuda().eval()
    rng = np.random.default_rng(int(os.environ.get("STRESS_SEED", "11")))
    for trial in range(4):
        lens = rng.integers(15, 1200, size=int(rng.integers(40, 220)))
        flat = torch.randn(int(lens.sum()), 24, device="cuda")
        lay = m._layout_for(lens)
        pipe = m._pipeline()
        stack = m._stack_params()[0]
        layers = list(m.time_context_layers)
        scs = [m._scratch_for(s) for s in range(2)]
        for sc in scs:
            sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
        xs = xs1 = flat
        rows = flat.shape[0]
        # reference: one launch per layer
        h = flat
        for i, layer in enumerate(layers[:-1]):
            w, bias, offs = stack[i]
            if i == 0 and pipe["window"] is not None:
                view = torch.as_strided(torch.cat([xs, xs.new_zeros(4, 24)]), (rows, 120), (24, 1))  # overlapping rows; windows past `rows` read as zero
                h = ops.tdnn_layer_flat(view, pipe["window"]["w"], 512, [0], bias, None, None, relu=True, out_dtype=m.act_dtype, cin=120)
            else:
                h = ops.tdnn_layer_flat(h, w, layer.output_size, offs, bias, None, None, relu=True, out_dtype=m.act_dtype, cin=layer.input_size)
        w, bias, offs = stack[-1]
        ref = torch.zeros((lay.n_slots, 2, 1500), device="cuda")
        ops.tdnn_pool_fused(h, w, 1500, offs, bias, lay.row_utt, lay.blk_slot_base, ref)
        torch.cuda.synchronize()
        streams = [torch.cuda.Stream() for _ in range(2)]
        for band in (0, 5, 9, 33, 0):
            parts = [[torch.zeros_like(ref) for _ in range(8)] for _ in range(2)]
            for rep in range(8):
                for s in range(2):
                    with torch.cuda.stream(streams[s]):
                        ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], xs if s == 0 else xs1, scs[s].act[0], scs[s].act[1], lay.row_utt,
                                       lay.blk_slot_base, parts[s][rep], scs[s].ctrl, band=band)
            torch.cuda.synchronize()
            for s in range(2):
                for rep in range(8):
                    if not torch.equal(parts[s][rep], ref):
                        bad += 1
                        print("MISMATCH", precision, trial, band, s, rep, (parts[s][rep] - ref).abs().max().item(), flush=True)
        print(precision, "trial", trial, "rows", lay.rows, "utts", len(lens), "ok" if bad == 0 else f"bad={bad}", flush=True)
print("watchdog", xvec_b200._lib.load().xvec_watchdog_code(), "mismatches", bad)
sys.exit(1 if bad else 0)
