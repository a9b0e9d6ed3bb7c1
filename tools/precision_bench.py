"""The three precisions side by side, in one process on one GPU: bf16, fp16 and tf32.

    python tools/precision_bench.py OUT_DIR [--reps 5] [--steps 30] [--stack-launches 100]

1. Config c2 of bench.py (1024 x 300 frames per step as 4 batches of 256, two batches in flight on two streams, inputs
   resident on the device in a pool larger than L2), the precisions alternated over `reps` repetitions (rotating which
   one goes first), device time per leg from CUDA events -> utt/s.
2. The tdnn_stack_kernel launch alone (xvec_tdnn_stack on one batch of 256 x 300), CUDA events around `stack-launches`
   back-to-back launches, alternated the same way.
3. Parity of a sample of utterances against the float64 CPU oracle (max-abs error per row / row norm, min cosine).
4. The device name, power limit and max SM clock, read with nvidia-smi (read-only query) in the same run.

Writes OUT_DIR/precision_bench.json.  Needs a CUDA device; without one it fails."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PRECISIONS = ("bf16", "fp16", "tf32")
BATCH, FRAMES, BATCHES_PER_STEP = 256, 300, 4
L2_BYTES = 126 * 2 ** 20


def gpu_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        line = r.stdout.strip().splitlines()[0]
        name, power, clock, driver = [v.strip() for v in line.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock, "driver": driver}
    except Exception as e:  # recorded, not fatal: the timings are still what this run measured
        return {"error": f"nvidia-smi query failed: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--stack-launches", type=int, default=100)
    args = ap.parse_args()

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        sys.exit("precision_bench.py needs a CUDA device")
    import bench
    import xvec_b200
    from oracle import xvector_oracle as ox

    dev = torch.device("cuda:0")
    info = gpu_info()
    info["torch_device_name"] = torch.cuda.get_device_name(dev)

    # device-resident inputs: a pool of distinct batches larger than L2, cycled through
    per_batch = BATCH * FRAMES * 24 * 4
    n_res = max(8, -(-2 * L2_BYTES // per_batch))
    g = torch.Generator().manual_seed(1)
    x_dev = [torch.randn(BATCH * FRAMES, 24, generator=g).to(dev) for _ in range(n_res)]
    lengths = [FRAMES] * BATCH

    models = {p: bench.synthetic_model(xvec_b200, p).to(dev).eval() for p in PRECISIONS}
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def leg(m, n_batches):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream()
        e0.record(cur)
        for st in streams:
            st.wait_event(e0)
        for i in range(n_batches):
            with torch.cuda.stream(streams[i % 2]):
                m.extract_x_vec_flat(x_dev[i % n_res], lengths, slot=i % 2)
        for st in streams:
            cur.wait_stream(st)
        e1.record(cur)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    # the stack kernel alone: the model's own operands and scratch, one batch
    from xvec_b200 import ops
    stack_args = {}
    for p, m in models.items():
        lay = m._layout_for(np.asarray(lengths))
        pipe = m._pipeline()
        sc = m._scratch_for(0)
        sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
        part = torch.zeros((lay.n_slots, 2, 1500), device=dev)
        stack_args[p] = (pipe, sc, lay, part)

    def stack_leg(p, n):
        pipe, sc, lay, part = stack_args[p]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], x_dev[i % n_res], sc.act[0], sc.act[1], lay.row_utt, lay.blk_slot_base, part, sc.ctrl)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n * 1e3  # us per launch

    for p, m in models.items():  # warm every shape: modules, plans, scratch
        leg(m, 2 * BATCHES_PER_STEP)
        stack_leg(p, 5)

    n_batches = args.steps * BATCHES_PER_STEP
    e2e = {p: [] for p in PRECISIONS}
    stack = {p: [] for p in PRECISIONS}
    for r in range(args.reps):
        order = PRECISIONS[r % 3:] + PRECISIONS[:r % 3]
        for p in order:
            ms = leg(models[p], n_batches)
            e2e[p].append(n_batches * BATCH / (ms / 1e3))
        for p in order:
            stack[p].append(stack_leg(p, args.stack_launches))

    # parity against the float64 oracle on a sample of one resident batch
    sd = models["tf32"].state_dict()
    sd = {k: v.detach().cpu() for k, v in sd.items()}
    sel = np.random.default_rng(0).choice(BATCH, 16, replace=False)
    xb0 = x_dev[0].view(BATCH, FRAMES, 24)
    ref = ox.extract_x_vec_t(sd, xb0[sel].cpu(), 6).double().numpy()
    parity = {}
    for p, m in models.items():
        got = m.extract_x_vec(xb0).double().cpu().numpy()[sel]
        rel = np.abs(got - ref).max(1) / np.linalg.norm(ref, axis=1)
        cos = (got * ref).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(ref, axis=1))
        parity[p] = {"max_rel_err": float(rel.max()), "min_cos": float(cos.min()), "finite": bool(np.isfinite(got).all())}

    def summary(v):
        a = np.asarray(v)
        return {"median": float(np.median(a)), "min": float(a.min()), "max": float(a.max()), "all": [float(t) for t in a]}

    res = {
        "what": "c2: 1024 x 300 frames per step as 4 batches of 256, two in flight, device-resident inputs "
                f"({n_res} distinct batches, {n_res * per_batch / 2**20:.0f} MiB > L2); precisions alternated",
        "gpu": info,
        "reps": args.reps, "steps_per_leg": args.steps, "stack_launches_per_leg": args.stack_launches,
        "c2_device_utt_per_s": {p: summary(v) for p, v in e2e.items()},
        "stack_kernel_us_per_launch_256x300": {p: summary(v) for p, v in stack.items()},
        "ratios": {
            "fp16_over_bf16_c2_utt_per_s": float(np.median(e2e["fp16"]) / np.median(e2e["bf16"])),
            "fp16_over_bf16_stack_time": float(np.median(stack["fp16"]) / np.median(stack["bf16"])),
            "tf32_over_bf16_c2_utt_per_s": float(np.median(e2e["tf32"]) / np.median(e2e["bf16"])),
        },
        "parity_vs_fp64_oracle_16_utts": parity,
        "watchdog_code": xvec_b200._lib.load().xvec_watchdog_code(),
        "unix_time": time.time(),
    }
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "precision_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "ratios", "parity_vs_fp64_oracle_16_utts")}))
    print(path)


if __name__ == "__main__":
    main()
