"""Windowed extraction against re-extraction of the sliced windows, in one process on one GPU.

    python tools/window_bench.py OUT_DIR [--precision bf16 tf32] [--recordings 24] [--reps 3]

Inputs: `recordings` 10-minute recordings (60 000 frames of 24 MFCCs each; 24 recordings = 138 MB of float32 frames, more than
the 126 MB of L2), device-resident.  For each window case (150/75, 300/150 and the dense 300/10 frames, layout.sliding_windows):
1. windowed: XVectorModel.extract_x_vec_windows over batches of consecutive whole recordings of <= 131 072 frames;
   re-extraction: the same windows cut out as utterances (the cutting is done once, outside the timed legs) through
   extract_x_vec_flat in batches of <= 131 072 frames.  Two streams, two scratch slots, the two paths alternated over `reps`
   repetitions (rotating which goes first); device time per leg from CUDA events -> windows/s.
2. Frame-level FLOPs of each path from shapes (bench.FLOPS_L / LOST per layer and output row) and their ratio.
3. The finalize (pool_finalize_kernel) and the stack kernel alone: summed kernel time of one windowed leg per case
   under torch.profiler (a separate, untimed run).
4. Agreement of the two paths: max-abs difference over max |re-extraction|.
5. The device name, power limit and max SM clock (nvidia-smi, read-only query) in the same run.

Writes OUT_DIR/window_bench.json.  Needs a CUDA device; without one it fails."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

FRAMES = 60_000          # 10 minutes at 100 frames/s
MAX_FRAMES = 1 << 17     # batch size of both paths (HostExtractor's default)
CASES = ((150, 75), (300, 150), (300, 10))


def frame_flops(rows):
    """Frame-level (TDNN1-5) FLOPs of one pass over `rows` frames, useful output rows only (bench.py's count)."""
    import bench
    return sum(f * (rows - l) for f, l in zip(bench.FLOPS_L, bench.LOST))


def kernel_us(prof, needle):
    """Summed device time (us) of the kernels whose name contains `needle`, and their count."""
    tot, n = 0.0, 0
    for e in prof.key_averages():
        if needle in e.key:
            tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            n += e.count
    return tot, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--precision", nargs="+", default=["bf16", "tf32"])
    ap.add_argument("--recordings", type=int, default=24)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        sys.exit("window_bench.py needs a CUDA device")
    import bench
    import xvec_b200
    from precision_bench import gpu_info

    dev = torch.device("cuda:0")
    info = gpu_info()
    info["torch_device_name"] = torch.cuda.get_device_name(dev)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(args.recordings * FRAMES, 24, generator=g).to(dev)
    per_batch = max(1, MAX_FRAMES // FRAMES)             # whole recordings per windowed batch
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def timed(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream()
        e0.record(cur)
        for st in streams:
            st.wait_event(e0)
        outs = []
        for i, c in enumerate(calls):
            with torch.cuda.stream(streams[i % 2]):
                outs.append(c(i % 2))
        for st in streams:
            cur.wait_stream(st)
        e1.record(cur)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), outs

    results = {}
    for precision in args.precision:
        m = bench.synthetic_model(xvec_b200, precision).to(dev).eval()
        res_p = {}
        for window, shift in CASES:
            w1 = xvec_b200.sliding_windows([FRAMES], window, shift)      # windows of one recording
            n_win = len(w1) * args.recordings
            # windowed: batches of `per_batch` whole recordings; the windows of each batch relative to it
            wins = np.concatenate([w1 + np.asarray([k, 0, 0]) for k in range(per_batch)])
            lens = [FRAMES] * per_batch
            win_calls = [(lambda s, r0=r0: m.extract_x_vec_windows(x[r0 * FRAMES:(r0 + per_batch) * FRAMES], lens, wins, slot=s))
                         for r0 in range(0, args.recordings, per_batch)]
            # re-extraction: every window cut out as an utterance, batches of <= MAX_FRAMES frames
            per_re = MAX_FRAMES // window
            idx = torch.from_numpy(np.concatenate([np.arange(a, a + n) + k * FRAMES
                                                   for k in range(args.recordings) for _, a, n in w1])).to(dev)
            xs = x.index_select(0, idx)
            del idx
            re_calls = []
            for i0 in range(0, n_win, per_re):
                nb = min(per_re, n_win - i0)
                re_calls.append(lambda s, i0=i0, nb=nb: m.extract_x_vec_flat(xs[i0 * window:(i0 + nb) * window], [window] * nb, slot=s))
            legs = {"windowed": win_calls, "re_extraction": re_calls}
            outs = {k: torch.cat(timed(c)[1]) for k, c in legs.items()}  # warm-up: modules, layouts, scratch of every shape
            ref = outs["re_extraction"]
            agree = float((outs["windowed"] - ref).abs().max() / ref.abs().max())
            del outs
            ms = {k: [] for k in legs}
            for r in range(args.reps):
                for k in (("windowed", "re_extraction") if r % 2 == 0 else ("re_extraction", "windowed")):
                    ms[k].append(timed(legs[k])[0])
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                timed(win_calls)
            fin_us, fin_n = kernel_us(prof, "pool_finalize_kernel")
            stack_us, stack_n = kernel_us(prof, "tdnn_stack_kernel")
            del xs, re_calls, legs
            torch.cuda.empty_cache()
            fl_win = (args.recordings // per_batch) * frame_flops(per_batch * FRAMES) + \
                (frame_flops((args.recordings % per_batch) * FRAMES) if args.recordings % per_batch else 0)
            fl_re = n_win * frame_flops(window)
            med = {k: float(np.median(v)) for k, v in ms.items()}
            res_p[f"{window}/{shift}"] = {
                "windows": n_win, "windows_per_recording": len(w1),
                "windows_per_s": {k: n_win / (v / 1e3) for k, v in med.items()},
                "leg_ms": {k: [float(t) for t in v] for k, v in ms.items()},
                "speedup_windowed_over_re_extraction": med["re_extraction"] / med["windowed"],
                "frame_level_flops": {"windowed": float(fl_win), "re_extraction": float(fl_re), "ratio_re_over_windowed": fl_re / fl_win},
                "profiled_windowed_leg": {"ranges_finalize_us": fin_us, "ranges_finalize_launches": fin_n,
                                          "stack_kernel_us": stack_us, "stack_kernel_launches": stack_n},
                "max_abs_diff_over_max_abs": agree,
            }
            print(precision, f"{window}/{shift}", json.dumps(res_p[f"{window}/{shift}"]["windows_per_s"]),
                  "finalize us", fin_us, "flop ratio", fl_re / fl_win, flush=True)
        results[precision] = res_p
        del m
        torch.cuda.empty_cache()

    out = {
        "what": f"{args.recordings} device-resident recordings of {FRAMES} frames ({args.recordings * FRAMES * 96 / 2**20:.0f} MiB of "
                f"float32 frames > L2), sliding windows window/shift in frames; windowed = extract_x_vec_windows on batches of "
                f"{per_batch} whole recordings, re_extraction = extract_x_vec_flat on the pre-cut windows in batches of <= "
                f"{MAX_FRAMES} frames; two streams; paths alternated over {args.reps} reps; medians",
        "gpu": info,
        "results": results,
        "watchdog_code": xvec_b200._lib.load().xvec_watchdog_code(),
        "unix_time": time.time(),
    }
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "window_bench.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["gpu"]))
    print(path)


if __name__ == "__main__":
    main()
