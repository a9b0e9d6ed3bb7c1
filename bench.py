#!/usr/bin/env python
"""Benchmark of the x-vector extraction hot path (BASELINE.json metric: x-vectors/sec & frames/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dtype bf16|tf32] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...        (one rank per GPU)

A step = one pass of the hot path (TDNN1-5 -> statistics pooling -> segment6) over the workload of BASELINE.json configs[1]:
1024 fixed-length 3 s utterances = 4 batches of 256 x 300 x 24 MFCC per step and GPU (weak scaling: every GPU runs its own set).
  value      utterances/s, device-resident inputs (more distinct batches than fit in L2), exactly K steps in one CUDA-event
             bracket, two batches in flight on two streams
  e2e        utterances/s through the public host API (HostExtractor): pinned host MFCCs -> H2D -> kernels -> D2H x-vectors
  long       the same two legs over ~0.6 s each (2048 batches), i.e. mostly under the 1000 W power cap, + host probes
             (H2D GB/s per rank with all ranks copying, host enqueue time per batch, CPU affinity)
  roofline   tcgen05 TDNN stack kernel: algorithmic FLOPs of a launch / its CUDA-event time, in TWO regimes, each against the
             measured cuBLAS peak of the same regime: burst (30 launches from idle / MEASURED_PEAKS bf16_tflops) and sustained
             (back to back for >= 1.2 s, last half / bf16_tflops_sustained); frac = the regime the driver's K-step leg ran in
  tf32       the same value / e2e / roofline in fp32-storage TF32-math mode (the reference's arithmetic is fp32), against a
             TF32 cuBLAS peak measured here the way MEASURED_PEAKS.json measures bf16
  c5         BASELINE.json configs[4]: 4874 utterances of 4-20 s sharded by utterance over the N GPUs (LPT), per-rank
             HostExtractor, one NCCL all-gather of the embeddings, 37,720 centred-cosine trials; wall utt/s (strong scaling)
  cpu_baseline  the oracle (port of the reference's fp32 PyTorch path) on this box's host cores, bounded sample
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH, FRAMES, CEPS, N_UTTS = int(os.environ.get("XVEC_BENCH_BATCH", "256")), 300, 24, 1024  # BASELINE.json configs[1]
N_UTTS = (N_UTTS // BATCH) * BATCH
BATCHES_PER_STEP = N_UTTS // BATCH
FLOPS_L = [122_880, 1_572_864, 1_572_864, 524_288, 1_536_000]  # per output frame, SURVEY §8d
LOST = [4, 8, 14, 14, 14]
SEG6_FLOPS = 3_072_000
LAUNCHES_PER_BATCH = 3  # tdnn_stack_kernel, pool_finalize_kernel, fc_small_kernel (segment6)
LONG_BATCHES = 2048     # the "long" legs: ~0.6 s of bf16 work per GPU
WORKLOAD = "c2: 1024 x 3 s utterances (300 x 24 MFCC) per step and GPU as 4 batches of 256, x_vec_extract_layer 6"
NCU_TENSOR_PIPE = {"sm__pipe_tensor_cycles_active_pct_of_elapsed": 84.1, "file": "profiles/r02f_stack_ncu_full_summary.txt",
                   "note": "ncu --set full capture of one tdnn_stack_kernel launch of the final code (cold, serialised, 241.5 us at 1.72 GHz = 414 k "
                           "cycles; before the last session's fence / hand-off / publication changes: 77.1-78.3 %, 445-452 k cycles); ~7 % of the issued "
                           "MMA work is padding (don't-care rows of the flat layout, N 1500 -> 1536, K 120 -> 128)"}
NCU_TENSOR_PIPE_TF32 = {"sm__pipe_tensor_cycles_active_pct_of_elapsed": 87.4, "file": "profiles/r02f_stack_tf32_ncu_full_summary.txt",
                        "note": "ncu --set full capture of one tdnn_stack_kernel<tf32> launch of the final code (471.2 us at 1.65 GHz)"}
# dram__bytes_read.sum + dram__bytes_write.sum of ONE tdnn_stack_kernel launch on this workload (ncu --set full; see profiles/README.md)
STACK_DRAM_BYTES = {"bf16": 186766336,   # 17.8 MB read + 169.0 MB written (final contents of the activation buffers)
                    "tf32": 713932032}   # 125.3 MB read + 588.6 MB written: float32 activations of a band do not fit in L2
STACK_DRAM_SOURCE = {"bf16": "profiles/r02f_stack_ncu_full_summary.txt", "tf32": "profiles/r02f_stack_tf32_ncu_full_summary.txt"}


def flops_per_utt(t):
    return sum(f * (t - l) for f, l in zip(FLOPS_L, LOST)) + SEG6_FLOPS


def tdnn_flops(n_utts, frames):
    return n_utts * sum(f * (frames - l) for f, l in zip(FLOPS_L, LOST))


def bench_config(world):
    """The `config` object of BOTH arms (product and reference): it names the workload only."""
    return {"workload": WORKLOAD, "utterances_per_step": N_UTTS * world, "batch": BATCH, "frames": FRAMES,
            "global_batch": BATCH * world, "parallelism": f"utterance-sharded x{world}, no data-path collective",
            "l2": "inputs larger than L2: the device-resident leg cycles >= 160 MiB of distinct batches; two batches in flight"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples SM clock, board power and throttle reasons of one GPU through NVML while a timed region runs."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.samples, self.power, self.reasons, self.max_mhz, self._stop_evt = index, [], [], set(), None, threading.Event()
        self.period = period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample_once(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1e3)
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._stop_evt.is_set():
            self.sample_once()
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        return self.summary()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s),
                "power_w_max": round(max(self.power), 1) if self.power else None}


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path, all host threads, on the product arm's config: the real modules
    (main.XVectorModel.extract_x_vec) when the reference is importable (oracle.ref_loader: $XVEC_REF_DIR, /root/reference,
    baseline/_ref), else the oracle port of its ATen op sequence.  Each step is a bounded sample of the 1024-utterance step
    (whole 256-utterance batches), sized so that the run ends within a few minutes."""
    if rank != 0:
        return
    import torch
    from oracle import ref_loader, xvector_oracle as ox
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    sd = ox.make_state_dict(seed=0)
    kind, fn = "port", None
    if ref_loader.available():
        try:
            _, main = ref_loader.load()
            model = main.XVectorModel()
            model.load_state_dict({k: v for k, v in sd.items() if k in model.state_dict()}, strict=False)
            model = model.eval()
            kind = "reference"

            def fn(x):
                with torch.no_grad():
                    return model.extract_x_vec(x)
        except Exception:
            kind, fn = "port", None
    if fn is None:
        def fn(x):
            return ox.extract_x_vec_aten(sd, x, 6)
    g = torch.Generator().manual_seed(1234)
    x_all = torch.randn(N_UTTS, FRAMES, CEPS, generator=g)  # the product arm's step: 4 batches of 256
    t0 = time.perf_counter()
    fn(x_all[:BATCH])
    t_batch = time.perf_counter() - t0
    budget = 150.0
    n_b = BATCHES_PER_STEP
    while n_b > 1 and n_b * t_batch * (args.steps + args.warmup) > budget:
        n_b -= 1
    sub = BATCH
    while n_b == 1 and sub > 32 and sub / BATCH * t_batch * (args.steps + args.warmup) > budget:
        sub //= 2
    sample = n_b * BATCH if n_b > 1 or sub == BATCH else sub

    def step():
        for b in range(n_b):
            fn(x_all[b * BATCH: b * BATCH + (BATCH if sample >= BATCH else sample)])

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = sample * args.steps / dt
    line = {"impl": "reference", "metric": "x-vectors/sec", "value": v, "unit": "utt/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "frames_per_sec": v * FRAMES,
            "config": bench_config(world),
            "cpu_baseline": {"value": v, "unit": "utt/s", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": f"{sample} of the {N_UTTS} utterances of a step (batches of {min(sample, BATCH)}), rank 0 only, all host threads; "
                                       + ("the unmodified reference modules (main.XVectorModel.extract_x_vec, fp32 torch CPU)" if kind == "reference" else
                                          "oracle/xvector_oracle.extract_x_vec_aten (the reference's ATen op sequence, fp32 torch CPU)")},
            "e2e": {"value": v, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
def cpu_baseline_leg(budget_s=12.0):
    import torch
    from oracle import xvector_oracle as ox
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    sd = ox.make_state_dict(seed=0)
    x = ox.synth_mfcc(64, FRAMES, seed=1234)  # BASELINE.json configs[0]
    for _ in range(2):
        ox.extract_x_vec_aten(sd, x, 6)
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < 5 or (time.perf_counter() < t_end and len(times) < 50):
        t0 = time.perf_counter()
        ox.extract_x_vec_aten(sd, x, 6)
        times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return {"value": 64 / med, "unit": "utt/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"config c1 (64 x 300 x 24, batch 64), median of {len(times)} runs of oracle.extract_x_vec_aten (the reference's ATen op sequence, fp32 torch CPU)",
            "frames_per_sec": 64 * FRAMES / med, "gflops": 64 * flops_per_utt(FRAMES) / med / 1e9, "best_utt_s": 64 / times[0]}


def synthetic_model(xvec_b200, precision):
    """Random-init weights of the reference architecture (PyTorch default initialisers, as main.XVectorModel() gets them) with
    non-trivial eval-mode BatchNorm statistics (default-init BN is the identity and would make the BN fold free)."""
    import torch
    torch.manual_seed(0)
    model = xvec_b200.XVectorModel(precision=precision)
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for layer in model.time_context_layers:
            n = layer.norm.num_features
            layer.norm.running_mean.copy_(0.5 * torch.randn(n, generator=g))
            layer.norm.running_var.copy_(0.3 + 1.7 * torch.rand(n, generator=g))
            layer.norm.weight.copy_(1.0 + 0.5 * torch.randn(n, generator=g))
            layer.norm.bias.copy_(0.5 * torch.randn(n, generator=g))
    return model


def pin_rank_to_cores(local_rank, world):
    """One disjoint block of host cores per rank: eight Python ranks that each enqueue ~10 k launches and copies per second
    otherwise migrate across (and share) cores."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // max(world, 1))
        mine = cores[local_rank * per: (local_rank + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:
        return None


def measure_matmul_peak(torch, dtype, allow_tf32, secs):
    """cuBLAS dense peak the way MEASURED_PEAKS.json takes it: torch.matmul 8192^3, best of 10 (burst) and back to back for
    `secs` seconds (sustained, last half)."""
    n = 8192
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = allow_tf32
    try:
        a = torch.randn(n, n, device="cuda", dtype=dtype)
        b = torch.randn(n, n, device="cuda", dtype=dtype)
        c = torch.empty(n, n, device="cuda", dtype=dtype)
        for _ in range(2):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        time.sleep(0.3)
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        flop = 2.0 * n ** 3
        rates, t_beg = [], time.perf_counter()
        while time.perf_counter() < t_beg + secs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            rates.append((time.perf_counter() - t_beg, 10 * flop / (e0.elapsed_time(e1) / 1e3) / 1e12))
        tail = [r for t, r in rates if t > secs / 2]
        return {"burst": flop / (best / 1e3) / 1e12, "sustained": sum(tail) / max(len(tail), 1)}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


class Arm:
    """One precision of the product on one rank: model, device-resident and pinned host inputs, the timed legs."""

    def __init__(self, torch, xvec_b200, precision, dev, rank, x_host, x_dev, n_res):
        self.torch, self.xb, self.precision, self.dev = torch, xvec_b200, precision, dev
        self.model = synthetic_model(xvec_b200, precision).to(dev).eval()
        self.x_host, self.x_dev, self.n_res = x_host, x_dev, n_res
        self.lengths = [FRAMES] * BATCH
        self.n_inflight = int(os.environ.get("XVEC_BENCH_INFLIGHT", "2"))  # batches in flight: the tail of one overlaps the next
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(self.n_inflight)]
        self.hx = None

    def batch(self, i):
        with self.torch.cuda.stream(self.streams[i % self.n_inflight]):
            return self.model.extract_x_vec_flat(self.x_dev[i % self.n_res], self.lengths, slot=i % self.n_inflight)

    def device_leg(self, n_batches, barrier):
        """n_batches batches, two in flight, one CUDA-event bracket; returns device milliseconds.  The x-vectors of the last
        step's batches stay in self.last_step."""
        torch = self.torch
        e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream()
        self.last_step = []
        barrier()
        e_beg.record(cur)
        for st in self.streams:
            st.wait_event(e_beg)
        for i in range(n_batches):
            y = self.batch(i)
            if i >= n_batches - BATCHES_PER_STEP:
                self.last_step.append(y)
        for st in self.streams:
            cur.wait_stream(st)
        e_end.record(cur)
        barrier()
        return e_beg.elapsed_time(e_end)

    def e2e_leg(self, n_batches, barrier, n_slots=6):
        """n_batches batches through HostExtractor.submit/result; returns (wall ms between barriers, checksum, enqueue us/batch)."""
        if self.hx is None:
            self.hx = self.xb.HostExtractor(self.model, n_slots=n_slots)
            for i in range(2 * n_slots):
                self.hx.result(self.hx.submit(self.x_host[i % BATCHES_PER_STEP], self.lengths))
        hx = self.hx
        barrier()
        hx.h2d_bytes = hx.d2h_bytes = 0
        t0 = time.perf_counter()
        tickets, checksum, t_enq = [], 0.0, 0.0
        for i in range(n_batches):
            t1 = time.perf_counter()
            tickets.append(hx.submit(self.x_host[i % BATCHES_PER_STEP], self.lengths))
            t_enq += time.perf_counter() - t1
            if len(tickets) == n_slots:
                checksum += float(hx.result(tickets.pop(0))[0, 0])
        while tickets:
            checksum += float(hx.result(tickets.pop(0))[0, 0])
        barrier()
        return (time.perf_counter() - t0) * 1e3, checksum, t_enq / n_batches * 1e6

    def stack_launch_times(self, local_rank):
        """CUDA-event time of the tdnn_stack_kernel launch (incl. its 5 KB control-block memset) in two regimes:
        burst = 30 launches from an idle (cool, unthrottled) GPU; sustained = back to back for >= 1.2 s, average of the second half."""
        torch = self.torch
        from xvec_b200 import ops
        m = self.model
        lay = m._layout_for(self.lengths)
        sc = m._scratch_for(0)
        sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
        pipe = m._pipeline()
        part = sc.part[: lay.n_slots]

        def launch(it):
            ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], m._frames_for(self.x_dev[it % self.n_res], pipe), sc.act[0], sc.act[1], lay.row_utt,
                           lay.blk_slot_base, part, sc.ctrl)

        for it in range(3):
            launch(it)
        torch.cuda.synchronize()
        time.sleep(0.7)  # let the board cool down to its idle clocks / power
        smp = ClockSampler(local_rank)
        evs = []
        for it in range(30):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch(it)
            e1.record()
            evs.append((e0, e1))
        smp.sample_once()
        torch.cuda.synchronize()
        smp.sample_once()
        burst_ms = sum(a.elapsed_time(b) for a, b in evs[2:]) / (len(evs) - 2)
        burst_clk = smp.summary()
        # sustained
        smp = ClockSampler(local_rank)
        smp.start()
        chunks, t_beg, it = [], time.perf_counter(), 0
        while time.perf_counter() < t_beg + 1.3:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(50):
                launch(it)
                it += 1
            e1.record()
            chunks.append((time.perf_counter() - t_beg, e0, e1))
            if len(chunks) > 8:
                chunks[-8][1].synchronize()  # bound the launch queue
        torch.cuda.synchronize()
        total_s = time.perf_counter() - t_beg
        sus_clk = smp.stop()
        tail = [a.elapsed_time(b) / 50 for t, a, b in chunks if t > 0.55 * total_s]
        sus_ms = sum(tail) / max(len(tail), 1)
        return burst_ms, burst_clk, sus_ms, sus_clk, it, total_s


def roofline_object(precision, burst_ms, burst_clk, sus_ms, sus_clk, n_launch, total_s, peak_burst, peak_sus, peak_source, regime):
    fl = tdnn_flops(BATCH, FRAMES)
    b_ach, s_ach = fl / (burst_ms / 1e3) / 1e12, fl / (sus_ms / 1e3) / 1e12
    burst = {"achieved": b_ach, "peak": peak_burst, "frac": b_ach / peak_burst, "ms_per_launch": burst_ms, "clocks": burst_clk,
             "timing": "CUDA events around each of 28 launches issued back to back from an idle GPU (0.7 s pause before), averaged"}
    sus = {"achieved": s_ach, "peak": peak_sus, "frac": s_ach / peak_sus, "ms_per_launch": sus_ms, "clocks": sus_clk,
           "timing": f"{n_launch} launches back to back for {total_s:.2f} s, CUDA events around groups of 50, average of the second half"}
    pick = burst if regime == "burst" else sus
    return {"kernel": "tdnn_stack_kernel (1 launch per batch: all tiles of TDNN1-5 from one work queue; TDNN5 epilogue = pooling partials)",
            "bound": "tensor", "achieved": pick["achieved"], "peak": pick["peak"], "unit": "TFLOP/s", "frac": pick["frac"],
            "regime": regime, "regime_note": "frac/achieved/peak repeat the regime the K-step `value` leg of this run was in "
                                             "(burst unless its timed region saw sw_power_cap for most of its length)",
            "traffic": STACK_DRAM_BYTES.get(precision), "traffic_source": STACK_DRAM_SOURCE.get(precision),
            "algorithmic_flops_per_launch": fl, "peak_source": peak_source, "burst": burst, "sustained": sus,
            "ncu": NCU_TENSOR_PIPE if precision == "bf16" else NCU_TENSOR_PIPE_TF32}


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import xvec_b200  # the product; nothing under oracle/ is imported on this arm except by cpu_baseline_leg()

    cores = pin_rank_to_cores(local_rank, world)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def min_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return t.tolist()

    g = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(N_UTTS, FRAMES, CEPS, generator=g).reshape(BATCHES_PER_STEP, BATCH * FRAMES, CEPS).pin_memory()
    # device-resident inputs: the 1024-utterance set replicated (with a per-copy scale) to n_res distinct batches so that the
    # inputs cycled through the timed region (n_res x 7.4 MB) are larger than the 126 MB L2
    n_res = max(BATCHES_PER_STEP, -(-(160 << 20) // (BATCH * FRAMES * CEPS * 4)))
    x_dev = torch.empty((n_res, BATCH * FRAMES, CEPS), dtype=torch.float32, device=dev)
    for i in range(n_res):
        x_dev[i].copy_(x_host[i % BATCHES_PER_STEP])
        x_dev[i].mul_(1.0 + 0.01 * (i // BATCHES_PER_STEP))
    warm = max(args.warmup, 3)
    peaks = load_peaks()
    steps_b = args.steps * BATCHES_PER_STEP

    def run_arm(precision):
        arm = Arm(torch, xvec_b200, precision, dev, rank, x_host, x_dev, n_res)
        for i in range(warm * BATCHES_PER_STEP):
            arm.batch(i)
        sampler = ClockSampler(local_rank)
        sampler.start()
        dev_ms = arm.device_leg(steps_b, barrier)
        clocks_value = sampler.stop()
        xvectors = torch.cat(arm.last_step).cpu().numpy() if args.dump_outputs else None
        sampler = ClockSampler(local_rank)
        sampler.start()
        e2e_ms, checksum, enq_us = arm.e2e_leg(steps_b, barrier)
        clocks_e2e = sampler.stop()
        h2d, d2h = arm.hx.h2d_bytes // args.steps, arm.hx.d2h_bytes // args.steps
        # long legs (~0.6 s each in bf16): the power-capped regime and the host side under sustained load
        sampler = ClockSampler(local_rank)
        sampler.start()
        long_dev_ms = arm.device_leg(LONG_BATCHES, barrier)
        long_e2e_ms, _, long_enq_us = arm.e2e_leg(LONG_BATCHES, barrier)
        clocks_long = sampler.stop()
        dev_ms, e2e_ms, long_dev_ms, long_e2e_ms = max_over_ranks([dev_ms, e2e_ms, long_dev_ms, long_e2e_ms])
        return arm, {"dev_ms": dev_ms, "e2e_ms": e2e_ms, "checksum": checksum, "enq_us": enq_us, "h2d": h2d, "d2h": d2h, "clocks_value": clocks_value,
                     "clocks_e2e": clocks_e2e, "long_dev_ms": long_dev_ms, "long_e2e_ms": long_e2e_ms, "long_enq_us": long_enq_us,
                     "clocks_long": clocks_long, "xvectors": xvectors}

    def arm_numbers(r):
        utts = N_UTTS * args.steps * world
        long_utts = BATCH * LONG_BATCHES * world
        return {"value": utts / (r["dev_ms"] / 1e3), "e2e": utts / (r["e2e_ms"] / 1e3), "long_value": long_utts / (r["long_dev_ms"] / 1e3),
                "long_e2e": long_utts / (r["long_e2e_ms"] / 1e3)}

    primary = args.dtype
    arm, res = run_arm(primary)
    num = arm_numbers(res)

    # ---- host-side probes, all ranks at once: H2D bandwidth of the step's input copies alone; NCCL-free
    barrier()
    st = torch.cuda.Stream(device=dev)
    reps, t0 = 0, time.perf_counter()
    with torch.cuda.stream(st):
        while time.perf_counter() - t0 < 0.25:
            for b in range(BATCHES_PER_STEP):
                x_dev[b].copy_(x_host[b], non_blocking=True)
            st.synchronize()
            reps += 1
    h2d_gbs = reps * BATCHES_PER_STEP * x_host[0].numel() * 4 / (time.perf_counter() - t0) / 1e9
    barrier()
    h2d_min, = min_over_ranks([h2d_gbs])
    h2d_max, = max_over_ranks([h2d_gbs])

    # ---- roofline of the dominant kernel, both regimes (rank 0 reports; every rank runs it so that the ranks stay in step)
    burst_ms, burst_clk, sus_ms, sus_clk, n_launch, total_s = arm.stack_launch_times(local_rank)
    layer_ms = instrumented_layer_times(arm.model, x_dev, arm.lengths, n_res, iters=10) if rank == 0 else None
    barrier()

    tf32_obj = None
    other = "tf32" if primary == "bf16" else "bf16"
    if not args.no_second_dtype:
        arm2, res2 = run_arm(other)
        num2 = arm_numbers(res2)
        b2, bc2, s2, sc2, nl2, ts2 = arm2.stack_launch_times(local_rank)
        barrier()
    tf32_peak = None
    if rank == 0 and (primary == "tf32" or not args.no_second_dtype):
        tf32_peak = measure_matmul_peak(torch, torch.float32, True, 2.0)
    barrier()

    def peaks_for(precision):
        if precision == "bf16":
            return peaks["bf16_tflops"], peaks["bf16_tflops_sustained"], f"{peaks['source']}: bf16_tflops (burst) / bf16_tflops_sustained"
        return tf32_peak["burst"], tf32_peak["sustained"], ("measured in this run like MEASURED_PEAKS.json does bf16: torch.matmul float32 8192^3 with "
                                                            "allow_tf32 (cuBLAS TF32), best of 10 (burst) / second half of 2 s back to back (sustained)")

    def regime_of(clk):
        return "sustained" if "sw_power_cap" in (clk.get("reasons") or []) and (clk.get("sm_mhz") or 1e9) < 0.9 * (clk.get("sm_max_mhz") or 1) else "burst"

    # ---- c5: the sharded workload (every rank takes part)
    c5 = None if args.no_c5 else run_c5(args, torch, dist, xvec_b200, arm.model, dev, rank, world, barrier, max_over_ranks, min_over_ranks)

    if rank == 0:
        pb, ps, psrc = peaks_for(primary)
        per_layer = {k: {"ms": round(v, 5)} for k, v in layer_ms.items()}
        for i in range(5):
            fl = BATCH * FLOPS_L[i] * (FRAMES - LOST[i])
            per_layer[f"tdnn{i + 1}"]["tflops"] = round(fl / (layer_ms[f"tdnn{i + 1}"] / 1e3) / 1e12, 2)
        line = {
            "metric": "x-vectors/sec", "value": num["value"], "unit": "utt/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": res["dev_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": primary, "data": "synthetic", "frames_per_sec": num["value"] * FRAMES,
            "config": bench_config(world),
            "e2e": {"value": num["e2e"], "unit": "utt/s", "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"],
                    "api": "HostExtractor.submit/result (pinned host MFCCs in, pinned host x-vectors out, 6 slots / streams)",
                    "frames_per_sec": num["e2e"] * FRAMES, "checksum": res["checksum"], "clocks": res["clocks_e2e"]},
            "gpu_launches": steps_b * LAUNCHES_PER_BATCH,
            "gpu_launches_note": f"{LAUNCHES_PER_BATCH} kernels per batch (tdnn_stack_kernel, pool_finalize_kernel, fc_small_kernel) x {BATCHES_PER_STEP} batches per step, per GPU",
            "clocks": res["clocks_value"],
            "timed_region_ms": {"value": res["dev_ms"], "e2e": res["e2e_ms"]},
            "long": {"batches": LONG_BATCHES, "value": num["long_value"], "e2e": num["long_e2e"], "unit": "utt/s",
                     "region_ms": {"value": res["long_dev_ms"], "e2e": res["long_e2e_ms"]}, "clocks": res["clocks_long"],
                     "note": "same legs over 2048 batches per GPU (>= 0.5 s): the regime a whole extraction job runs in (1000 W cap active)"},
            "host": {"h2d_gbs_per_rank_all_ranks_copying": {"min": h2d_min, "max": h2d_max},
                     "h2d_gbs_needed_by_e2e_per_rank": num["long_e2e"] / world * FRAMES * CEPS * 4 / 1e9,
                     "enqueue_us_per_batch": {"K_step_leg": res["enq_us"], "long_leg": res["long_enq_us"]},
                     "cpu_affinity_rank0": cores, "host_cores": os.cpu_count()},
            "roofline": roofline_object(primary, burst_ms, burst_clk, sus_ms, sus_clk, n_launch, total_s, pb, ps, psrc, regime_of(res["clocks_value"])),
            # for comparison only: the same layers as one tdnn_gemm_kernel launch each (segment6 here is the tcgen05 split-K GEMM)
            "per_layer_launches": per_layer,
        }
        if not args.no_second_dtype:
            pb2, ps2, psrc2 = peaks_for(other)
            line[other] = {"value": num2["value"], "e2e": {"value": num2["e2e"], "unit": "utt/s", "h2d_bytes_per_step": res2["h2d"],
                                                           "d2h_bytes_per_step": res2["d2h"], "checksum": res2["checksum"]},
                           "unit": "utt/s", "ms_per_step": res2["dev_ms"] / args.steps, "steps": args.steps, "clocks": res2["clocks_value"],
                           "long": {"value": num2["long_value"], "e2e": num2["long_e2e"], "clocks": res2["clocks_long"]},
                           "roofline": roofline_object(other, b2, bc2, s2, sc2, nl2, ts2, pb2, ps2, psrc2, regime_of(res2["clocks_value"])),
                           "note": ("fp32 storage + TF32 tensor-core math in every layer: the mode that meets the fp32 parity bound (1e-3 of the norm)"
                                    if other == "tf32" else "bf16 activations / weights, TDNN1 in TF32 on the fp32 MFCCs")}
        if tf32_peak is not None:
            line["tf32_cublas_peak_tflops"] = tf32_peak
        if c5 is not None:
            line["c5"] = c5
        if world == 1:
            line["roofline_pool"] = pooling_roofline(arm.model, dev, peaks)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_leg()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {f"xvectors_{primary}": res["xvectors"]})
            if not args.no_second_dtype:
                dump_outputs(args.dump_outputs, {f"xvectors_{other}": res2["xvectors"]})
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ c5: sharded set + trials
C5_N, C5_TRIALS, C5_SPK = 4874, 37_720, 40


def c5_lengths():
    import numpy as np
    return np.random.default_rng(3).integers(400, 2001, C5_N).astype(np.int64)  # 4-20 s at 100 frames/s


def c5_fill(torch, flat, idx, lengths):
    """Synthetic MFCCs of utterances idx (in that order) into the flat pinned tensor: unit noise around a per-speaker offset
    (speaker = utterance index mod 40) plus a per-utterance session offset of similar size, so that the trial scores overlap
    (a non-trivial EER); utterance i depends on i only, so every sharding sees the same data."""
    import numpy as np
    spk = (0.12 * np.random.default_rng(99).standard_normal((C5_SPK, CEPS))).astype(np.float32)
    out = flat.numpy()
    row = 0
    for i in idx:
        t = int(lengths[i])
        seg = out[row:row + t]
        rng = np.random.default_rng(100_000 + int(i))
        sess = (0.10 * rng.standard_normal(CEPS)).astype(np.float32)
        rng.standard_normal((t, CEPS), dtype=np.float32, out=seg)
        seg += spk[int(i) % C5_SPK] + sess
        row += t


def c5_trials():
    import numpy as np
    rng = np.random.default_rng(4)
    half = C5_TRIALS // 2
    members = [np.arange(s, C5_N, C5_SPK) for s in range(C5_SPK)]
    s = rng.integers(0, C5_SPK, half)
    e_t = np.asarray([rng.choice(members[k]) for k in s])
    t_t = np.asarray([rng.choice(members[k][members[k] != e]) for k, e in zip(s, e_t)])
    s1 = rng.integers(0, C5_SPK, half)
    s2 = (s1 + rng.integers(1, C5_SPK, half)) % C5_SPK
    e_n = np.asarray([rng.choice(members[k]) for k in s1])
    t_n = np.asarray([rng.choice(members[k]) for k in s2])
    enrol = np.concatenate([e_t, e_n]).astype(np.int32)
    test = np.concatenate([t_t, t_n]).astype(np.int32)
    target = np.concatenate([np.ones(half, bool), np.zeros(half, bool)])
    perm = rng.permutation(C5_TRIALS)
    return enrol[perm], test[perm], target[perm]


def run_c5(args, torch, dist, xvec_b200, model, dev, rank, world, barrier, max_over_ranks, min_over_ranks):
    import numpy as np
    from xvec_b200 import ops, scoring, sharding
    lengths = c5_lengths()
    # whole batches are the unit of sharding: which utterances share a batch does not depend on the number of GPUs, so the
    # x-vectors (and everything derived from them) are bit-identical for N = 1, 2, 4, 8
    parts, batch_sizes = sharding.shard_batches(lengths, world, target_frames=args.c5_batch_frames)
    mine = parts[rank]
    rows = int(lengths[mine].sum())
    flat = torch.empty((rows, CEPS), dtype=torch.float32).pin_memory()
    c5_fill(torch, flat, mine, lengths)
    enrol, test, target = c5_trials()
    en, te = torch.from_numpy(enrol).to(dev), torch.from_numpy(test).to(dev)
    hx = xvec_b200.HostExtractor(model, n_slots=6)
    gather = sharding.RowGather(parts, C5_N, 512, dev)
    scores_host = torch.empty(C5_TRIALS, dtype=torch.float32).pin_memory()
    emb_host = torch.empty((C5_N, 512), dtype=torch.float32).pin_memory()
    lens_mine = lengths[mine]

    def whole(instrument):
        """host MFCC shard -> H2D -> kernels -> all-gather -> trials -> host scores + embeddings (rank 0)."""
        t = [time.perf_counter()]
        hx.extract_flat(flat, lens_mine, to_host=False, batch_sizes=batch_sizes[rank], out_dev=gather.local_view)
        if instrument:
            torch.cuda.synchronize()
            t.append(time.perf_counter())
        full = gather()
        if instrument:
            torch.cuda.synchronize()
            t.append(time.perf_counter())
        if rank == 0:
            sc = ops.cosine_trials(full, en, te, center=True)
            if instrument:
                torch.cuda.synchronize()
                t.append(time.perf_counter())
            scores_host.copy_(sc, non_blocking=True)
            emb_host.copy_(full, non_blocking=True)
        torch.cuda.synchronize()
        t.append(time.perf_counter())
        return t

    whole(False)
    whole(False)  # warm-up: layouts, scratch, NCCL channels
    walls = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        whole(False)
        barrier()
        walls.append(max_over_ranks([(time.perf_counter() - t0) * 1e3])[0])
    barrier()
    t = whole(True)
    barrier()
    ph = [(b - a) * 1e3 for a, b in zip(t, t[1:])]
    extract_ms, gather_ms = max_over_ranks([ph[0], ph[1]])
    # the two halves of the extract phase, each alone: H2D of the shard; kernels on a device-resident copy of the shard
    x_res = torch.empty((rows, CEPS), dtype=torch.float32, device=dev)
    barrier()
    t0 = time.perf_counter()
    x_res.copy_(flat, non_blocking=True)
    torch.cuda.synchronize()
    h2d_ms = (time.perf_counter() - t0) * 1e3
    ends = np.cumsum(lens_mine)
    plan, lo = [], 0
    for b in batch_sizes[rank]:
        plan.append((lo, lo + b, int(ends[lo - 1]) if lo else 0, int(ends[lo + b - 1])))
        lo += b
    out_dev = torch.empty((len(mine), 512), dtype=torch.float32, device=dev)
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def kernels_only():
        for k, (lo, hi, r0, r1) in enumerate(plan):
            with torch.cuda.stream(streams[k % 2]):
                model.extract_x_vec_flat(x_res[r0:r1], lens_mine[lo:hi], slot=k % 2, out=out_dev[lo:hi])
        torch.cuda.synchronize()

    kernels_only()
    barrier()
    t0 = time.perf_counter()
    kernels_only()
    kern_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    h2d_ms_max, kern_ms_max = max_over_ranks([h2d_ms, kern_ms])
    h2d_gbs_min, = min_over_ranks([rows * CEPS * 4 / (h2d_ms / 1e3) / 1e9])
    loads = np.asarray([int((lengths[p] - 14).sum()) for p in parts], dtype=np.float64)
    if rank != 0:
        return None
    s = scores_host.numpy().astype(np.float64)
    eer, thr0 = scoring.eer(s, target)
    # decision threshold: the middle of the widest score gap among the 40 gaps around the EER point, so that the decisions (and
    # their hash) do not hinge on a score that sits within rounding of the threshold
    ss = np.sort(s)
    k = int(np.searchsorted(ss, thr0))
    lo_k, hi_k = max(1, k - 20), min(len(ss) - 1, k + 20)
    gaps = ss[lo_k:hi_k + 1] - ss[lo_k - 1:hi_k]
    j = lo_k + int(np.argmax(gaps))
    thr, margin = 0.5 * (ss[j] + ss[j - 1]), 0.5 * (ss[j] - ss[j - 1])
    decisions = (s >= thr)
    wall = sorted(walls)[len(walls) // 2]
    total_frames = int(lengths.sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"c5_embeddings": emb_host.numpy(), "c5_scores": scores_host.numpy()})
    return {"workload": "c5: 4874 utterances of 4-20 s (5.86 M frames, 563 MB of fp32 MFCC) LPT-sharded by utterance over the GPUs, "
                        "x-vectors gathered on the devices, 37,720 centred-cosine trials scored on GPU 0, scores + embeddings to the host",
            "scaling": "strong", "dtype": model.precision, "n_gpus": world, "n_utts": C5_N, "frames": total_frames, "trials": C5_TRIALS,
            "e2e_utt_s": C5_N / (wall / 1e3), "e2e_frames_s": total_frames / (wall / 1e3), "wall_ms": wall, "wall_ms_runs": walls,
            "wall_definition": "barrier -> per-rank HostExtractor.extract_flat(pinned host shard, to_host=False) -> all_gather_into_tensor (NCCL) -> "
                               "xvec_cosine_trials -> D2H of scores and embeddings -> barrier; max over ranks, median of 3",
            "phase_ms": {"extract_h2d_plus_kernels": extract_ms, "gather_nccl_all_gather_plus_reorder": gather_ms,
                         "trials_rank0": ph[2] if len(ph) > 3 else None, "d2h_rank0": ph[-1],
                         "note": "one instrumented pass with a device synchronisation between phases; extract/gather are max over ranks"},
            "alone_ms": {"h2d_of_the_shard": h2d_ms_max, "kernels_on_device_resident_shard": kern_ms_max,
                         "h2d_gbs_per_rank_min": h2d_gbs_min,
                         "note": "the extract phase overlaps these two; whichever is larger bounds it (all ranks run them at the same time)"},
            "device_utt_s": C5_N / (kern_ms_max / 1e3), "device_tflops": tdnn_flops_ragged(lengths) / (kern_ms_max / 1e3) / 1e12,
            "batches_per_rank": len(plan), "batch_frames_target": args.c5_batch_frames,
            "sharding": "layout.balanced_batches: the set is cut into a multiple of 8 contiguous batches of equal frames (+- one utterance); "
                        "rank r takes batches r, r + N, ... — batch composition is independent of N",
            "shard_imbalance_max_over_mean": float(loads.max() / loads.mean()), "gather_bytes_total": C5_N * 512 * 4,
            "eer": eer, "threshold": thr, "threshold_margin": margin,
            "embeddings_sha1": hashlib.sha1(emb_host.numpy().tobytes()).hexdigest(),
            "scores_sha1": hashlib.sha1(scores_host.numpy().tobytes()).hexdigest(),
            "decisions_sha1": hashlib.sha1(np.packbits(decisions).tobytes()).hexdigest(),
            "scores_sum": float(s.sum()), "embeddings_abs_sum": float(np.abs(emb_host.numpy().astype(np.float64)).sum()),
            "identity_note": "the three sha1 are over the raw float32 bytes of all 4874 x 512 embeddings, of the 37,720 scores and over the "
                             "decision bits: identical for N = 1, 2, 4, 8 because batches, not utterances, are the unit of sharding"}


def dump_outputs(dirname, arrays):
    """<dirname>/<name>.npy in float32 for every array: the inputs are seeded, so two builds run with the same arguments can be
    compared output for output."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(a, dtype=np.float32))


def tdnn_flops_ragged(lengths):
    return float(sum(sum(f * (int(t) - l) for f, l in zip(FLOPS_L, LOST)) for t in lengths))


def instrumented_layer_times(model, x_dev, lengths, n_batches, iters):
    """CUDA-event time of every launch of one batch run ONE LAUNCH PER LAYER (the fallback path), averaged over `iters` batches."""
    import torch
    from xvec_b200 import ops
    names = ["tdnn1", "tdnn2", "tdnn3", "tdnn4", "tdnn5", "pool_finalize", "segment6"]
    acc = dict.fromkeys(names, 0.0)
    layers = list(model.time_context_layers)
    lay = model._layout_for(lengths)
    sc = model._scratch_for(0)
    sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
    part, pooled = sc.part[: lay.n_slots], sc.pooled[: lay.n_utts]
    pooled_lp = None if sc.pooled_lp is None else sc.pooled_lp[: lay.n_utts]
    stack, (scale5, shift5) = model._stack_params()
    pipe = model._pipeline()
    all_evs = []
    for it in range(iters + 2):  # no host sync inside: the launches queue up and run back to back on the device
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        h = model._frames_for(x_dev[it % n_batches], pipe)
        evs[0].record()
        for i, layer in enumerate(layers[:-1]):
            w, bias, offs = stack[i]
            h = ops.tdnn_layer_flat(h, w, layer.output_size, offs, bias, None, None, relu=True,
                                    out=sc.act[i & 1][: lay.rows, : layer.output_size], cin=layer.input_size)
            evs[i + 1].record()
        last = layers[-1]
        w, bias, offs = stack[-1]
        ops.tdnn_pool_fused(h, w, last.output_size, offs, bias, lay.row_utt, lay.blk_slot_base, part)
        evs[5].record()
        ops.pool_finalize(part, lay.utt_slot_start, lay.n_pool, last.output_size, scale5, shift5, out=pooled, out_lp=pooled_lp)
        evs[6].record()
        model._head(pooled, pooled_lp, 6)
        evs[7].record()
        all_evs.append(evs)
    torch.cuda.synchronize()
    for evs in all_evs[2:]:
        for k, name in enumerate(names):
            acc[name] += evs[k].elapsed_time(evs[k + 1])
    return {k: v / iters for k, v in acc.items()}


def pooling_roofline(model, dev, peaks):
    """Standalone statistics pooling (XVectorModel.stat_pool) on a long-form activation larger than L2: HBM roofline."""
    import torch
    b, t, p = 64, 5986, 1500                      # 64 of the 256 long-form (60 s) utterances of config c4: 2.3 GB fp32
    a = torch.randn(b, t, p, device=dev)
    for _ in range(3):
        model.stat_pool(a)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
    for e0, e1 in evs:
        e0.record()
        model.stat_pool(a)
        e1.record()
    torch.cuda.synchronize()
    ms = sorted(e0.elapsed_time(e1) for e0, e1 in evs)[len(evs) // 2]
    nbytes = b * t * p * 4 + b * 2 * p * 4
    gbs = nbytes / (ms / 1e3) / 1e9
    del a
    return {"kernel": "stats_pool_partial_kernel + pool_finalize_kernel (standalone stat_pool, 64 x 5986 x 1500 fp32)", "bound": "hbm",
            "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
            "traffic": 2448198720,  # dram__bytes_read + write of stats_pool_partial_kernel per launch (2.437 GB + 11.6 MB), profiles/r02_pool_tf32_ncu_full_summary.txt
            "algorithmic_bytes": nbytes, "ms": ms, "peak_source": f"{peaks['source']} hbm_gbs"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)  # 400 batches, ~0.12 s per leg; the `long` legs cover the power-capped regime
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "tf32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--c5-batch-frames", type=int, default=49152)
    ap.add_argument("--no-second-dtype", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's x-vectors of the last timed step (xvectors_<dtype>.npy, one row per utterance, for each precision run) and the c5 "
                         "embeddings and trial scores (c5_embeddings.npy, c5_scores.npy) to DIR as float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run, one rank per GPU
        import subprocess
        port = 29500 + (os.getpid() % 2000)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
