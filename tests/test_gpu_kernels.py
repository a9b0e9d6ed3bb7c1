"""Kernel-level parity on a B200: every C-ABI entry point against the oracle / a plain torch fp32 statement of the op.

Tolerances (north_star): TF32 path max-abs error <= 1e-3 relative to the norm of the reference row;
bf16 path cosine >= 0.9999 per row.  Integer / layout logic is exact.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xb():
    import xvec_b200
    assert xvec_b200._lib.load().xvec_device_check() == 0, xvec_b200._lib.load().xvec_last_error()
    return xvec_b200


def _ref_layer(x2d, W, b, offs, scale=None, shift=None, relu=True):
    """fp64 statement on the flat matrix: y[r] = bn(relu(sum_j W_j x[r+off_j] + b)), rows past the end read zero."""
    rows, cin = x2d.shape
    xp = torch.cat([x2d.double(), torch.zeros(max(offs) + 1, cin, dtype=torch.float64)], 0)
    u = torch.cat([xp[o:o + rows] for o in offs], 1)
    y = u @ W.double().t() + (b.double() if b is not None else 0)
    if relu:
        y = y.clamp_min(0)
    if scale is not None:
        y = y * scale.double() + shift.double()
    return y


def _check(got, ref, dtype):
    got = got.double().cpu()
    ref = ref.cpu()
    assert torch.isfinite(got).all()
    if dtype == torch.float32:
        err = (got - ref).abs().max(dim=1).values / ref.norm(dim=1).clamp_min(1e-6)
        assert err.max().item() < 1e-3, err.max().item()
    else:
        cos = torch.nn.functional.cosine_similarity(got, ref, dim=1)
        assert cos.min().item() > 0.9999, cos.min().item()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows,cin,n,offs", [
    (300, 512, 512, [0]),            # plain k=1 GEMM (TDNN4)
    (1000, 512, 512, [0, 2, 4]),     # dilated taps (TDNN2)
    (777, 512, 512, [0, 3, 6]),      # TDNN3, ragged tile edge
    (515, 24, 512, [0, 1, 2, 3, 4]), # TDNN1: Cin smaller than one K chunk (zero-filled by TMA)
    (260, 512, 1500, [0]),           # TDNN5 shape, N not a multiple of the tile
    (129, 40, 96, [0, 3, 6]),        # odd sizes
    (64, 3000, 512, [0]),            # segment6: long K, few rows
])
def test_tdnn_layer_matches_reference(xb, dtype, rows, cin, n, offs):
    if dtype == torch.bfloat16 and cin % 8:
        pytest.skip("bf16 rows must be 16-byte aligned")
    g = torch.Generator().manual_seed(rows * 7 + cin)
    x = torch.randn(rows, cin, generator=g)
    W = torch.randn(n, cin * len(offs), generator=g) / (cin * len(offs)) ** 0.5
    b = torch.randn(n, generator=g) * 0.1
    scale = 1 + 0.5 * torch.randn(n, generator=g)
    shift = 0.5 * torch.randn(n, generator=g)
    xd = x.cuda().to(dtype)
    wp = xb.ops.pack_weight(W.cuda(), len(offs), cin, dtype)
    assert wp.shape == (-(-n // 256) * 256, len(offs) * (-(-cin // (32 if dtype == torch.float32 else 64))) * (32 if dtype == torch.float32 else 64))
    y = xb.ops.tdnn_layer_flat(xd, wp, n, offs, b.cuda(), scale.cuda(), shift.cuda(), relu=True)
    torch.cuda.synchronize()
    assert y.shape == (rows, n) and y.dtype == dtype
    ref = _ref_layer(xd.float().cpu(), W.to(dtype).float() if dtype == torch.bfloat16 else W, b, offs, scale, shift)
    _check(y, ref, dtype)
    # no relu / no bn / fp32 output from any input type
    y2 = xb.ops.tdnn_layer_flat(xd, wp, n, offs, b.cuda(), None, None, relu=False, out_dtype=torch.float32)
    ref2 = _ref_layer(xd.float().cpu(), W.to(dtype).float() if dtype == torch.bfloat16 else W, b, offs, relu=False)
    _check(y2, ref2, dtype)
    assert xb._lib.load().xvec_watchdog_code() == 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows,cin,n", [(256, 3000, 512), (100, 512, 512), (700, 3000, 96)])
def test_split_k_matches_reference(xb, dtype, rows, cin, n):
    """Few output tiles + long K (segment6/7): K is split over CTA pairs into a workspace, second pass applies the epilogue."""
    g = torch.Generator().manual_seed(rows + cin)
    x = torch.randn(rows, cin, generator=g).cuda().to(dtype)
    W = torch.randn(n, cin, generator=g) / cin ** 0.5
    b = torch.randn(n, generator=g) * 0.1
    wp = xb.ops.pack_weight(W.cuda(), 1, cin, dtype)
    ws = xb.ops.splitk_workspace(rows, cin, 1, n, dtype, "cuda")
    assert ws is not None
    Wr = W.to(dtype).float() if dtype == torch.bfloat16 else W
    for relu, out_dtype in ((False, torch.float32), (True, dtype)):
        y = xb.ops.tdnn_layer_flat(x, wp, n, [0], b.cuda(), None, None, relu=relu, out_dtype=out_dtype, workspace=ws)
        y0 = xb.ops.tdnn_layer_flat(x, wp, n, [0], b.cuda(), None, None, relu=relu, out_dtype=out_dtype)
        _check(y, _ref_layer(x.float().cpu(), Wr, b, [0], relu=relu), dtype)
        assert (y.float() - y0.float()).abs().max().item() < 2e-2 * y0.float().abs().max().item()
        assert torch.equal(y, xb.ops.tdnn_layer_flat(x, wp, n, [0], b.cuda(), None, None, relu=relu, out_dtype=out_dtype, workspace=ws))
    assert xb.ops.splitk_workspace(76800, 512, 3, 512, dtype, "cuda") is None   # big GEMMs never split


def test_tdnn_layer_many_tiles_exercises_pipeline_wraparound(xb):
    # > 148*2 tiles per CTA round and > 4 stages: phases of every barrier wrap several times
    rows, cin, n, offs = 148 * 128 * 3 + 77, 512, 512, [0, 2, 4]
    g = torch.Generator().manual_seed(3)
    x = torch.randn(rows, cin, generator=g).cuda().bfloat16()
    W = torch.randn(n, cin * 3, generator=g) / (cin * 3) ** 0.5
    wp = xb.ops.pack_weight(W.cuda(), 3, cin, torch.bfloat16)
    y = xb.ops.tdnn_layer_flat(x, wp, n, offs, None, None, None, relu=False, out_dtype=torch.float32)
    xp = torch.cat([x.float(), torch.zeros(8, cin, device="cuda")], 0)
    ref = torch.cat([xp[o:o + rows] for o in offs], 1) @ W.cuda().bfloat16().float().t()
    err = (y - ref).abs().max().item()
    assert err < 2e-2 * ref.abs().max().item(), err


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_stats_pool_standalone(xb, dtype):
    g = torch.Generator().manual_seed(5)
    lens = [1, 2, 17, 128, 129, 300, 1000]
    starts = np.concatenate(([0], np.cumsum(lens)[:-1]))
    x = (torch.randn(sum(lens), 1500, generator=g) + 0.7).cuda().to(dtype)
    out = xb.ops.stats_pool_ragged(x, starts, np.asarray(lens))
    for u, (s, l) in enumerate(zip(starts, lens)):
        seg = x[s:s + l].double()
        assert torch.allclose(out[u, :1500].double(), seg.mean(0), atol=2e-5, rtol=1e-5)
        if l > 1:
            assert torch.allclose(out[u, 1500:].double(), seg.std(0), atol=5e-5, rtol=1e-4)
        else:
            assert torch.isnan(out[u, 1500:]).all()   # torch.std of one frame is NaN (main.py:61)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_stats_pool_large_mean_small_std(xb, dtype):
    """|mean| >> std: a one-pass float32 sum of squares loses the variance (1e4 * 2^-24 per term against a variance of 1); the
    kernel sums x - (first row) instead.  torch.std (main.py:61) is two-pass, so the public stat_pool surface must hold 1e-4 here."""
    g = torch.Generator().manual_seed(6)
    x = (100.0 + torch.randn(7, 900, 1500, generator=g)).cuda().to(dtype)
    x[3] -= 250.0  # a negative mean as well
    m = xb.XVectorModel().cuda().eval()
    got = m.stat_pool(x).double()
    xd = x.double()
    ref = torch.cat((xd.mean(1), xd.std(1)), 1)
    assert torch.allclose(got[:, :1500], ref[:, :1500], rtol=1e-6, atol=1e-5)
    assert ((got[:, 1500:] - ref[:, 1500:]).abs() / ref[:, 1500:]).max().item() < 1e-4


def test_stat_pool_module_surface(xb, state_dict):
    m = xb.XVectorModel().cuda().eval()
    x = torch.randn(5, 61, 1500, device="cuda")
    ref = torch.cat((x.mean(1), x.std(1)), 1)
    assert torch.allclose(m.stat_pool(x), ref, atol=5e-5, rtol=1e-4)
    xs = x[:, :40]  # strided view like a TdnnLayer output
    assert torch.allclose(m.stat_pool(xs), torch.cat((xs.mean(1), xs.std(1)), 1), atol=5e-5, rtol=1e-4)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fused_tdnn5_pool_matches_unfused(xb, dtype):
    """TDNN5 + pooling fused (activation never stored) == TDNN5 store kernel + masked pooling, on a ragged batch
    whose utterance boundaries fall inside 32-row blocks and 128-row tiles."""
    lens = np.asarray([15, 16, 47, 300, 33, 129, 640, 20])
    lay = xb.build_layout(lens)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(lay.rows, 512, generator=g).cuda().to(dtype)
    W = torch.randn(1500, 512, generator=g) / 512 ** 0.5
    b = torch.randn(1500, generator=g) * 0.2
    scale = (1 + 0.5 * torch.randn(1500, generator=g)).cuda()
    shift = (0.5 * torch.randn(1500, generator=g)).cuda()
    wp = xb.ops.pack_weight(W.cuda(), 1, 512, dtype)
    part = torch.full((lay.n_slots, 2, 1500), float("nan"), device="cuda")
    xb.ops.tdnn_pool_fused(x, wp, 1500, [0], b.cuda(), torch.from_numpy(lay.row_utt).cuda(),
                           torch.from_numpy(lay.blk_slot_base).cuda(), part)
    assert torch.isfinite(part).all()       # every slot written exactly by the kernel
    pooled = xb.ops.pool_finalize(part, torch.from_numpy(lay.utt_slot_start).cuda(), torch.from_numpy(lay.n_pool).cuda(),
                                  1500, scale, shift)
    r = xb.ops.tdnn_layer_flat(x, wp, 1500, [0], b.cuda(), None, None, relu=True, out_dtype=torch.float32).double()
    z = r * scale.double() + shift.double()
    for u in range(len(lens)):
        seg = z[lay.starts[u]: lay.starts[u] + lay.n_pool[u]]
        assert torch.allclose(pooled[u, :1500].double(), seg.mean(0), atol=1e-4, rtol=1e-4), u
        if lay.n_pool[u] > 1:
            assert torch.allclose(pooled[u, 1500:].double(), seg.std(0), atol=2e-4, rtol=2e-4), u
        else:
            assert torch.isnan(pooled[u, 1500:]).all()
    # run-to-run bit reproducibility (fixed-order reduction, no atomics)
    part2 = torch.empty_like(part)
    xb.ops.tdnn_pool_fused(x, wp, 1500, [0], b.cuda(), torch.from_numpy(lay.row_utt).cuda(),
                           torch.from_numpy(lay.blk_slot_base).cuda(), part2)
    assert torch.equal(part, part2)


def test_cast_and_cosine(xb):
    g = torch.Generator().manual_seed(1)
    x = torch.randn(100, 24, generator=g).cuda()
    assert torch.equal(xb.ops.cast(x, torch.bfloat16), x.bfloat16())
    xv = torch.randn(50, 512, generator=g).cuda()
    e = torch.randint(0, 50, (1000,), generator=g).int().cuda()
    t = torch.randint(0, 50, (1000,), generator=g).int().cuda()
    ref = torch.nn.functional.cosine_similarity(xv[e.long()].double(), xv[t.long()].double(), dim=1)
    assert (xb.ops.cosine_trials(xv, e, t).double() - ref).abs().max().item() < 1e-5
    xc = xv.double() - xv.double().mean(0)
    refc = torch.nn.functional.cosine_similarity(xc[e.long()], xc[t.long()], dim=1)
    assert (xb.ops.cosine_trials(xv, e, t, center=True).double() - refc).abs().max().item() < 1e-5


def test_argument_errors(xb):
    x = torch.randn(64, 512, device="cuda")
    wp = xb.ops.pack_weight(torch.randn(512, 512, device="cuda"), 1, 512, torch.float32)
    with pytest.raises(ValueError):
        xb.ops.tdnn_layer_flat(x.cpu(), wp, 512, [0])              # no CPU path
    with pytest.raises(xb._lib.XvecError):
        xb.ops.tdnn_layer_flat(x, wp, 512, [0] * 9)                # too many taps
    with pytest.raises(xb._lib.XvecError):
        xb.ops.tdnn_layer_flat(x[:, 1:], wp, 511, [0], cin=511)    # misaligned rows
    with pytest.raises(ValueError):
        xb.TdnnLayer(24, 32, [-1, 0, 2]).cuda().eval()(torch.randn(1, 30, 24, device="cuda"))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "tf32"])
@pytest.mark.parametrize("band", [0, 5, 7, 1000])
def test_stack_kernel_equals_per_layer_launches(xb, state_dict, precision, band, monkeypatch):
    """xvec_tdnn_stack (one persistent launch, dynamic tile queue, per-tile dependency flags) must reproduce the per-layer
    launches bit for bit — same tiles, same K order, same epilogues — for every band height of the work-item order."""
    from xvec_b200 import ops
    from oracle import xvector_oracle as ox
    m = xb.XVectorModel(precision=precision)
    m.load_state_dict(state_dict)
    m = m.cuda().eval()
    lens = np.asarray([300] * 9 + [45, 16, 777, 1503, 15, 64, 2200])
    utts = ox.synth_ragged(lens, seed=7)
    flat = torch.cat(utts).cuda()
    lay = m._layout_for(lens)
    pipe = m._pipeline()
    stack = pipe["keep"][0]
    layers = list(m.time_context_layers)
    sc = m._scratch_for(0)
    sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
    xs, rows = flat, flat.shape[0]
    h = flat
    acts = []
    for i, layer in enumerate(layers[:-1]):
        w, bias, offs = stack[i]
        if i == 0 and pipe["window"] is not None:
            # TDNN1 in window form — one K = 120 GEMM over overlapping rows of the frames (windows past the end read as zero)
            view = torch.as_strided(torch.cat([xs, xs.new_zeros(4, 24)]), (rows, 5 * 24), (24, 1))  # storage must cover the nominal view
            h = ops.tdnn_layer_flat(view, pipe["window"]["w"], 512, [0], bias, None, None, relu=True, out_dtype=m.act_dtype, cin=120)
        else:
            h = ops.tdnn_layer_flat(h, w, layer.output_size, offs, bias, None, None, relu=True, out_dtype=m.act_dtype, cin=layer.input_size)
        acts.append(h)
    w, bias, offs = stack[-1]
    part_ref = torch.zeros((lay.n_slots, 2, 1500), device="cuda")
    ops.tdnn_pool_fused(h, w, 1500, offs, bias, lay.row_utt, lay.blk_slot_base, part_ref)
    for rep in range(3):  # repeated launches reuse (and re-zero) the same control block
        part = torch.zeros((lay.n_slots, 2, 1500), device="cuda")
        sc.act[0].zero_(); sc.act[1].zero_()
        ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], xs, sc.act[0], sc.act[1], lay.row_utt, lay.blk_slot_base, part, sc.ctrl, band=band)
        torch.cuda.synchronize()
        assert torch.equal(part, part_ref)
        # layer 3 / layer 4 outputs are what is left in the ping-pong buffers
        assert torch.equal(sc.act[0][: lay.rows, :512], acts[2])
        assert torch.equal(sc.act[1][: lay.rows, :512], acts[3])
    assert xb._lib.load().xvec_watchdog_code() == 0


def test_stack_kernel_two_launches_in_flight(xb, state_dict, monkeypatch):
    """Two tdnn_stack_kernel launches on two streams (separate scratch, dynamic tile queues) cannot starve or corrupt each other:
    every result equals the single-launch result bit for bit (tools/stack_stress.py is the long version)."""
    from xvec_b200 import ops
    from oracle import xvector_oracle as ox
    m = xb.XVectorModel(precision="bf16")
    m.load_state_dict(state_dict)
    m = m.cuda().eval()
    lens = np.random.default_rng(3).integers(15, 900, size=90)
    flat = torch.cat(ox.synth_ragged(lens, seed=8)).cuda()
    lay = m._layout_for(lens)
    pipe = m._pipeline()
    scs = [m._scratch_for(s) for s in range(2)]
    for sc in scs:
        sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
    xs = [(flat, flat.shape[0]) for _ in scs]
    ref = torch.zeros((lay.n_slots, 2, 1500), device="cuda")
    ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], xs[0][0], scs[0].act[0], scs[0].act[1], lay.row_utt, lay.blk_slot_base, ref, scs[0].ctrl)
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(2)]
    for band in (0, 7):
        parts = [[torch.zeros_like(ref) for _ in range(4)] for _ in range(2)]
        for rep in range(4):
            for s in range(2):
                with torch.cuda.stream(streams[s]):
                    ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], xs[s][0], scs[s].act[0], scs[s].act[1], lay.row_utt, lay.blk_slot_base,
                                   parts[s][rep], scs[s].ctrl, band=band)
        torch.cuda.synchronize()
        assert all(torch.equal(pt, ref) for ps in parts for pt in ps)
    assert xb._lib.load().xvec_watchdog_code() == 0


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("rows,k,n,relu,out_dtype", [(256, 3000, 512, False, torch.float32), (77, 3000, 512, True, torch.bfloat16),
                                                       (5, 512, 512, False, torch.float32), (300, 512, 1211, True, torch.float32),
                                                       (33, 40, 24, False, torch.float32)])
def test_linear_small_matches_reference(xb, dtype, rows, k, n, relu, out_dtype):
    """xvec_linear_small (mma.sync, 5 KiB smem — the segment layers next to a resident stack kernel) against float64: bf16
    operands are exact inputs (only fp32 accumulation order differs), float32 operands go through TF32 (1e-3 bound)."""
    g = torch.Generator().manual_seed(rows * 7 + k)
    x = (torch.randn(rows, k, generator=g)).to(dtype)
    W = (torch.randn(n, k, generator=g) / k ** 0.5).to(dtype)
    b = torch.randn(n, generator=g)
    ref = x.double() @ W.double().t() + b.double()
    if relu:
        ref = ref.clamp_min(0)
    got = xb.ops.linear_small(x.cuda(), W.cuda(), b.cuda(), relu=relu, out_dtype=out_dtype).double().cpu()
    assert got.shape == ref.shape and torch.isfinite(got).all()
    tol = 1e-2 if out_dtype == torch.bfloat16 else (2e-5 if dtype == torch.bfloat16 else 1e-3)
    assert ((got - ref).abs().max() / ref.abs().max()).item() < tol
    with pytest.raises(Exception):
        xb.ops.linear_small(x[:, :-3].contiguous().cuda(), W[:, :-3].contiguous().cuda())  # k not a multiple of 16 bytes


def test_watchdog_code_is_readable():
    """A protocol failure inside the stack kernel must leave a readable code.  The debug library (-DXVEC_DEBUG) can be told to skip
    the completion signalling (XVEC_STACK_DBG bit 2) with a short spin limit (bit 8) and a watchdog that reports without trapping
    (bit 16; a real trap is an Xid event and destroys the context): the dependency warps then give up with code 7.  The code is
    read back from the mapped host word — it used to live in a per-translation-unit __device__ variable that the reader, in
    another unit, never saw.  Child process: the parent has already loaded the product library."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dbg_lib = os.path.join(root, "speaker-recognition-x-vectors_b200", "libxvec_b200_debug.so")
    if not os.path.exists(dbg_lib):
        import importlib
        importlib.import_module("speaker-recognition-x-vectors_b200.build").build(debug=True)
    child = r"""
import sys, torch
sys.path.insert(0, %r)
import xvec_b200
lib = xvec_b200._lib.load()
m = xvec_b200.XVectorModel(precision="bf16").cuda().eval()
x = torch.randn(4, 200, 24, device="cuda")
assert lib.xvec_watchdog_code() == 0
m.extract_x_vec(x)
torch.cuda.synchronize()
code = lib.xvec_watchdog_code()
lib.xvec_watchdog_reset()
print("watchdog", code, "after reset", lib.xvec_watchdog_code(), flush=True)
""" % root
    env = dict(os.environ, XVEC_LIB=dbg_lib, XVEC_STACK_DBG="26")
    r = subprocess.run([sys.executable, "-c", child], env=env, capture_output=True, text=True, timeout=300)
    assert "watchdog 7 after reset 0" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])
    # ... and the same child with the switches off runs clean
    env = dict(os.environ, XVEC_LIB=dbg_lib, XVEC_STACK_DBG="0")
    r = subprocess.run([sys.executable, "-c", child], env=env, capture_output=True, text=True, timeout=300)
    assert "watchdog 0 after reset 0" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])
