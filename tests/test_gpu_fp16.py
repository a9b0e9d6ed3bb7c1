"""precision="fp16" on a B200: float16 activations and weights on the kind::f16 tensor pipe, held to the TF32 bound of the
suite (max-abs error per row <= 1e-3 * ||ref||, cosine >= 0.9999) against the goldens of the unmodified reference and the
CPU oracle, plus the kernel entry points it adds, bit-equality of the one-launch stack with the per-layer launches, the
BatchNorm fold and its float16 range guard."""

import numpy as np
import pytest
import torch

from oracle import xvector_oracle as ox

pytestmark = pytest.mark.gpu

TOL = 1e-3      # max-abs error relative to the norm of the reference row (the TF32 bound)
MIN_COS = 0.9999


@pytest.fixture(scope="module")
def xb():
    import xvec_b200
    assert xvec_b200._lib.load().xvec_device_check() == 0, xvec_b200._lib.load().xvec_last_error()
    return xvec_b200


def _model(xb, sd, precision="fp16", layer=6):
    m = xb.XVectorModel(x_vec_extract_layer=layer, precision=precision)
    assert not m.load_state_dict(sd, strict=True).missing_keys
    return m.cuda().eval()


def _parity(got, ref, tol=TOL):
    got = np.asarray(got.detach().float().cpu() if torch.is_tensor(got) else got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert got.shape == ref.shape and np.isfinite(got).all()
    rel = np.abs(got - ref).max(1) / np.linalg.norm(ref, axis=1)
    cos = (got * ref).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(ref, axis=1))
    assert rel.max() < tol, rel.max()
    assert cos.min() > MIN_COS, cos.min()
    return rel.max(), cos.min()


# ------------------------------------------------------------------------------------------------ model level
@pytest.mark.parametrize("tag", ["b4_t299", "b8_t300", "b3_t16"])
def test_extract_matches_reference_golden(xb, golden, state_dict, tag):
    b, t, seed = golden[tag + "_shape_seed"].tolist()
    x = ox.synth_mfcc(b, t, seed=seed).cuda()
    for layer, key in ((6, "_l6"), (7, "_l7"), (3, "_l3")):
        _parity(_model(xb, state_dict, layer=layer).extract_x_vec(x), golden[tag + key])
    m = _model(xb, state_dict)
    _parity(m(x), golden[tag + "_fwd"])
    out = m.test_step((x.double(), torch.arange(b), [f"id{i}" for i in range(b)]))
    assert torch.equal(out[0][0], m.extract_x_vec(x)) and out[0][2][0] == "id0"
    assert xb._lib.load().xvec_watchdog_code() == 0


def test_layer_activations_match_reference_golden(xb, golden, state_dict):
    """TdnnLayer on float16 input computes in float16 (no upcast); layer 1 reads the float32 frames (TF32), as in the model."""
    m = _model(xb, state_dict)
    h = ox.synth_mfcc(2, 40, seed=21).cuda()
    layers = list(m.time_context_layers)
    h1 = layers[0](h)
    hs, cur = [h1], h1.half()
    for layer in layers[1:]:
        cur = layer(cur.contiguous())
        assert cur.dtype == torch.float16
        hs.append(cur)
    for i, a in enumerate(hs):
        ref = golden[f"act_l{i + 1}"]
        assert tuple(a.shape) == ref.shape
        got = a.float().cpu().numpy().reshape(-1, ref.shape[-1])
        r = ref.reshape(-1, ref.shape[-1])
        rel = np.abs(got - r).max(1) / np.linalg.norm(r, axis=1)
        assert rel.max() < 2e-3, (i, rel.max())  # the tf32 bound of the bf16 / tf32 activation test


def test_single_pooled_frame_is_nan_like_reference(xb, golden, state_dict):
    b, t, seed = golden["b2_t15_shape_seed"].tolist()
    got = _model(xb, state_dict).extract_x_vec(ox.synth_mfcc(b, t, seed=seed).cuda())
    assert torch.isnan(got).all() and np.isnan(golden["b2_t15_l6"]).all()


def test_trial_decisions_identical(xb, state_dict):
    """Centred-cosine trial decisions of the fp16 embeddings == those of the float64 oracle embeddings at the oracle's EER
    threshold, with the score error inside the oracle's decision margin."""
    n, nspk = 240, 24
    lens = ox.synth_lengths(n, 100, 400, seed=3)
    utts = ox.synth_speaker_utts(lens, nspk, seed=55)
    ref = ox.extract_ragged_t(state_dict, utts, 6).numpy()
    enrol, test, target = ox.synth_trials(n, 6000, n_speakers=nspk, seed=4)
    s_ref = ox.cosine_scores_np(ref, enrol, test, center=True)
    eer, thr, margin = ox.eer_threshold_np(s_ref, target)
    m = _model(xb, state_dict)
    xv = m.extract_x_vec_flat(torch.cat(utts).cuda(), lens)
    _parity(xv, ref)
    s = xb.ops.cosine_trials(xv, torch.from_numpy(enrol).int().cuda(), torch.from_numpy(test).int().cuda(), center=True).cpu().numpy()
    assert np.abs(s - s_ref).max() < margin, (np.abs(s - s_ref).max(), margin)
    assert np.array_equal(s >= thr, s_ref >= thr)


def _small_var_state_dict(stride, dead=False):
    """running_var = 1e-6 on every `stride`-th channel of every TDNN layer: folded BatchNorm scales of about 300.  dead=True makes
    those channels what such a variance comes from in a trained model: rows that never leave ReLU's zero, running_mean 0."""
    sd = ox.make_state_dict(seed=0, randomize_bn=True)
    for i in range(5):
        p = f"time_context_layers.{i}."
        sd[p + "norm.running_var"][::stride] = 1e-6
        if dead:
            sd[p + "linear.weight"][::stride] = 0.0
            sd[p + "linear.bias"][::stride] = -1.0
            sd[p + "norm.running_mean"][::stride] = 0.0
    return sd


def _fp16_stored_max(sd, x):
    """Largest |value| the fp16 path stores in float16 for x_vec_extract_layer 6, taken from the reference's own fp64 forward: the
    ReLU outputs of TDNN1-4 (TDNN5's output is pooled in float32 and never stored) and the pooled statistics after TDNN5's
    BatchNorm, which segment6 reads."""
    h, top = x.double(), 0.0
    for i, ctx in enumerate(ox.LAYER_CONTEXTS):
        p = f"time_context_layers.{i}."
        y = torch.clamp_min(ox.unfold_t(h, ctx) @ sd[p + "linear.weight"].double().t() + sd[p + "linear.bias"].double(), 0.0)
        if i < 4:
            top = max(top, float(y.abs().max()))
        g, b, mu, var = (sd[p + "norm." + k].double() for k in ("weight", "bias", "running_mean", "running_var"))
        h = (y - mu) / torch.sqrt(var + 1e-5) * g + b
    return max(top, float(torch.cat((h.mean(1), h.std(1)), 1).abs().max()))


@pytest.mark.parametrize("stride,dead", [(512, False), (128, True)])
def test_small_batchnorm_variance_fits_fp16(xb, stride, dead):
    """running_var = 1e-6 on some channels of every layer: the folded weights grow by ~300 and still fit float16, and so does every
    value the reference itself produces where fp16 stores it (one moving channel in 512: up to ~1.3e4; dead channels: no growth);
    parity then holds at the TF32 bound."""
    sd = _small_var_state_dict(stride, dead)
    x = ox.synth_mfcc(8, 300, seed=5)
    assert _fp16_stored_max(sd, x) < 65504.0
    m = _model(xb, sd)
    stack, _ = m._stack_params()
    big = max(float(w.float().abs().max()) for w, _, _ in stack[1:])
    assert 5.0 < big < 65504.0, big  # the fold is visible and still fits float16
    _parity(m.extract_x_vec(x.cuda()), ox.extract_x_vec_t(sd, x, 6).numpy())


def test_activation_beyond_fp16_range_gives_non_finite_x_vectors(xb):
    """One channel in 16 of every layer with running_var = 1e-6: every folded weight still fits float16 (no ValueError), but the
    reference's own TDNN4 activations (and pooled statistics) exceed 65504.  fp16 then stores +inf and the x-vectors come out
    non-finite instead of as plausible wrong numbers; tf32 (float32 range) gives finite x-vectors for the same model."""
    sd = _small_var_state_dict(16)
    x = ox.synth_mfcc(8, 300, seed=5)
    assert _fp16_stored_max(sd, x) > 65504.0
    assert np.isfinite(ox.extract_x_vec_t(sd, x, 6).numpy()).all()
    assert not torch.isfinite(_model(xb, sd).extract_x_vec(x.cuda())).all()
    assert torch.isfinite(_model(xb, sd, "tf32").extract_x_vec(x.cuda())).all()


def test_fp16_range_guard(xb, state_dict):
    """A BatchNorm gamma whose fold puts a weight of the next layer beyond 65504 is refused when the fp16 model is prepared; the
    same model runs in tf32."""
    sd = {k: v.clone() for k, v in state_dict.items()}
    sd["time_context_layers.1.norm.weight"][0] = 1e7
    x = ox.synth_mfcc(2, 100, seed=6).cuda()
    with pytest.raises(ValueError, match="tf32"):
        _model(xb, sd).extract_x_vec(x)
    assert torch.isfinite(_model(xb, sd, "tf32").extract_x_vec(x)).all()
    lay = xb.TdnnLayer(input_size=64, output_size=256, context=[0]).cuda().eval()
    with torch.no_grad():
        lay.linear.weight[0, 0] = 7e4
    with pytest.raises(ValueError, match="tf32"):
        lay(torch.randn(1, 10, 64, device="cuda").half())


# ------------------------------------------------------------------------------------------------ stack kernel
@pytest.mark.parametrize("band", [0, 5, 7, 1000])
def test_stack_kernel_equals_per_layer_launches(xb, state_dict, band):
    """The fp16 one-launch stack kernel reproduces the fp16 per-layer launches bit for bit, for every band height."""
    from xvec_b200 import ops
    m = _model(xb, state_dict)
    lens = np.asarray([300] * 9 + [45, 16, 777, 1503, 15, 64, 2200])
    flat = torch.cat(ox.synth_ragged(lens, seed=7)).cuda()
    lay = m._layout_for(lens)
    pipe = m._pipeline()
    assert pipe["tdnn"][1].dtype == xb._lib.F16 and pipe["tdnn"][0].dtype == xb._lib.F32
    stack = pipe["keep"][0]
    layers = list(m.time_context_layers)
    sc = m._scratch_for(0)
    sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
    rows = flat.shape[0]
    h, acts = flat, []
    for i, layer in enumerate(layers[:-1]):
        w, bias, offs = stack[i]
        if i == 0 and pipe["window"] is not None:
            view = torch.as_strided(torch.cat([flat, flat.new_zeros(4, 24)]), (rows, 5 * 24), (24, 1))
            h = ops.tdnn_layer_flat(view, pipe["window"]["w"], 512, [0], bias, None, None, relu=True, out_dtype=torch.float16, cin=120)
        else:
            h = ops.tdnn_layer_flat(h, w, layer.output_size, offs, bias, None, None, relu=True, out_dtype=torch.float16, cin=layer.input_size)
        acts.append(h)
    w, bias, offs = stack[-1]
    part_ref = torch.zeros((lay.n_slots, 2, 1500), device="cuda")
    ops.tdnn_pool_fused(h, w, 1500, offs, bias, lay.row_utt, lay.blk_slot_base, part_ref)
    for _ in range(2):
        part = torch.zeros((lay.n_slots, 2, 1500), device="cuda")
        sc.act[0].zero_(); sc.act[1].zero_()
        ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], flat, sc.act[0], sc.act[1], lay.row_utt, lay.blk_slot_base, part, sc.ctrl, band=band)
        torch.cuda.synchronize()
        assert torch.equal(part, part_ref)
        assert torch.equal(sc.act[0][: lay.rows, :512], acts[2])
        assert torch.equal(sc.act[1][: lay.rows, :512], acts[3])
    assert xb._lib.load().xvec_watchdog_code() == 0


def test_stack_kernel_two_launches_in_flight(xb, state_dict):
    from xvec_b200 import ops
    m = _model(xb, state_dict)
    lens = np.random.default_rng(3).integers(15, 900, size=90)
    flat = torch.cat(ox.synth_ragged(lens, seed=8)).cuda()
    lay = m._layout_for(lens)
    pipe = m._pipeline()
    scs = [m._scratch_for(s) for s in range(2)]
    for sc in scs:
        sc.ensure(lay.rows, lay.n_slots, lay.n_utts)
    ref = torch.zeros((lay.n_slots, 2, 1500), device="cuda")
    ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], flat, scs[0].act[0], scs[0].act[1], lay.row_utt, lay.blk_slot_base, ref, scs[0].ctrl)
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(2)]
    for band in (0, 7):
        parts = [[torch.zeros_like(ref) for _ in range(3)] for _ in range(2)]
        for rep in range(3):
            for s in range(2):
                with torch.cuda.stream(streams[s]):
                    ops.tdnn_stack(pipe["tdnn"], pipe["n_tdnn"], flat, scs[s].act[0], scs[s].act[1], lay.row_utt, lay.blk_slot_base,
                                   parts[s][rep], scs[s].ctrl, band=band)
        torch.cuda.synchronize()
        assert all(torch.equal(pt, ref) for ps in parts for pt in ps)
    assert xb._lib.load().xvec_watchdog_code() == 0


# ------------------------------------------------------------------------------------------------ kernel level
def _ref_layer(x2d, W, b, offs, scale=None, shift=None, relu=True):
    rows, cin = x2d.shape
    xp = torch.cat([x2d.double(), torch.zeros(max(offs) + 1, cin, dtype=torch.float64)], 0)
    y = torch.cat([xp[o:o + rows] for o in offs], 1) @ W.double().t() + (b.double() if b is not None else 0)
    if relu:
        y = y.clamp_min(0)
    if scale is not None:
        y = y * scale.double() + shift.double()
    return y


def _rows_within(got, ref, tol=TOL):
    got, ref = got.double().cpu(), ref.cpu()
    assert torch.isfinite(got).all()
    err = (got - ref).abs().max(dim=1).values / ref.norm(dim=1).clamp_min(1e-6)
    assert err.max().item() < tol, err.max().item()


@pytest.mark.parametrize("rows,cin,n,offs", [(300, 512, 512, [0]), (1000, 512, 512, [0, 2, 4]), (777, 512, 512, [0, 3, 6]),
                                             (260, 512, 1500, [0]), (129, 40, 96, [0, 3, 6]), (64, 3000, 512, [0])])
def test_tdnn_layer_fp16_matches_fp64(xb, rows, cin, n, offs):
    """xvec_tdnn_layer with float16 operands against float64 on the same (float16-exact) operands: float16 and float32 output."""
    g = torch.Generator().manual_seed(rows * 7 + cin)
    x = torch.randn(rows, cin, generator=g).half()
    W = (torch.randn(n, cin * len(offs), generator=g) / (cin * len(offs)) ** 0.5)
    b = torch.randn(n, generator=g) * 0.1
    scale = 1 + 0.5 * torch.randn(n, generator=g)
    shift = 0.5 * torch.randn(n, generator=g)
    wp = xb.ops.pack_weight(W.cuda(), len(offs), cin, torch.float16)
    Wh = W.half().float()
    y = xb.ops.tdnn_layer_flat(x.cuda(), wp, n, offs, b.cuda(), scale.cuda(), shift.cuda(), relu=True)
    assert y.dtype == torch.float16 and y.shape == (rows, n)
    _rows_within(y, _ref_layer(x.float(), Wh, b, offs, scale, shift))
    y2 = xb.ops.tdnn_layer_flat(x.cuda(), wp, n, offs, b.cuda(), None, None, relu=True)  # ReLU folded into the convert
    _rows_within(y2, _ref_layer(x.float(), Wh, b, offs))
    y3 = xb.ops.tdnn_layer_flat(x.cuda(), wp, n, offs, b.cuda(), None, None, relu=False, out_dtype=torch.float32)
    _rows_within(y3, _ref_layer(x.float(), Wh, b, offs, relu=False), tol=1e-4)
    assert xb._lib.load().xvec_watchdog_code() == 0


@pytest.mark.parametrize("out_dtype", [torch.float16, torch.float32])
def test_tdnn_layer_fp16_split_k(xb, out_dtype):
    """Segment6 shape (256, 3000 -> 512): split-K over a workspace, the fixed-order reduce writes float16 or float32; the same
    result as the unsplit GEMM up to float32 summation order."""
    rows, cin, n = 256, 3000, 512
    g = torch.Generator().manual_seed(11)
    x = torch.randn(rows, cin, generator=g).half().cuda()
    W = torch.randn(n, cin, generator=g) / cin ** 0.5
    b = torch.randn(n, generator=g) * 0.1
    wp = xb.ops.pack_weight(W.cuda(), 1, cin, torch.float16)
    ws = xb.ops.splitk_workspace(rows, cin, 1, n, torch.float16, x.device)
    assert ws is not None
    for relu in (True, False):
        y = xb.ops.tdnn_layer_flat(x, wp, n, [0], b.cuda(), None, None, relu=relu, out_dtype=out_dtype, workspace=ws)
        ref = _ref_layer(x.float().cpu(), W.half().float(), b, [0], relu=relu)
        assert y.dtype == out_dtype
        _rows_within(y, ref, tol=TOL if out_dtype == torch.float16 else 1e-4)
        y_plain = xb.ops.tdnn_layer_flat(x, wp, n, [0], b.cuda(), None, None, relu=relu, out_dtype=out_dtype)
        _rows_within(y, y_plain.double().cpu(), tol=TOL if out_dtype == torch.float16 else 1e-4)


@pytest.mark.parametrize("rows,k,n,relu,out_dtype", [(256, 3000, 512, False, torch.float32), (77, 3000, 512, True, torch.float16),
                                                       (5, 512, 512, False, torch.float16), (300, 512, 1211, True, torch.float32)])
def test_linear_small_fp16(xb, rows, k, n, relu, out_dtype):
    """xvec_linear_small with float16 operands (mma.sync m16n8k16 f16) against float64 on the same operands."""
    g = torch.Generator().manual_seed(rows * 7 + k)
    x = torch.randn(rows, k, generator=g).half()
    W = (torch.randn(n, k, generator=g) / k ** 0.5).half()
    b = torch.randn(n, generator=g)
    ref = x.double() @ W.double().t() + b.double()
    if relu:
        ref = ref.clamp_min(0)
    got = xb.ops.linear_small(x.cuda(), W.cuda(), b.cuda(), relu=relu, out_dtype=out_dtype)
    assert got.dtype == out_dtype
    got = got.double().cpu()
    assert got.shape == ref.shape and torch.isfinite(got).all()
    tol = 1e-3 if out_dtype == torch.float16 else 2e-5
    assert ((got - ref).abs().max() / ref.abs().max()).item() < tol


def test_pack_weight_and_cast_fp16_are_round_to_nearest(xb):
    g = torch.Generator().manual_seed(2)
    x = torch.randn(100, 24, generator=g).cuda() * 100
    x[0, :3] = torch.tensor([float("nan"), 1e6, -70000.0])
    got, exp = xb.ops.cast(x, torch.float16), x.half()
    assert torch.equal(torch.isnan(got), torch.isnan(exp)) and torch.isnan(got[0, 0])
    ok = ~torch.isnan(exp)
    assert torch.equal(got[ok].view(torch.int16), exp[ok].view(torch.int16))  # inf beyond the range, no saturation
    for n, taps, cin in ((300, 3, 40), (512, 1, 3000), (96, 5, 24)):
        W = torch.randn(n, taps * cin, generator=g).cuda()
        wp = xb.ops.pack_weight(W, taps, cin, torch.float16)
        n_pad, k_pad = wp.shape
        tap_k = k_pad // taps
        # chunk-major layout [K chunk of 64][row][element] back to (n_pad, k_pad), then the zero padding removed
        dense = wp.reshape(-1).view(k_pad // 64, n_pad, 64).permute(1, 0, 2).reshape(n_pad, k_pad)
        exp = torch.zeros(n_pad, taps, tap_k, dtype=torch.float16, device="cuda")
        exp[:n, :, :cin] = W.view(n, taps, cin).half()
        assert torch.equal(dense.view(torch.int16), exp.view(n_pad, k_pad).view(torch.int16))


def test_stats_pool_partial_rejects_fp16(xb):
    """Standalone statistics pooling has no float16 input: the entry point rejects dtype 2 with XVEC_E_ARG."""
    lib = xb._lib.load()
    p = 64
    x = torch.zeros(128, p, dtype=torch.float16, device="cuda")
    row_start = torch.zeros(1, dtype=torch.int64, device="cuda")
    n_rows = torch.full((1,), 128, dtype=torch.int32, device="cuda")
    slot_start = torch.tensor([0, 1], dtype=torch.int32, device="cuda")
    part = torch.zeros(1, 2, p, device="cuda")
    rc = lib.xvec_stats_pool_partial(x.data_ptr(), xb._lib.F16, p, p, row_start.data_ptr(), n_rows.data_ptr(), slot_start.data_ptr(), 1, 1,
                                     part.data_ptr(), None, xb._lib.stream_ptr())
    assert rc == xb._lib.E_ARG, lib.xvec_last_error()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ full size
def test_c2_1024_fixed_length_batch256(xb, state_dict):
    x = ox.synth_mfcc(1024, 300, seed=1234)
    m = _model(xb, state_dict)
    out = torch.cat([m.extract_x_vec(x[i:i + 256].cuda()).clone() for i in range(0, 1024, 256)]).cpu().numpy()
    sel = np.random.default_rng(0).choice(1024, 48, replace=False)
    _parity(out[sel], ox.extract_x_vec_t(state_dict, x[sel], 6).numpy())
    perm = torch.from_numpy(np.random.default_rng(1).permutation(1024)[:256])
    again = m.extract_x_vec(x[perm].cuda()).cpu().numpy()
    assert np.abs(again - out[perm.numpy()]).max() < 1e-3 * np.abs(out).max()


def test_c3_ragged_4096_bucketed(xb, state_dict):
    lens = ox.synth_lengths(4096, 100, 2000, seed=2)
    utts = ox.synth_ragged(lens, seed=31)
    m = _model(xb, state_dict)
    hx = xb.HostExtractor(m)
    out = hx.extract_all(utts, max_frames=1 << 17)
    assert out.shape == (4096, 512) and np.isfinite(out).all()
    sel = np.random.default_rng(2).choice(4096, 24, replace=False)
    _parity(out[sel], ox.extract_ragged_t(state_dict, [utts[i] for i in sel], 6).numpy())
    out2 = hx.extract_all(utts, max_frames=90_000, max_utts=300)
    assert np.abs(out2 - out).max() < 1e-3 * np.abs(out).max()


def test_c4_long_form_256x6000(xb, state_dict):
    x = ox.synth_mfcc(256, 6000, seed=77)
    m = _model(xb, state_dict)
    out = torch.cat([m.extract_x_vec(x[i:i + 64].cuda()).clone() for i in range(0, 256, 64)]).cpu().numpy()
    sel = np.asarray([0, 101, 255])
    _parity(out[sel], ox.extract_x_vec_t(state_dict, x[sel], 6).numpy())
    assert np.isfinite(out).all()


def test_edge_shapes_many_tiny_and_one_huge_utterance(xb, state_dict):
    m = _model(xb, state_dict)
    lens = np.concatenate([np.full(1500, 16), np.full(700, 15), ox.synth_lengths(800, 16, 40, seed=11)])
    np.random.default_rng(12).shuffle(lens)
    utts = ox.synth_ragged(lens, seed=13)
    out = m.extract_x_vec_flat(torch.cat(utts).cuda(), lens).cpu().numpy()
    one_frame = lens == 15
    assert np.isnan(out[one_frame]).all() and np.isfinite(out[~one_frame]).all()
    sel = np.nonzero(~one_frame)[0][:: 97]
    _parity(out[sel], ox.extract_ragged_t(state_dict, [utts[i] for i in sel], 6).numpy())
    huge = ox.synth_mfcc(1, 60_000, seed=14)
    _parity(m.extract_x_vec(huge.cuda()), ox.extract_x_vec_t(state_dict, huge, 6).numpy())
    assert xb._lib.load().xvec_watchdog_code() == 0
