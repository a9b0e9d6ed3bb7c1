"""Model-level parity on a B200 through the reference's module surface: TdnnLayer.forward, XVectorModel.extract_x_vec /
forward / stat_pool / test_step against the CPU oracle and the committed golden vectors of the unmodified reference."""
import numpy as np
import pytest
import torch

from oracle import xvector_oracle as ox

pytestmark = pytest.mark.gpu

TOL_TF32 = 1e-3       # max-abs error relative to the norm of the reference embedding (north_star)
MIN_COS_BF16 = 0.9999


def _model(xb, sd, precision, layer=6):
    m = xb.XVectorModel(x_vec_extract_layer=layer, precision=precision)
    assert not m.load_state_dict(sd, strict=True).missing_keys
    return m.cuda().eval()


def _assert_parity(got, ref, precision):
    got = np.asarray(got.detach().float().cpu(), np.float64)
    ref = np.asarray(ref, np.float64)
    assert got.shape == ref.shape and np.isfinite(got).all()
    rel = np.abs(got - ref).max(1) / np.linalg.norm(ref, axis=1)
    cos = (got * ref).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(ref, axis=1))
    if precision == "tf32":
        assert rel.max() < TOL_TF32, rel.max()
    assert cos.min() > MIN_COS_BF16, cos.min()
    return rel.max(), cos.min()


@pytest.fixture(scope="module")
def xb():
    import xvec_b200
    return xvec_b200


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("tag", ["b4_t299", "b8_t300", "b3_t16"])
def test_extract_matches_reference_golden(xb, golden, state_dict, precision, tag):
    b, t, seed = golden[tag + "_shape_seed"].tolist()
    x = ox.synth_mfcc(b, t, seed=seed).cuda()
    for layer, key in ((6, "_l6"), (7, "_l7"), (3, "_l3")):
        m = _model(xb, state_dict, precision, layer)
        _assert_parity(m.extract_x_vec(x), golden[tag + key], precision)
    m = _model(xb, state_dict, precision)
    _assert_parity(m(x), golden[tag + "_fwd"], precision)
    out = m.test_step((x.double(), torch.arange(b), [f"id{i}" for i in range(b)]))
    assert torch.equal(out[0][0], m.extract_x_vec(x)) and out[0][2][0] == "id0"


def test_single_pooled_frame_is_nan_like_reference(xb, golden, state_dict):
    b, t, seed = golden["b2_t15_shape_seed"].tolist()
    got = _model(xb, state_dict, "tf32").extract_x_vec(ox.synth_mfcc(b, t, seed=seed).cuda())
    assert torch.isnan(got).all() and np.isnan(golden["b2_t15_l6"]).all()
    with pytest.raises(ValueError):
        _model(xb, state_dict, "tf32").extract_x_vec(torch.randn(2, 14, 24, device="cuda"))


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_layer_activations_match_reference_golden(xb, golden, state_dict, precision):
    m = _model(xb, state_dict, precision)
    h = ox.synth_mfcc(2, 40, seed=21).cuda()
    if precision == "bf16":
        h1 = m.time_context_layers[0](h)           # fp32 in (TF32 math)
        hs = [h1]
        cur = h1.bfloat16()
        for layer in list(m.time_context_layers)[1:]:
            cur = layer(cur.contiguous())
            hs.append(cur)
    else:
        hs, cur = [], h
        for layer in m.time_context_layers:
            cur = layer(cur.contiguous())
            hs.append(cur)
    for i, a in enumerate(hs):
        ref = golden[f"act_l{i + 1}"]
        assert tuple(a.shape) == ref.shape
        got = a.float().cpu().numpy().reshape(-1, ref.shape[-1])
        r = ref.reshape(-1, ref.shape[-1])
        rel = np.abs(got - r).max(1) / np.linalg.norm(r, axis=1)
        assert rel.max() < (2e-3 if precision == "tf32" else 3e-2), (i, rel.max())


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_ragged_matches_per_utterance_reference(xb, golden, state_dict, precision):
    lens = golden["ragged_lengths"]
    utts = ox.synth_ragged(lens, seed=77)
    m = _model(xb, state_dict, precision)
    got = m.extract_x_vec_flat(torch.cat(utts).cuda(), lens)
    _assert_parity(got, golden["ragged_l6"], precision)
    # permuting the utterances permutes the embeddings bit-for-bit-tolerantly (no cross-utterance leakage)
    perm = np.random.default_rng(0).permutation(len(lens))
    got_p = m.extract_x_vec_flat(torch.cat([utts[i] for i in perm]).cuda(), lens[perm])
    assert torch.allclose(got_p, got[perm], atol=1e-5 if precision == "tf32" else 5e-3)


def test_layer_without_bn_matches_reference_golden(xb, golden):
    lay = xb.TdnnLayer(input_size=40, output_size=96, context=[-3, 0, 3], batch_norm=False)
    with torch.no_grad():
        lay.linear.weight.copy_(torch.from_numpy(golden["layer_nobn_w"]))
        lay.linear.bias.copy_(torch.from_numpy(golden["layer_nobn_b"]))
    lay = lay.cuda().eval()
    y = lay(ox.synth_mfcc(3, 50, 40, seed=9).cuda())
    ref = golden["layer_nobn_y"]
    assert tuple(y.shape) == ref.shape == (3, 44, 96)
    assert np.abs(y.cpu().numpy() - ref).max() < 5e-3
    # parameters changed in place -> packed weights are rebuilt
    with torch.no_grad():
        lay.linear.weight.mul_(2.0)
        lay.linear.bias.mul_(2.0)
    assert np.abs(lay(ox.synth_mfcc(3, 50, 40, seed=9).cuda()).cpu().numpy() - 2 * ref).max() < 1e-2


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_config1_batch64_against_oracle(xb, state_dict, precision):
    """BASELINE.json config 1 (64 x 300 x 24, batch 64) — oracle computed here on the host cores."""
    x = ox.synth_mfcc(64, 300, seed=1234)
    ref = ox.extract_x_vec_t(state_dict, x, 6).numpy()
    m = _model(xb, state_dict, precision)
    rel, cos = _assert_parity(m.extract_x_vec(x.cuda()), ref, precision)
    # bitwise reproducible from run to run
    assert torch.equal(m.extract_x_vec(x.cuda()), m.extract_x_vec(x.cuda()))


def test_trial_decisions_identical(xb, state_dict):
    """Centred-cosine trial decisions from GPU embeddings == decisions from oracle embeddings at the oracle's EER
    threshold; the score perturbation must stay inside the oracle's decision margin."""
    n, nspk = 240, 24
    lens = ox.synth_lengths(n, 100, 400, seed=3)
    utts = ox.synth_speaker_utts(lens, nspk, seed=55)
    ref = ox.extract_ragged_t(state_dict, utts, 6).numpy()
    enrol, test, target = ox.synth_trials(n, 6000, n_speakers=nspk, seed=4)
    s_ref = ox.cosine_scores_np(ref, enrol, test, center=True)
    eer, thr, margin = ox.eer_threshold_np(s_ref, target)
    assert eer < 0.05 and margin > 1e-3
    for precision in ("tf32", "bf16"):
        m = _model(xb, state_dict, precision)
        xv = m.extract_x_vec_flat(torch.cat(utts).cuda(), lens)
        s = xb.ops.cosine_trials(xv, torch.from_numpy(enrol).int().cuda(), torch.from_numpy(test).int().cuda(), center=True).cpu().numpy()
        assert np.abs(s - s_ref).max() < margin, (precision, np.abs(s - s_ref).max(), margin)
        assert np.array_equal(s >= thr, s_ref >= thr)


def test_scoring_module_trial_file(xb, state_dict):
    """Product scoring path: trial file -> GPU centred cosine -> EER / minDCF, against fp64 numpy on the same embeddings."""
    from xvec_b200 import scoring
    n, nspk = 60, 6
    lens = ox.synth_lengths(n, 60, 200, seed=8)
    utts = ox.synth_speaker_utts(lens, nspk, seed=9)
    m = _model(xb, state_dict, "tf32")
    xv = m.extract_x_vec_flat(torch.cat(utts).cuda(), lens)
    ids = [f"id{10000 + i % nspk}/vid{i}/00001.wav" for i in range(n)]
    enrol, test, target = ox.synth_trials(n, 400, n_speakers=nspk, seed=2)
    lines = [f"{int(t)} {ids[e]} {ids[k]}\n" for e, k, t in zip(enrol, test, target)]
    s, tgt = scoring.score_trial_file(xv, ids, lines)
    assert np.array_equal(tgt, target)
    ref = ox.cosine_scores_np(xv.double().cpu().numpy(), enrol, test, center=True)
    assert np.abs(s - ref).max() < 1e-5
    e, thr = scoring.eer(s, tgt)
    d, _ = scoring.min_dcf(s, tgt)
    assert 0.0 <= d <= e + 1e-9 <= 0.5
    with pytest.raises(ValueError):
        scoring.score_trial_file(xv, ids, ["1 nope/a/b.wav " + ids[0] + "\n"])


def test_plda_trial_scores_and_decisions(xb):
    """PldaScorer (two split-TF32 GEMMs + xvec_plda_rowterm / xvec_plda_trials) against the float64 oracle on a synthetic model of
    the reference's size (x-vector dim 512, rank_f 150, plda_classifier.py:40): score error far inside the decision margin of
    the float64 scores at their EER threshold, identical decisions.  (Parity with SpeechBrain itself is unpinned.)"""
    from oracle import plda_oracle as po
    from xvec_b200 import scoring
    d, rank, nspk, per = 512, 150, 40, 12
    mean, F, S = po.synth_plda(d, rank, seed=5)
    F = 0.3 * F  # speaker variability small enough for a non-trivial EER (~3 %) and a narrow decision margin (~7e-3 of scores up to 48)
    rng = np.random.default_rng(6)
    spk = np.arange(nspk * per) % nspk  # the round-robin speaker assignment synth_trials assumes
    y = rng.standard_normal((nspk, rank))[spk]
    xs = (mean + y @ F.T + rng.standard_normal((nspk * per, d)) @ np.linalg.cholesky(S).T).astype(np.float32)
    enrol, test, target = ox.synth_trials(nspk * per, 8000, n_speakers=nspk, seed=4)
    ref = po.trial_scores(xs.astype(np.float64), enrol, test, mean, F, S, scaling_factor=1.0)
    eer, thr, margin = ox.eer_threshold_np(ref, target)
    assert 0.01 < eer < 0.06
    sc = scoring.PldaScorer(mean, F, S, scaling_factor=1.0)
    got = sc.score_trials(torch.from_numpy(xs).cuda(), enrol, test)
    err = np.abs(got - ref).max()
    assert err < 2e-5 * np.abs(ref).max(), (err, np.abs(ref).max())  # split-TF32 GEMMs + float32 dots
    assert err < margin, (err, margin)
    assert np.array_equal(got >= thr, ref >= thr)
    assert abs(scoring.eer(got, target)[0] - scoring.eer(ref, target)[0]) < 1e-9
    with pytest.raises(ValueError):
        sc.score_trials(torch.zeros(4, 100).cuda(), [0], [1])


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_strided_frame_matrix_is_not_read_as_windows(xb, state_dict, precision):
    """A (rows, 24) view of a wider buffer (what ops.mfcc(out=...) may hand over): TDNN1's window form is only valid on dense
    rows, so the model must not describe this input as overlapping 120-value windows (it would mix the padding columns into the
    taps).  Same bits as the dense copy, and parity with the oracle."""
    m = _model(xb, state_dict, precision)
    lens = np.asarray([120, 45, 300, 77])
    utts = ox.synth_ragged(lens, seed=91)
    dense = torch.cat(utts).cuda()
    wide = torch.full((dense.shape[0], 32), 1e6, device="cuda")  # poison in the padding columns
    wide[:, :24] = dense
    view = wide[:, :24]
    assert view.stride(0) == 32
    a = m.extract_x_vec_flat(view, lens).clone()
    b = m.extract_x_vec_flat(dense, lens).clone()
    assert torch.equal(a, b)
    pa, _ = m.pooled_stats_flat(view, lens)
    pa = pa.clone()
    pb, _ = m.pooled_stats_flat(dense, lens)
    assert torch.equal(pa, pb)
    ref = ox.extract_ragged_t(state_dict, utts, 6).numpy()
    got = a.cpu().numpy()
    cos = (got * ref).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(ref, axis=1))
    assert cos.min() > 0.9999


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_wide_context_falls_back_to_per_layer_launches(xb, precision):
    """A stack the one-launch kernel does not take (tap span 10 > XVEC_STACK_MAX_TAP_OFFSET = 8): xvec_extract_forward falls back
    to one launch per layer, and what it computes through extract_x_vec_flat and through pooled_stats_flat / forward must agree
    with a plain torch fp32 statement of the reference's op sequence (tdnn_layer.py:26-41, main.py:59-63, 81-94)."""
    torch.manual_seed(3)
    m = xb.XVectorModel(precision=precision)
    m.time_context_layers[1] = xb.TdnnLayer(input_size=512, output_size=512, context=[-5, 0, 5])
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        for layer in m.time_context_layers:
            layer.norm.running_mean.copy_(0.3 * torch.randn(layer.norm.num_features, generator=g))
            layer.norm.running_var.copy_(0.5 + torch.rand(layer.norm.num_features, generator=g))
    m = m.cuda().eval()
    assert not m._stack_kernel_ok() and m.lost_frames == 4 + 10 + 6
    x = torch.randn(3, 90, 24, generator=g)

    def ref_forward(x):
        h = x.double()
        for layer in m.time_context_layers:
            offs = xb.tap_offsets(layer.context)
            t_out = h.shape[1] - offs[-1]
            u = torch.cat([h[:, o:o + t_out] for o in offs], 2)
            h = torch.relu(u @ layer.linear.weight.double().cpu().t() + layer.linear.bias.double().cpu())
            n = layer.norm
            h = (h - n.running_mean.double().cpu()) / torch.sqrt(n.running_var.double().cpu() + n.eps) * n.weight.double().cpu() + n.bias.double().cpu()
        pooled = torch.cat((h.mean(1), h.std(1)), 1)
        return pooled, pooled @ m.segment_layer6.weight.double().cpu().t() + m.segment_layer6.bias.double().cpu()

    with torch.no_grad():
        pooled_ref, xv_ref = ref_forward(x)
    got = m.extract_x_vec(x.cuda()).double().cpu()
    pooled, _ = m.pooled_stats_flat(x.reshape(-1, 24).cuda(), [90] * 3)
    pooled = pooled.double().cpu()
    tol = 1e-3 if precision == "tf32" else 3e-2
    assert ((got - xv_ref).abs().max(1).values / xv_ref.norm(dim=1)).max().item() < tol
    assert ((pooled - pooled_ref).abs().max(1).values / pooled_ref.norm(dim=1)).max().item() < tol
    cos = torch.nn.functional.cosine_similarity(got, xv_ref, dim=1)
    assert cos.min().item() > 0.9999
    assert torch.isfinite(m.forward(x.cuda())).all()


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_other_tap_counts_run_in_the_stack_kernel(xb, precision):
    """The one-launch kernel specialises its MMA loop for the tap counts of the reference's stack (1 and 3; main.py:39-43) and keeps
    a generic loop for every other context get_time_context accepts (tdnn_layer.py:43-60).  A stack with a 2-tap layer
    ([-2, 2], extra/time_context_test.py:25), a 5-tap 512-channel layer and a 3-tap POOLED last layer stays on the stack kernel
    (tap spans <= 8) and must agree with a plain torch fp64 statement of the reference's op sequence."""
    torch.manual_seed(5)
    m = xb.XVectorModel(precision=precision)
    m.time_context_layers[1] = xb.TdnnLayer(input_size=512, output_size=512, context=[-2, 2])
    m.time_context_layers[2] = xb.TdnnLayer(input_size=512, output_size=512, context=[-2, -1, 0, 1, 2])
    m.time_context_layers[4] = xb.TdnnLayer(input_size=512, output_size=1500, context=[-1, 0, 1])
    g = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for layer in m.time_context_layers:
            layer.norm.running_mean.copy_(0.3 * torch.randn(layer.norm.num_features, generator=g))
            layer.norm.running_var.copy_(0.5 + torch.rand(layer.norm.num_features, generator=g))
    m = m.cuda().eval()
    assert m._stack_kernel_ok() and m.lost_frames == 4 + 4 + 4 + 0 + 2
    x = torch.randn(5, 150, 24, generator=g)

    def ref_forward(x):
        h = x.double()
        for layer in m.time_context_layers:
            offs = xb.tap_offsets(layer.context)
            t_out = h.shape[1] - offs[-1]
            u = torch.cat([h[:, o:o + t_out] for o in offs], 2)
            h = torch.relu(u @ layer.linear.weight.double().cpu().t() + layer.linear.bias.double().cpu())
            n = layer.norm
            h = (h - n.running_mean.double().cpu()) / torch.sqrt(n.running_var.double().cpu() + n.eps) * n.weight.double().cpu() + n.bias.double().cpu()
        pooled = torch.cat((h.mean(1), h.std(1)), 1)
        return pooled, pooled @ m.segment_layer6.weight.double().cpu().t() + m.segment_layer6.bias.double().cpu()

    with torch.no_grad():
        pooled_ref, xv_ref = ref_forward(x)
    got = m.extract_x_vec(x.cuda()).double().cpu()
    pooled, _ = m.pooled_stats_flat(x.reshape(-1, 24).cuda(), [150] * 5)
    pooled = pooled.double().cpu()
    tol = 1e-3 if precision == "tf32" else 3e-2
    assert ((got - xv_ref).abs().max(1).values / xv_ref.norm(dim=1)).max().item() < tol
    assert ((pooled - pooled_ref).abs().max(1).values / pooled_ref.norm(dim=1)).max().item() < tol
    cos = torch.nn.functional.cosine_similarity(got, xv_ref, dim=1)
    assert cos.min().item() > 0.9999
    assert xb._lib.load().xvec_watchdog_code() == 0
