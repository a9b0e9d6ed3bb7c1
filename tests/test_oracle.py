"""Pins oracle/xvector_oracle.py to the reference: known-answer fixtures and golden vectors produced by the
unmodified reference (tests/golden/make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import xvector_oracle as ox


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.linalg.norm(b, axis=-1).min(), 1e-30)


# ---------------------------------------------------------------- reference KATs (extra/time_context_test.py)
@pytest.mark.parametrize("name,shape,first", [("c5", (5, 11, 5), [1, 2, 3, 4, 5]), ("c2", (5, 11, 2), [1, 5]),
                                              ("c5d2", (5, 7, 5), [1, 3, 5, 7, 9]), ("c11", (5, 5, 11), list(range(1, 12)))])
def test_time_context_kat(kat, name, shape, first):
    got = ox.unfold_np(kat["x"], kat[name + "_ctx"].tolist())
    assert got.shape == shape                      # shapes listed in SURVEY §4
    assert got[0, 0].tolist() == first
    assert np.array_equal(got, kat[name])          # bit-exact against the reference's get_time_context + cat
    assert torch.equal(ox.unfold_t(torch.from_numpy(kat["x"]), kat[name + "_ctx"].tolist()), torch.from_numpy(kat[name]))


def test_time_context_docstring_example(kat):
    got = ox.unfold_np(kat["doc_x"], [-1, 0, 1])
    assert np.array_equal(got, kat["doc"])
    assert got[0].tolist() == [[1, 2, 3, 4, 5, 6], [3, 4, 5, 6, 7, 8], [5, 6, 7, 8, 9, 0]]
    assert ox.unfold_np(np.zeros((1, 100, 10)), [-1, 0, 1]).shape == (1, 98, 30)


def test_asymmetric_context_rejected():
    for ctx in ([-1, 0, 2], [0, 1, 2]):
        with pytest.raises(ValueError):
            ox.time_context_index(20, ctx)
    with pytest.raises(ValueError):
        ox.time_context_index(4, [-2, -1, 0, 1, 2])
    assert ox.time_context_index(5, [-2, -1, 0, 1, 2]).shape == (1, 5)


# ---------------------------------------------------------------- golden vectors from the unmodified reference
def test_weight_init_matches_reference(golden):
    assert ox.state_dict_digest(ox.make_state_dict(seed=0, randomize_bn=False)) == str(golden["default_init_digest"])
    assert ox.state_dict_digest(ox.make_state_dict(seed=0, randomize_bn=True)) == str(golden["state_digest"])


@pytest.mark.parametrize("tag", ["b4_t299", "b8_t300", "b3_t16"])
def test_extract_matches_golden(golden, state_dict, tag):
    b, t, seed = golden[tag + "_shape_seed"].tolist()
    x = ox.synth_mfcc(b, t, seed=seed)
    for layer, key in ((6, "_l6"), (7, "_l7"), (3, "_l3")):
        got = ox.extract_x_vec_t(state_dict, x, layer).numpy()
        assert got.shape == (b, 512)
        assert rel_err(got, golden[tag + key]) < 2e-6, (tag, layer)
    assert np.array_equal(golden[tag + "_l3"], golden[tag + "_l6"])     # "anything else behaves as 6"
    assert rel_err(ox.forward_t(state_dict, x).numpy(), golden[tag + "_fwd"]) < 2e-6
    # float64 truth agrees with the fp32 reference to fp32 rounding
    assert rel_err(ox.extract_x_vec_np(state_dict, x.numpy(), 6), golden[tag + "_l6"]) < 2e-5


def test_aten_sequence_port_matches_golden(golden, state_dict):
    """The operator-sequence port that bench.py times as the CPU baseline gives the reference's numbers."""
    b, t, seed = golden["b8_t300_shape_seed"].tolist()
    x = ox.synth_mfcc(b, t, seed=seed)
    for layer, key in ((6, "_l6"), (7, "_l7")):
        assert rel_err(ox.extract_x_vec_aten(state_dict, x, layer).numpy(), golden["b8_t300" + key]) < 2e-6


def test_single_pooled_frame_is_nan_like_reference(golden, state_dict):
    b, t, seed = golden["b2_t15_shape_seed"].tolist()
    got = ox.extract_x_vec_t(state_dict, ox.synth_mfcc(b, t, seed=seed), 6).numpy()
    assert np.isnan(golden["b2_t15_l6"]).all() and np.isnan(got).all()


def test_layer_activations_match_golden(golden, state_dict):
    h = ox.synth_mfcc(2, 40, seed=21)
    frames = [36, 32, 26, 26, 26]
    for i, ctx in enumerate(ox.LAYER_CONTEXTS):
        h = ox.tdnn_layer_t(h, state_dict[f"time_context_layers.{i}.linear.weight"],
                            state_dict[f"time_context_layers.{i}.linear.bias"], ctx, ox._bn_of(state_dict, i, ox._as_t))
        ref = golden[f"act_l{i + 1}"]
        assert h.shape[1] == frames[i] and h.shape == ref.shape
        assert np.abs(h.numpy() - ref).max() < 2e-5 * max(1.0, np.abs(ref).max())
    assert np.abs(ox.stat_pool_t(h).numpy() - golden["act_pool"]).max() < 2e-5
    assert np.abs(ox.stat_pool_np(h.numpy().astype(np.float64)) - golden["act_pool"]).max() < 2e-5


def test_ragged_matches_golden(golden, state_dict):
    lens = golden["ragged_lengths"]
    assert np.array_equal(lens, ox.synth_lengths(12, 16, 420, seed=2))
    utts = ox.synth_ragged(lens, seed=77)
    got = ox.extract_ragged_t(state_dict, utts, 6).numpy()
    assert rel_err(got, golden["ragged_l6"]) < 2e-6


def test_layer_without_bn_matches_golden(golden):
    x = ox.synth_mfcc(3, 50, 40, seed=9)
    y = ox.tdnn_layer_t(x, torch.from_numpy(golden["layer_nobn_w"]), torch.from_numpy(golden["layer_nobn_b"]), [-3, 0, 3], None)
    assert y.shape == (3, 44, 96)
    assert np.abs(y.numpy() - golden["layer_nobn_y"]).max() < 1e-5


# ---------------------------------------------------------------- whole-stack entry points against the stored reference outputs
def test_oracle_matches_stored_reference(golden, state_dict):
    """The reference's extract_x_vec at layer 7 and its stat_pool(time_context_layers(x)), as stored by make_golden.py, against
    the oracle's extract_x_vec_t and its whole-stack tdnn_stack_t + stat_pool_t."""
    b, t, seed = golden["b3_t16_shape_seed"].tolist()
    x = ox.synth_mfcc(b, t, seed=seed)
    assert rel_err(ox.extract_x_vec_t(state_dict, x, 7).numpy(), golden["b3_t16_l7"]) < 2e-6
    x = ox.synth_mfcc(2, 40, seed=21)
    assert np.abs(ox.stat_pool_t(ox.tdnn_stack_t(state_dict, x)).numpy() - golden["act_pool"]).max() < 2e-5


# ---------------------------------------------------------------- scoring helpers
def test_trials_and_eer_threshold():
    enrol, test, target = ox.synth_trials(200, 2000, n_speakers=10, seed=4)
    assert len(enrol) == 2000 and target.sum() == 1000
    spk = np.arange(200) % 10
    assert (spk[enrol[target]] == spk[test[target]]).all() and (spk[enrol[~target]] != spk[test[~target]]).all()
    rng = np.random.default_rng(0)
    xv = rng.standard_normal((10, 32))[spk] + 0.8 * rng.standard_normal((200, 32))
    s = ox.cosine_scores_np(xv, enrol, test)
    eer, thr, margin = ox.eer_threshold_np(s, target)
    assert 0 <= eer < 0.3 and margin > 0
    far = ((s >= thr) & ~target).sum() / (~target).sum()
    frr = ((s < thr) & target).sum() / target.sum()
    assert abs(far - frr) < 0.01 and abs(0.5 * (far + frr) - eer) < 1e-9


def test_flops_formula():
    assert abs(ox.flops_per_utt(300) / 1.5378e9 - 1) < 1e-3


def test_plda_fast_scoring_equals_model_definition():
    """oracle/plda_oracle.py restates the published fast PLDA scoring (parity with SpeechBrain unpinned).  What can be pinned:
    its score equals the log-likelihood ratio of the two-covariance model evaluated straight from the Gaussian densities,
    constant included, and the per-trial form equals the N x N matrix form."""
    from oracle import plda_oracle as po
    mean, F, S = po.synth_plda(32, 8, seed=1)
    rng = np.random.default_rng(0)
    x = rng.standard_normal((9, 32)) + mean
    sm = po.fast_plda_scoring(x[:4], x[4:], mean, F, S, scaling_factor=1.0)
    direct = np.array([[po.llr_direct(e, t, mean, F, S) for t in x[4:]] for e in x[:4]])
    assert np.abs(sm - direct).max() < 1e-10
    e, t = np.array([0, 1, 3, 2]), np.array([4, 8, 5, 5])
    assert np.abs(po.trial_scores(x, e, t, mean, F, S, 0.7) - 0.7 * sm[e, t - 4]).max() < 1e-12
    # same-speaker pairs of the generative model score higher than different-speaker pairs on average
    y = rng.standard_normal((200, 8))
    L = np.linalg.cholesky(S)
    a = mean + y @ F.T + rng.standard_normal((200, 32)) @ L.T
    b = mean + y @ F.T + rng.standard_normal((200, 32)) @ L.T
    same = po.trial_scores(np.vstack([a, b]), np.arange(200), 200 + np.arange(200), mean, F, S)
    diff = po.trial_scores(np.vstack([a, b]), np.arange(200), 200 + np.roll(np.arange(200), 1), mean, F, S)
    assert same.mean() > diff.mean() + 1.0


def test_mfcc_oracle_pieces_agree_with_torchaudio():
    """INDEPENDENT (not pinning) evidence for oracle/mfcc_oracle.py — python_speech_features itself is not available offline, so
    row f4 stays 'parity unpinned'.  torchaudio ships the same textbook pieces written by other people:
      * DCT-II (ortho): torchaudio.functional.create_dct == dct_matrix, to rounding;
      * sinusoidal lifter: torchaudio.compliance.kaldi._get_lifter_coeffs == lifter_weights, to rounding;
      * HTK mel scale + triangular filters: torchaudio places the triangle corners at exact frequencies, python_speech_features
        (and the oracle) on floor()ed FFT bins, so the banks cannot be equal — they must agree in centre frequency to one bin
        and overlap to > 0.9 (cosine between corresponding filters);
      * the whole chain with torchaudio's pieces substituted for the DCT and the lifter gives the oracle's MFCCs to 1e-5."""
    torchaudio = pytest.importorskip("torchaudio")
    import torchaudio.functional as AF
    from torchaudio.compliance import kaldi
    from oracle import mfcc_oracle as mo
    dct = AF.create_dct(mo.NUMCEP, mo.NFILT, norm="ortho").double().numpy().T          # (numcep, nfilt)
    assert np.abs(dct - mo.dct_matrix()).max() < 5e-6                                    # torchaudio builds a float32 table
    lift = kaldi._get_lifter_coeffs(mo.NUMCEP, float(mo.CEPLIFTER)).double().numpy()
    assert np.abs(lift - mo.lifter_weights()).max() < 1e-5
    fb_ta = AF.melscale_fbanks(mo.NFFT // 2 + 1, 0.0, mo.SAMPLE_RATE / 2.0, mo.NFILT, mo.SAMPLE_RATE, norm=None, mel_scale="htk").double().numpy().T
    fb = mo.filterbank()
    assert fb.shape == fb_ta.shape == (mo.NFILT, mo.NFFT // 2 + 1)
    assert np.abs(fb.argmax(1) - fb_ta.argmax(1)).max() <= 1                             # same centre bins (+- the floor)
    cos = (fb * fb_ta).sum(1) / (np.linalg.norm(fb, axis=1) * np.linalg.norm(fb_ta, axis=1))
    assert cos.min() > 0.9, cos.min()
    # mel scale itself: the filter edges in Hz are the HTK formula's
    edges_hz = mo.mel2hz(np.linspace(mo.hz2mel(0.0), mo.hz2mel(8000.0), mo.NFILT + 2))
    m_ta = 2595.0 * np.log10(1.0 + edges_hz / 700.0)
    assert np.abs(np.diff(m_ta) - np.diff(m_ta).mean()).max() < 1e-9                     # equally spaced on torchaudio's HTK mel axis
    # the chain with torchaudio's DCT / lifter substituted
    rng = np.random.default_rng(0)
    sig = rng.standard_normal(16000)
    ref = mo.mfcc_np(sig)
    y = np.append(sig[0], sig[1:] - mo.PREEMPH * sig[:-1])
    nf = mo.num_frames(len(y))
    padded = np.zeros((nf - 1) * mo.FRAME_STEP + mo.FRAME_LEN)
    padded[: len(y)] = y
    frames = padded[np.arange(mo.FRAME_LEN)[None, :] + mo.FRAME_STEP * np.arange(nf)[:, None]]
    pspec = np.abs(np.fft.rfft(frames, mo.NFFT)) ** 2 / mo.NFFT
    ceps = np.log(pspec @ fb.T) @ dct.T * lift[None, :]
    ceps[:, 0] = np.log(pspec.sum(1))
    assert np.abs(ceps - ref).max() < 1e-5 * np.abs(ref).max()
