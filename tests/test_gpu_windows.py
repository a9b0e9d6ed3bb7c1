"""Windowed extraction on a B200 (XVectorModel.extract_x_vec_windows, HostExtractor.extract_windows): one pass of the frame-level
stack over whole recordings, one x-vector per window.  A window's x-vector must be what the same frames cut out as an utterance
give: bitwise for windows = whole recordings (same layout), else within the batch-composition bounds of test_gpu_fullsize.py (the
fp32 summation order of the pooling follows where the rows sit in the 128-row blocks), and at the oracle bounds of `_parity`."""
import numpy as np
import pytest
import torch

from oracle import xvector_oracle as ox

pytestmark = pytest.mark.gpu

BOUND = {"tf32": 1e-4, "bf16": 5e-3, "fp16": 5e-3}  # max-abs / max|out|, batch composition (test_gpu_fullsize.py)
MAX_FRAMES = 1 << 17


@pytest.fixture(scope="module")
def xb():
    import xvec_b200
    return xvec_b200


def _model(xb, sd, precision, layer=6):
    m = xb.XVectorModel(precision=precision, x_vec_extract_layer=layer)
    m.load_state_dict(sd)
    return m.cuda().eval()


def _parity(got, ref, precision):
    """_parity of test_gpu_fullsize.py; fp16 is held to the TF32 bound (test_gpu_fp16.py)."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    rel = np.abs(got - ref).max(1) / np.linalg.norm(ref, axis=1)
    cos = (got * ref).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(ref, axis=1))
    assert np.isfinite(got).all()
    if precision in ("tf32", "fp16"):
        assert rel.max() < 1e-3, rel.max()
    assert cos.min() > 0.9999, cos.min()


def _slices(utts, w):
    return [utts[k][a:a + n] for k, a, n in w]


def _resliced(m, utts, w):
    """extract_x_vec_flat over the windows cut out as utterances, in batches of <= MAX_FRAMES frames."""
    pieces = _slices(utts, w)
    out, i = [], 0
    while i < len(pieces):
        j, frames = i, 0
        while j < len(pieces) and (j == i or frames + pieces[j].shape[0] <= MAX_FRAMES):
            frames += pieces[j].shape[0]
            j += 1
        batch = pieces[i:j]
        out.append(m.extract_x_vec_flat(torch.cat(batch).cuda(), [p.shape[0] for p in batch]).cpu())
        i = j
    return torch.cat(out).numpy()


def _arbitrary_windows(lengths, lost, seed):
    """Unsorted windows with duplicates, nested windows, the shortest windows with a std (n = lost + 2), shifts of 1-3 frames and
    windows touching both recording ends."""
    rng = np.random.default_rng(seed)
    out = []
    for k, t in enumerate(lengths):
        for _ in range(6):
            n = int(rng.integers(lost + 2, min(t, 700) + 1))
            out.append((k, int(rng.integers(0, t - n + 1)), n))
        k_, a, n = out[-1]
        out += [(k, a, n), (k, a + 1, n - 2), (k, a + n // 3, n // 3)] if n // 3 > lost + 1 else [(k, a, n)]   # duplicate, nested
        n = min(t, 150)
        a = int(rng.integers(0, t - n + 1 - 3)) if t - n >= 3 else 0
        out += [(k, a + s, n) for s in range(4) if a + s + n <= t]
        out += [(k, 0, lost + 2), (k, t - lost - 2, lost + 2), (k, 0, t)]
    w = np.asarray(out, dtype=np.int64)
    return w[rng.permutation(len(w))]


@pytest.mark.parametrize("layer", [6, 7])
@pytest.mark.parametrize("precision", ["tf32", "bf16", "fp16"])
def test_whole_recording_windows_are_bitwise_extract_x_vec_flat(xb, state_dict, precision, layer):
    lens = np.asarray([300, 45, 1000, 15, 16, 129, 2000, 257, 128])
    flat = torch.cat(ox.synth_ragged(lens, seed=21)).cuda()
    m = _model(xb, state_dict, precision, layer)
    w = np.stack([np.arange(lens.size), np.zeros(lens.size, dtype=np.int64), lens], 1)
    ref = m.extract_x_vec_flat(flat, lens).clone()
    got = m.extract_x_vec_windows(flat, lens, w)
    assert torch.equal(got.view(torch.int32), ref.view(torch.int32))  # bitwise, the NaN of the 15-frame recording included
    assert torch.isnan(got[3]).all() and torch.isfinite(got[np.arange(lens.size) != 3]).all()


@pytest.mark.parametrize("precision", ["tf32", "bf16", "fp16"])
def test_sliding_and_arbitrary_windows_match_resliced_extraction_and_the_oracle(xb, state_dict, precision):
    lens = np.asarray([3000, 1200, 800, 151, 40])
    utts = ox.synth_ragged(lens, seed=22)
    flat = torch.cat(utts).cuda()
    m = _model(xb, state_dict, precision)
    w = np.concatenate([xb.sliding_windows(lens, 150, 75), _arbitrary_windows(lens, 14, 23), [[2, 100, 15], [4, 25, 15]]])
    got = m.extract_x_vec_windows(flat, lens, w).cpu().numpy()
    ref = _resliced(m, utts, w)
    one = w[:, 2] == 15  # one pooled frame: NaN, like torch.std of one frame
    assert np.isnan(got[one]).all() and np.isnan(ref[one]).all()
    assert np.isfinite(got[~one]).all()
    assert np.abs(got[~one] - ref[~one]).max() <= BOUND[precision] * np.abs(ref[~one]).max()
    sel = np.random.default_rng(24).choice(np.nonzero(~one)[0], 16, replace=False)
    _parity(got[sel], ox.extract_ragged_t(state_dict, _slices(utts, w[sel]), 6).numpy(), precision)


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_wide_context_windows_use_the_per_layer_fallback(xb, precision):
    """The wide-context model of test_wide_context_falls_back_to_per_layer_launches (tap span 10: not taken by the stack
    kernel, lost_frames = 20): windows agree with its own extract_x_vec_flat over the sliced windows."""
    torch.manual_seed(3)
    m = xb.XVectorModel(precision=precision)
    m.time_context_layers[1] = xb.TdnnLayer(input_size=512, output_size=512, context=[-5, 0, 5])
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        for layer in m.time_context_layers:
            layer.norm.running_mean.copy_(0.3 * torch.randn(layer.norm.num_features, generator=g))
            layer.norm.running_var.copy_(0.5 + torch.rand(layer.norm.num_features, generator=g))
    m = m.cuda().eval()
    assert not m._stack_kernel_ok() and m.lost_frames == 20
    lens = np.asarray([700, 90, 300])
    utts = ox.synth_ragged(lens, seed=25)
    w = np.concatenate([xb.sliding_windows(lens, 100, 30), _arbitrary_windows(lens, 20, 26)])
    with pytest.raises(ValueError, match="more than 20"):
        m.extract_x_vec_windows(torch.cat(utts).cuda(), lens, [[0, 0, 20]])
    got = m.extract_x_vec_windows(torch.cat(utts).cuda(), lens, w).cpu().numpy()
    ref = _resliced(m, utts, w)
    assert np.isfinite(got).all()
    assert np.abs(got - ref).max() <= BOUND[precision] * np.abs(ref).max()


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_one_long_recording_with_sliding_windows(xb, state_dict, precision):
    x = ox.synth_mfcc(1, 60_000, seed=27)[0]
    w = xb.sliding_windows([60_000], 150, 75)
    assert len(w) == 799
    m = _model(xb, state_dict, precision)
    got = m.extract_x_vec_windows(x.cuda(), [60_000], w).cpu().numpy()
    assert got.shape == (799, 512) and np.isfinite(got).all()
    sel = np.asarray([0, 1, 400, 797, 798])
    _parity(got[sel], ox.extract_ragged_t(state_dict, _slices([x], w[sel]), 6).numpy(), precision)


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_host_extractor_windows_match_the_device_method(xb, state_dict, precision):
    """Batches of consecutive whole recordings (max_frames 5000: the 6000-frame recording is a batch of its own, one recording
    has no window), results in the order of `windows`."""
    lens = np.asarray([1000, 6000, 2000, 800, 3000, 500, 1200])
    utts = ox.synth_ragged(lens, seed=28)
    flat = torch.cat(utts)
    w = np.concatenate([xb.sliding_windows(lens, 150, 75), _arbitrary_windows(lens, 14, 29)])
    w = w[w[:, 0] != 5]
    w = w[np.random.default_rng(30).permutation(len(w))]
    m = _model(xb, state_dict, precision)
    hx = xb.HostExtractor(m)
    got = hx.extract_windows(flat.pin_memory(), lens, w, max_frames=5000)
    assert got.dtype == np.float64 and got.shape == (len(w), 512) and np.isfinite(got).all()
    ref = m.extract_x_vec_windows(flat.cuda(), lens, w).cpu().numpy()
    assert np.abs(got - ref).max() <= BOUND[precision] * np.abs(ref).max()
    dev = hx.extract_windows(flat, lens, w, max_frames=5000, to_host=False)
    assert dev.is_cuda and np.array_equal(dev.cpu().numpy().astype(np.float64), got)
