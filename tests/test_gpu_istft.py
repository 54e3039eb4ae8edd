"""The inverse STFT on the GPU (k_istft: iris_istft, Engine.istft, data_utils.to_waveform) against torch.istft in
float64 on the CPU: random spectra and real STFTs over channels, batch, frame counts and lengths, the ignored
imaginary parts of DC and Nyquist, load_wav round trips, the pipeline batch and the 'se' triple as audio,
phase_vocoder output, argument errors and determinism.

The bound is per sample, oracle/f64_ops.py istft_value_bound (tests/test_gpu_istft_f64.py has the edge shapes and
quiet inputs): the covering frames' overlap-add weights times their channel pair's norm, so that every item, pair
and channel is held to its own frames; the load_wav round trips add what the forward STFT's bound moves the exact
inverse (istft_carry).  Each test prints the largest ratio error / bound it measured, which must be <= 1."""
import numpy as np
import pytest

from oracle import f64, f64_ops as F
from test_gpu_istft_f64 import round_trip_value_bound

pytestmark = pytest.mark.gpu


def istft_ratio(got, spec, length=None):
    """Largest |got - value| / bound of istft_value_bound; samples no frame covers must be exactly +0."""
    val, bnd = F.istft_value_bound(spec, length)
    got = np.asarray(got)
    T = np.shape(spec)[-2]
    z = got[..., 256 * T:]
    assert not (np.any(z != 0) or np.signbit(z).any()), 'not +0 from 256 T on'
    return f64.worst(F.ratio(got, val, bnd))[0]


def _np(t):
    return t.detach().float().cpu().numpy()


def _random_spec(rng, shape):
    return rng.standard_normal(shape).astype(np.float32)


@pytest.mark.parametrize('T', [1, 2, 3, 626])
@pytest.mark.parametrize('B', [1, 5])
@pytest.mark.parametrize('C', [1, 2, 3, 4])
def test_random_spectra(engine, C, B, T):
    """Default, shorter and longer lengths; the 3-D form of one item gives the same samples as B = 1."""
    rng = np.random.default_rng(1000 * C + 10 * B + T)
    x = _random_spec(rng, (B, 257, T, 2 * C))
    default = 256 * (T - 1)
    lengths = ([None, default // 2 + 3, default + 300] if T > 1 else [100, 256, 700])
    worst = 0.0
    for length in lengths:
        got = _np(engine.istft(x, length))
        L = default if length is None else length
        assert got.shape == (B, C, L)
        worst = max(worst, istft_ratio(got, x, length))
        if B == 1:
            assert np.array_equal(_np(engine.istft(x[0], length)), got[0])
    print('C=%d B=%d T=%d ratio %.3g' % (C, B, T, worst))
    assert worst <= 1
    if T == 1:
        with pytest.raises(ValueError):
            engine.istft(x)


@pytest.mark.parametrize('C', [1, 2, 3])
def test_real_stfts(engine, C):
    """Spectrograms of real signals (float64 STFT rounded to float32), with and without a length."""
    from oracle import f64
    rng = np.random.default_rng(40 + C)
    for n in (256 * 300, 256 * 300 + 131):
        spec = np.stack([f64.spec_f64(rng.standard_normal((C, n))) for _ in range(3)]).astype(np.float32)
        for length in (None, n):
            r = istft_ratio(_np(engine.istft(spec, length)), spec, length)
            print('C=%d n=%d length=%s ratio %.3g' % (C, n, length, r))
            assert r <= 1


def test_dc_and_nyquist_imaginary_parts_are_ignored(engine):
    rng = np.random.default_rng(7)
    x = _random_spec(rng, (2, 257, 40, 6))
    z = x.copy()
    z[:, [0, 256], :, 3:] = 0.0
    a, b = _np(engine.istft(x, 40 * 256)), _np(engine.istft(z, 40 * 256))
    assert np.array_equal(a, b)
    assert istft_ratio(a, z, 40 * 256) <= 1


@pytest.mark.parametrize('n', [256 * 250, 256 * 250 + 1, 256 * 250 + 255, 40000 - 17])
@pytest.mark.parametrize('C', [1, 2])
def test_round_trip_through_load_wav(engine, n, C):
    """to_waveform(load_wav(w)) gives back normalize(w) (float64): the whole clip with length=n."""
    from challenge_b200 import data_utils as D
    w = np.random.default_rng(n + C).standard_normal((C, n)).astype(np.float32)
    spec = D.load_wav(w)
    length = None if n % 256 == 0 else n
    got = _np(D.to_waveform(spec, length=length))
    assert got.shape == (C, n)
    r = f64.worst(F.ratio(got, *round_trip_value_bound(w, _np(spec))))[0]
    print('round trip C=%d n=%d ratio %.3g' % (C, n, r))
    assert r <= 1


def _pipeline(separate, wave):
    from challenge_b200 import _ops as O
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import make_pipeline
    from challenge_b200.synth import synthetic_banks
    bgs, voices, labels, noises = synthetic_banks(5, 2, n_bg=3, n_voice=12, n_noise=4, bg_seconds=4.0)
    O.set_seed(91)
    ds = make_pipeline(bgs, voices, labels, noises, n_frame=120, max_voices=4, max_noises=2, min_ratio=1,
                       seperate_noise_voice=separate)
    ds = ds.map(D.to_frame_labels).map(D.augment).map(D.stft_filter(3)).batch(8)
    if wave:
        ds = ds.map(D.to_waveform)
    return [(x.clone(), tuple(v.clone() for v in y) if isinstance(y, tuple) else y.clone()) for x, y in ds.take(2)]


@pytest.mark.parametrize('separate', [False, True])
def test_pipeline_batch_as_audio(engine, separate):
    """make_pipeline(...).map(to_frame_labels).map(augment).map(stft_filter(3)).batch(8).map(to_waveform): the audio
    is the float64 inverse of the COMPLEX batch of the same seed, each item within the bound of its own frames, and
    the labels are bit-identical.  With seperate_noise_voice=True, only_voice and only_noise become audio too."""
    plain, wave = _pipeline(separate, False), _pipeline(separate, True)
    for (x, y), (xw, yw) in zip(plain, wave):
        assert tuple(xw.shape) == (8, 2, 256 * 119)
        pairs = [(xw, x)]
        if separate:
            assert torch_equal(yw[0], y[0])
            pairs += [(yw[1], y[1]), (yw[2], y[2])]
        else:
            assert torch_equal(yw, y)
        for got, spec in pairs:
            spec = _np(spec)
            r = istft_ratio(_np(got), spec)
            print('separate=%d ratio %.3g (peak %.3g)' % (separate, r, np.abs(spec).max()))
            assert r <= 1


def torch_equal(a, b):
    import torch
    return torch.equal(a, b)


def test_phase_vocoder_as_audio(engine):
    from challenge_b200 import data_utils as D
    from challenge_b200 import transforms as TR
    x = _random_spec(np.random.default_rng(11), (257, 200, 4))
    for rate in (0.8, 1.3):
        st = TR.phase_vocoder(x, rate)
        T2 = int(st.shape[1])
        got = _np(D.to_waveform(st))
        assert got.shape == (2, 256 * (T2 - 1))
        assert istft_ratio(got, _np(st)) <= 1


def test_bad_arguments(engine):
    import ctypes as C
    import torch
    from challenge_b200 import _lib as L
    x = torch.zeros((2, 257, 10, 4), device='cuda')
    out = torch.empty((2, 2, 2304), device='cuda')
    lib, ctx, st = engine.lib, engine._ctx, engine._stream()
    p = C.c_void_p(x.data_ptr())
    o = C.c_void_p(out.data_ptr())
    with pytest.raises(ValueError):
        L.check(lib.iris_istft(ctx, None, 2, 10, 2, 0, o, st))
    with pytest.raises(ValueError):
        L.check(lib.iris_istft(ctx, p, 2, 10, 2, 0, None, st))
    for B, T, Cn in ((0, 10, 2), (2, 0, 2), (2, 10, 0)):
        with pytest.raises(ValueError):
            L.check(lib.iris_istft(ctx, p, B, T, Cn, 0, o, st))
    with pytest.raises(ValueError):   # misaligned
        L.check(lib.iris_istft(ctx, C.c_void_p(x.data_ptr() + 4), 2, 10, 2, 0, o, st))
    with pytest.raises(ValueError):   # one frame, default length: no samples
        L.check(lib.iris_istft(ctx, p, 2, 1, 2, 0, o, st))
    with pytest.raises(NotImplementedError):
        L.check(lib.iris_istft(ctx, p, 1, 10, 33, 0, o, st))
    with pytest.raises(NotImplementedError):
        L.check(lib.iris_istft(ctx, p, 65536, 1, 1, 100, o, st))
    with pytest.raises(NotImplementedError):
        L.check(lib.iris_istft(ctx, p, 1, 10, 1, 1 << 31, o, st))
    with pytest.raises(ValueError):
        engine.istft(torch.zeros((257, 10, 3), device='cuda'))
    # a view at an offset that is not 16-byte aligned is copied first
    big = torch.as_tensor(_random_spec(np.random.default_rng(3), (257 * 5 * 2 + 1,)), device='cuda')
    view = big[1:].view(257, 5, 2)
    assert np.array_equal(_np(engine.istft(view)), _np(engine.istft(view.clone())))


def test_deterministic(engine):
    x = _random_spec(np.random.default_rng(5), (4, 257, 300, 4))
    a = _np(engine.istft(x, 300 * 256 + 99))
    b = _np(engine.istft(x, 300 * 256 + 99))
    assert np.array_equal(a, b)
