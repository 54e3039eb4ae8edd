"""CPU side of the inverse STFT (iris_istft, Engine.istft, data_utils.to_waveform): the entry point is declared,
bound and optional; shapes are checked before anything reaches a device; a trailing to_waveform stage leaves the
fused part of a chain as it is; and the float64 reference the GPU tests compare against (torch.istft on the CPU)
gives back a known signal from its float64 STFT.  The reference and its error bound live here and are imported
by tests/test_gpu_istft.py."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def istft_f64(spec, length=None):
    """torch.istft(n_fft=512, hop_length=256, periodic Hann, center=True, length) in float64 on the CPU of
    ``[.., 257, T, 2C]`` spectrograms in load_wav's layout (real parts, then imaginary parts) -> ``[.., C, L]``."""
    import warnings
    import torch
    x = torch.as_tensor(np.asarray(spec, np.float64))
    C = x.shape[-1] // 2
    z = torch.complex(x[..., :C], x[..., C:]).movedim(-1, -3)          # [.., C, 257, T]
    lead = z.shape[:-2]
    with warnings.catch_warnings():   # a length past the last frame is padded with zeros on purpose
        warnings.simplefilter('ignore', UserWarning)
        y = torch.istft(z.reshape(-1, 257, z.shape[-1]), 512, 256, window=torch.hann_window(512, dtype=torch.float64),
                        center=True, length=length)
    return y.reshape(*lead, y.shape[-1]).numpy()


def ola_gain(T, L):
    """Per output sample, sum w / sum w^2 over the frames that cover it (0 where none does): how much an absolute
    error of the frames' samples grows in the output.  1 / envelope <= 2 where two frames overlap; 1 / w past the
    last frame's centre, where torch divides by a single window square."""
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(512) / 512)   # periodic Hann
    m = np.arange(L) + 256
    s1 = np.zeros(L)
    s2 = np.zeros(L)
    for t0 in (m // 256 - 1, m // 256):
        ok = (t0 >= 0) & (t0 < T) & (m - 256 * t0 < 512)
        wt = np.where(ok, w[np.clip(m - 256 * t0, 0, 511)], 0.0)
        s1 += wt
        s2 += wt * wt
    return np.where(s2 > 0, s1 / np.where(s2 > 0, s2, 1.0), 0.0)


def frame_peak(spec):
    """Largest |sample| of the float64 inverse FFTs of all frames and channels."""
    import torch
    x = torch.as_tensor(np.asarray(spec, np.float64))
    C = x.shape[-1] // 2
    z = torch.complex(x[..., :C], x[..., C:])
    return float(torch.fft.irfft(z, n=512, dim=-3).abs().max())


def istft_ratio(got, spec, length=None, ref=None):
    """max over samples of |got - ref| / (peak * ola_gain): the error per element in units of the frames' peak,
    scaled by how much the overlap-add divides it.  Where no frame covers a sample both must be exactly 0."""
    ref = istft_f64(spec, length) if ref is None else ref
    got = np.asarray(got, np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    g = ola_gain(np.shape(spec)[-2], ref.shape[-1])
    assert (got[..., g == 0] == 0).all() and (ref[..., g == 0] == 0).all()
    sel = g > 0
    if not sel.any():
        return 0.0
    return float((np.abs(got - ref)[..., sel] / (frame_peak(spec) * g[sel])).max())


def test_entry_point_is_declared_bound_and_optional():
    from challenge_b200 import _lib
    text = open(os.path.join(ROOT, 'include', 'iris.h')).read()
    assert 'int iris_istft(' in text and '#define IRIS_ABI_VERSION 2' in text
    assert 'iris_istft' in _lib.OPTIONAL and len(_lib.SIGNATURES['iris_istft'][1]) == 8
    assert hasattr(_lib.load(), 'iris_istft')


@pytest.mark.parametrize('shape,length', [
    ((256, 10, 4), None), ((257, 10), None), ((257, 10, 3), None), ((2, 3, 257, 10, 4), None),
    ((257, 0, 4), None), ((0, 257, 10, 4), None), ((257, 1, 4), None), ((257, 10, 4), 0), ((257, 10, 4), -5)])
def test_to_waveform_checks_shapes_before_the_device(shape, length):
    """A bad shape or length raises ValueError without a CUDA device (the check runs first)."""
    from challenge_b200 import data_utils as D
    with pytest.raises(ValueError):
        D.to_waveform(np.zeros(shape, np.float32), length=length)
    with pytest.raises(ValueError):   # the only_voice / only_noise members of a 'se' label are checked too
        D.to_waveform(np.zeros((257, 10, 4), np.float32), (None, np.zeros(shape, np.float32), None), length=length)


def test_istft_shape():
    from challenge_b200.engine import istft_shape
    assert istft_shape((257, 626, 4)) == (1, 626, 2, 160000)
    assert istft_shape((5, 257, 3, 6), 1000) == (5, 3, 3, 1000)
    assert istft_shape((1, 257, 1, 2), 100) == (1, 1, 1, 100)


def test_trailing_to_waveform_leaves_the_fused_chain_alone():
    """``.map(to_waveform)`` after ``.batch()`` runs on the un-fused COMPLEX batch: the lowering of the chain in
    front of it is what it is without the stage."""
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import IrisDataset
    for separate in (False, True):
        src = dict(n_chan=2, separate=separate)
        base = IrisDataset(src).map(D.to_frame_labels).map(D.augment).map(D.stft_filter(3)).batch(8)
        fused, rest = base._lower()
        fused_w, rest_w = base.map(D.to_waveform)._lower()
        assert fused_w == fused and fused['mode'] == 0 and rest == []
        assert rest_w == [D.to_waveform]


@pytest.mark.parametrize('n', [256 * 40, 256 * 40 + 77, 1000])
@pytest.mark.parametrize('C', [1, 2, 3])
def test_float64_reference_inverts_the_float64_stft(n, C):
    """The reference gives back a signal from its float64 STFT (oracle.f64: load_wav's STFT in float64, layout
    [257, T, 2C]); the default length is 256 (T - 1), ``length=n`` covers the rest."""
    from oracle import f64
    wav = np.random.default_rng(n + C).standard_normal((C, n))
    spec = f64.spec_f64(wav)
    T = spec.shape[1]
    assert T == 1 + n // 256
    ref = f64.normalize_f64(wav)
    y = istft_f64(spec)
    assert y.shape == (C, 256 * (T - 1))
    assert np.abs(y - ref[:, :y.shape[1]]).max() <= 1e-12 * np.abs(ref).max()
    y = istft_f64(spec, n)
    assert y.shape == (C, n)
    assert np.abs(y - ref).max() <= 1e-9 * np.abs(ref).max()
    assert istft_ratio(y.astype(np.float32), spec, n) <= 1e-6   # a float32 rounding alone: inside the GPU bound


def test_ola_gain_is_the_inverse_envelope():
    g = ola_gain(4, 256 * 5)
    assert np.allclose(g[:256 * 3], 1 / ((0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(256 * 3) % 256) / 512)) ** 2
                                          + (0.5 + 0.5 * np.cos(2 * np.pi * (np.arange(256 * 3) % 256) / 512)) ** 2))
    assert g[:256 * 3].max() <= 2 and g[:256 * 3].min() >= 1
    assert (g[256 * 3:256 * 4] >= 1).all() and (g[256 * 4:] == 0).all()
