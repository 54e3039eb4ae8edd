"""CPU side of the inverse STFT (iris_istft, Engine.istft, data_utils.to_waveform): the entry point is declared,
bound and optional; shapes are checked before anything reaches a device; a trailing to_waveform stage leaves the
fused part of a chain as it is; the float64 reference (oracle/f64_ops.py istft_f64: torch.istft on the CPU) gives
back a known signal from its float64 STFT; float32 inverses lie within its per-sample bound, whose constants are
re-measured here; and small defects planted in a float32 inverse break that bound, most of which pass the
global-peak bar (istft_ratio) the GPU tests used before it."""
import os
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
    """The global-peak bar: max over samples of |got - ref| / (peak * ola_gain), the error per element in units of
    the largest frame sample of the whole call, scaled by how much the overlap-add divides it; where no frame covers
    a sample both must be exactly 0.  Kept to show which defects it lets through (test_mutations_fail_the_bound)."""
    from oracle import f64_ops as F
    ref = F.istft_f64(spec, length) if ref is None else ref
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
    from oracle import f64, f64_ops as F
    wav = np.random.default_rng(n + C).standard_normal((C, n))
    spec = f64.spec_f64(wav)
    T = spec.shape[1]
    assert T == 1 + n // 256
    ref = f64.normalize_f64(wav)
    y = F.istft_f64(spec)
    assert y.shape == (C, 256 * (T - 1))
    assert np.abs(y - ref[:, :y.shape[1]]).max() <= 1e-12 * np.abs(ref).max()
    y = F.istft_f64(spec, n)
    assert y.shape == (C, n)
    assert np.abs(y - ref).max() <= 1e-9 * np.abs(ref).max()
    assert _worst(y.astype(np.float32), *F.istft_value_bound(spec, n))[0] <= 1   # a float32 rounding alone


def test_ola_gain_is_the_inverse_envelope():
    g = ola_gain(4, 256 * 5)
    assert np.allclose(g[:256 * 3], 1 / ((0.5 - 0.5 * np.cos(2 * np.pi * (np.arange(256 * 3) % 256) / 512)) ** 2
                                          + (0.5 + 0.5 * np.cos(2 * np.pi * (np.arange(256 * 3) % 256) / 512)) ** 2))
    assert g[:256 * 3].max() <= 2 and g[:256 * 3].min() >= 1
    assert (g[256 * 3:256 * 4] >= 1).all() and (g[256 * 4:] == 0).all()


def _worst(got, val, bnd):
    from oracle import f64, f64_ops as F
    return f64.worst(F.ratio(got, val, bnd))


def istft_f32(spec, length):
    """torch.istft in float32 on the CPU, with the periodic Hann window rounded to float32 from float64.
    (torch.hann_window(512) in float32 computes 0.5 - 0.5 cos in float32: 8e-4 off at w[511], which the division by
    w^2 past the last frame's centre brings into the output.)"""
    import torch
    x = torch.as_tensor(np.asarray(spec, np.float32))
    C = x.shape[-1] // 2
    z = torch.complex(x[..., :C], x[..., C:]).movedim(-1, -3)
    lead = z.shape[:-2]
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', UserWarning)
        y = torch.istft(z.reshape(-1, 257, z.shape[-1]), 512, 256,
                        window=torch.hann_window(512, dtype=torch.float64).float(), center=True, length=length)
    return y.reshape(*lead, y.shape[-1]).numpy()


def kernel_model_f32(spec, length, dc_imag_pairs=(), halo_from_next_hop=False, tail_ola_weights=False):
    """k_istft's arithmetic in float32 on the CPU: unnormalised float32 inverse FFT of each channel (512 x the
    frame), the kernel's float32 weights (the 1 / 512 on them), fmaf(x_h, hi, x_n * lo) where two frames cover a
    sample and x_h * tail past the last frame's centre, zeros from 256 T on.  The flags plant defects:
    ``dc_imag_pairs`` keeps the imaginary parts of bins 0 and 256 in the pair FFT of those channel pairs;
    ``halo_from_next_hop`` takes the halo frame of every 7-hop tile from the hop after it; ``tail_ola_weights``
    uses the overlap weight hi in place of the tail weight."""
    import torch
    x = np.asarray(spec, np.float32)
    C = x.shape[-1] // 2
    T = x.shape[-2]
    z = torch.complex(torch.as_tensor(x[..., :C]), torch.as_tensor(x[..., C:])).movedim(-1, -3)
    fr = torch.fft.irfft(z, n=512, dim=-2, norm='forward').numpy().astype(np.float64)   # [.., C, 512, T]
    alt = (-1.0) ** np.arange(512)
    for p in dc_imag_pairs:     # z = X_a + i X_b with Im X[0], Im X[256] kept: a gets -Im b, b gets +Im a
        a, b = 2 * p, 2 * p + 1
        fr[..., a, :, :] -= x[..., 0, None, :, C + b] + alt[:, None] * x[..., 256, None, :, C + b]
        fr[..., b, :, :] += x[..., 0, None, :, C + a] + alt[:, None] * x[..., 256, None, :, C + a]
    fr = fr.astype(np.float32)
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(512) / 512)
    r = np.arange(256)
    env = w[r] ** 2 + w[r + 256] ** 2
    lo, hi = np.float32(w[r] / (512 * env)), np.float32(w[r + 256] / (512 * env))
    tail = np.float32(1 / (512 * w[r + 256]))
    out = np.zeros(fr.shape[:-2] + (length,), np.float32)
    for h in range(min(T, -(-length // 256))):
        s0, s1 = 256 * h, min(256 * h + 256, length)
        n = s1 - s0
        xh = fr[..., 256:256 + n, h].astype(np.float64)
        if h + 1 < T:
            nxt = h + 2 if halo_from_next_hop and h % 7 == 6 and h + 2 < T else h + 1
            p = (fr[..., :n, nxt] * lo[:n]).astype(np.float64)
            out[..., s0:s1] = xh * hi[:n] + p                       # one rounding: fmaf
        else:
            out[..., s0:s1] = xh * (hi[:n] if tail_ola_weights else tail[:n])
    return out


def istft_cases():
    """(tag, float32 spectrum, length): the float64 STFT of every F.SIGNALS kind at C = 1, 2, 3 (rounded to
    float32, the whole clip and the tail past the last frame's centre), and a random [2, 257, 40, 8] batch with an
    item 120 dB down and, in the loud item, a pair 100 dB below the other."""
    from oracle import f64, f64_ops as F
    out = []
    for i, kind in enumerate(F.SIGNALS):
        for C in (1, 2, 3):
            n = 256 * 40 + 77
            w = F.signal(np.random.default_rng(100 * i + C), kind, C, n)
            out.append(('%s C=%d' % (kind, C), f64.spec_f64(w).astype(np.float32), n))
    out.append(('random quiet item / pair', quiet_batch(), 256 * 40 + 700))
    return out


def quiet_batch(seed=0):
    x = np.random.default_rng(seed).standard_normal((2, 257, 40, 8)).astype(np.float32)
    x[1] *= np.float32(1e-6)
    x[0, ..., [2, 3, 6, 7]] *= np.float32(1e-5)
    return x


def istft_ratios(fn):
    """-> (largest |fn - f64| / (u S) and where, largest ratio to the full bound) over istft_cases."""
    from oracle import f64_ops as F
    scale, full = (0.0, None), 0.0
    for tag, spec, L in istft_cases():
        val, bnd = F.istft_value_bound(spec, L)
        T = spec.shape[-2]
        S = F.istft_spread(F.istft_frame_norms(spec) / np.sqrt(512), T, L)
        got = fn(spec, L)
        r, at = _worst(got, val, F.U * S)
        if r > scale[0]:
            scale = (r, (tag, at))
        full = max(full, _worst(got, val, bnd)[0])
    return scale, full


def subnormal_spectrum():
    x = np.random.default_rng(3).standard_normal((2, 257, 20, 4)) * 1e-40
    x[1] *= 1e-3                                        # bins around 1e-43: the frames' samples are a few 2^-149
    return x.astype(np.float32)


def test_istft_kappa_remeasured():
    """KAPPA_ISTFT = 4x the largest |float32 torch.istft - f64| / (u S) over istft_cases, SUB_ISTFT = 4x the largest
    |kernel_model_f32 - f64| / (2^-149 G) on spectra around 1e-40 (torch's x w / w^2 underflows there: its product
    is rounded at the subnormal spacing before the division, which the kernel's single weight avoids); the written
    measurements are current.  The float32 kernel model lies within the full bound on every case."""
    from oracle import f64_ops as F
    (r, at), full = istft_ratios(istft_f32)
    print('istft: largest |torch.istft f32 - f64| / (u S) = %.3f at %s (written %.3f), ratio to the bound %.3f'
          % (r, at, F.MEASURED_RATIO_ISTFT, full))
    assert 0.5 * F.MEASURED_RATIO_ISTFT < r <= F.MEASURED_RATIO_ISTFT
    assert F.KAPPA_ISTFT == 4 * F.MEASURED_RATIO_ISTFT and full <= 1
    (r_model, at), full_model = istft_ratios(kernel_model_f32)
    print('istft: float32 kernel model, largest / (u S) %.3f at %s, ratio to the bound %.3f' % (r_model, at, full_model))
    assert full_model <= 1
    x = subnormal_spectrum()
    L = 256 * 20 + 30
    val, bnd = F.istft_value_bound(x, L)
    nrm = F.istft_frame_norms(x)
    G = F.istft_spread((nrm > 0).astype(np.float64), 20, L)
    sub = _worst(kernel_model_f32(x, L), val, F.TINY * G)[0]
    print('istft: subnormal spectra, largest |model - f64| / (2^-149 G) = %.3f (written %.3f)'
          % (sub, F.MEASURED_SUB_ISTFT))
    assert 0.5 * F.MEASURED_SUB_ISTFT < sub <= F.MEASURED_SUB_ISTFT and F.SUB_ISTFT == 4 * F.MEASURED_SUB_ISTFT
    assert _worst(kernel_model_f32(x, L), val, bnd)[0] <= 1


def test_istft_bound_edges():
    """No frame covers a sample from 256 T on, and an all-zero frame pair has norm 0: the bound is exactly 0 there
    (the output must be exactly 0); one frame (T = 1) covers 256 samples with the tail weight; istft_carry of a
    one-bin error is that bin's exact contribution at most."""
    from oracle import f64_ops as F
    x = np.random.default_rng(1).standard_normal((257, 9, 8)).astype(np.float32)
    x[:, 4, [2, 3, 6, 7]] = 0                     # frame 4 of pair 1 (channels 2 and 3) all zero
    val, bnd = F.istft_value_bound(x, 256 * 9 + 300)
    assert (bnd[:, 256 * 9:] == 0).all() and (val[:, 256 * 9:] == 0).all()
    # at r = 0 of hop 4, frame 5's weight w[0] / env is 0: only frame 4 covers the sample
    assert (bnd[2:4, 256 * 4] == 0).all() and (val[2:4, 256 * 4] == 0).all() and (bnd[0:2, 256 * 4] > 0).all()
    assert (bnd[2:4, 256 * 4 + 1] > 0).all()
    val1, bnd1 = F.istft_value_bound(x[:, :1], 300)
    assert (bnd1[:, :256] > 0).all() and (bnd1[:, 256:] == 0).all() and (val1[:, 256:] == 0).all()
    e = np.zeros((257, 9, 8))
    e[37, 5, 1] = 1e-3                            # the real part of bin 37, frame 5, channel 1
    carried = np.abs(F.istft_f64(x + e, 256 * 9) - F.istft_f64(x, 256 * 9))
    carry = F.istft_carry(e, 9, 256 * 9)
    assert (carried <= carry * (1 + 1e-9) + 1e-15).all()
    assert carried[1].max() > 0.5 * carry[1].max() and np.delete(carried, 1, 0).max() < 1e-15


def test_mutations_fail_the_bound():
    """Small defects planted in the float32 inverse (kernel_model_f32) of a random [2, 257, 40, 8] batch (item 1 at
    -120 dB, pair 1 of item 0 at -100 dB; length 256 T + 700): each breaks the per-sample bound.  The table shows which of them pass
    the global-peak bar (istft_ratio <= 1e-6) that held the GPU inverse before."""
    from oracle import f64_ops as F
    x = quiet_batch()
    T, L = 40, 256 * 40 + 700
    val, bnd = F.istft_value_bound(x, L)
    base = kernel_model_f32(x, L)
    assert _worst(base, val, bnd)[0] <= 1
    rows = []

    def record(name, got):
        try:
            old = istft_ratio(got, x, L, ref=val)
        except AssertionError:      # a non-zero sample where no frame covers: the old bar fails it too
            old = np.inf
        rows.append((name, _worst(got, val, bnd), old))

    g = base.copy()
    g[1] *= np.float32(1 + 1e-3)
    record('a quiet item\'s gain off by 1e-3', g)
    g = base.copy()
    g[0, 2:4] += np.float32(1e-3) * base[0, 0:2]
    record('1e-3 of the loud pair leaking into the quiet pair', g)
    record('bins 0 / 256 imaginary parts kept for pair 1 only (kC = 0)', kernel_model_f32(x, L, dc_imag_pairs=(1,)))
    g = base.copy()
    g[1] = kernel_model_f32(x, L, halo_from_next_hop=True)[1]
    record('the quiet item: halo frame of each tile from the next hop', g)
    g = base.copy()
    g[1] = kernel_model_f32(x, L, tail_ola_weights=True)[1]
    record('the quiet item: overlap weights in the tail instead of 1 / w', g)
    g = base.copy()
    g[1, :, 256 * T + 5] = np.float32(1e-30)
    record('1e-30 written past 256 T', g)
    print('\n%-64s %12s %16s %12s  %s' % ('planted defect', 'ratio/bound', 'at', 'old bar', 'old bar (1e-6)'))
    for name, (r, at), old in rows:
        print('%-64s %12.3g %16s %12.3g  %s' % (name, r, str(at), old, 'passes' if old <= 1e-6 else 'fails'))
    for name, (r, at), old in rows:
        assert r > 1, (name, r, at)
    assert sum(old <= 1e-6 for _, _, old in rows) >= 3
