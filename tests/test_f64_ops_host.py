"""The float64 values and per-cell bounds of the stand-alone operations (oracle/f64_ops.py) on the CPU: the float32
oracle lies within every bound, or equals the bit-exact float32 form, on the signals the GPU test uses; the one
calibrated constant (KAPPA_LOAD, for load_wav) is re-measured; and a list of small defects planted in the float32
oracle breaks the bounds, most of which pass the normalised max-error bar of the test they would otherwise meet."""
import numpy as np
import pytest

from conftest import nmax_err

SEED = 20261022


def _sig(kind, C, n, seed=0):
    from oracle import f64_ops as F
    return F.signal(np.random.default_rng(seed), kind, C, n)


def _worst(got, val, bnd):
    from oracle import f64, f64_ops as F
    return f64.worst(F.ratio(got, val, bnd))


LOAD_CASES = [(kind, C, n, norm) for kind, C, n, norm in (
    ('white', 2, 257, True), ('tones', 1, 300, True), ('chirp', 3, 513, True), ('pair80', 2, 768, True),
    ('burst_tail', 2, 4001, True), ('pair100', 2, 4000, False), ('dc_nyquist', 1, 2048, True), ('clicks', 4, 3000, True),
    ('quiet', 5, 2500, False), ('zeros', 2, 48001, True), ('brown', 2, 48000, True), ('pink', 3, 16000, True))]


def load_wav_ratios(scale_only=True):
    """-> largest |oracle - f64| / (u * S_pair) over LOAD_CASES, or (scale_only False) the largest ratio to the
    bound."""
    from oracle import data_utils as OD, f64, f64_ops as F
    worst = 0.0
    for i, (kind, C, n, norm) in enumerate(LOAD_CASES):
        w = _sig(kind, C, n, i)
        got = OD.load_wav_array(w, do_normalize=norm)
        val, bnd = F.stft_value_bound(w, normalize=norm, kappa=1.0 if scale_only else F.KAPPA_LOAD)
        if scale_only:     # the scale alone: bound - R_OUT u |v|
            bnd = bnd - f64.R_OUT * F.U * np.abs(val)
        worst = max(worst, _worst(got, val, bnd)[0])
    return worst


def test_load_wav_kappa_remeasured():
    """load_wav's bound is the 'complex' cell of oracle/f64.py with KAPPA_LOAD = 4x the ratio the float32 oracle
    reaches on these signals; the written measurement is current."""
    from oracle import f64_ops as F
    r = load_wav_ratios()
    print('load_wav: largest |oracle - f64| / (u S_pair) = %.3f (written %.3f)' % (r, F.MEASURED_RATIO_LOAD))
    assert 0.5 * F.MEASURED_RATIO_LOAD < r <= F.MEASURED_RATIO_LOAD
    assert F.KAPPA_LOAD == 4 * F.MEASURED_RATIO_LOAD
    assert load_wav_ratios(scale_only=False) <= 1


RATES = [(22050, 16000), (44100, 16000), (48000, 16000), (96000, 16000), (8000, 16000), (11025, 16000),
         (12000, 16000), (44101, 16000)]


@pytest.mark.parametrize('orig,new', RATES)
def test_resample_oracle_within_bound(orig, new):
    from oracle import data_utils as OD, f64_ops as F
    table = F.kaldi_table(orig, new)
    for kind, n in (('burst_tail', 6001), ('pair100', 3000), ('tones', 2000)):
        w = _sig(kind, 2, n, orig)
        val, bnd = F.resample_value_bound(w, orig, new, table)
        got = OD.resample_waveform(w, orig, new)
        r, at = _worst(got, val, bnd)
        print('%d -> %d %-10s ratio %.3f at %s' % (orig, new, kind, r, at))
        assert r <= 1, (kind, r, at)


@pytest.mark.parametrize('orig,new', [(44100, 16000), (8000, 16000), (11025, 16000), (44101, 16000)])
def test_kaldi_table_within_half_a_tab(orig, new):
    """numpy's float32 table against the same table in float64 from the same float32 time offsets and cos / sin
    arguments (both float32 tables round those identically): within half of the A_TAB allowance between two float32
    tables."""
    from oracle import f64_ops as F
    first, w, s, u_in, u_out = F.kaldi_table(orig, new)
    cutoff = 0.99 * 0.5 * min(orig, new)
    width = 6 / (2.0 * cutoff)
    t = np.arange(u_out, dtype=np.float32) / np.float32(new)
    dt = ((first.astype(np.float32)[:, None] + np.arange(w.shape[1], dtype=np.float32)[None, :]) / np.float32(orig)
          - t[:, None]).astype(np.float64)
    d32 = dt.astype(np.float32)
    a = (np.float32(2 * np.pi * cutoff / 6) * d32).astype(np.float64)        # the float32 arguments of cos / sin
    b = (np.float32(2 * np.pi * cutoff) * d32).astype(np.float64)
    h = np.where(np.abs(dt) < np.float32(width), 0.5 * (1 + np.cos(a)), 0.0)
    with np.errstate(divide='ignore', invalid='ignore'):
        sinc = np.where(dt == 0, 2 * cutoff, np.sin(b) / (np.pi * dt))
    w64 = h * sinc / orig
    r = float((np.abs(w - w64) / (F.U * s + 1e-300)).max())
    print('%d -> %d: W = %d, max |w32 - w64| / (u |s|) = %.2f' % (orig, new, w.shape[1], r))
    assert r <= F.A_TAB / 2


def test_pointwise_oracle_within_bounds():
    """complex_to_magphase, magphase_to_complex, log_magphase, log_on_mel and multiply_label of the float32 oracle
    on values spanning 1e-30 .. 1e18 (+-0, subnormals, overflowing squares)."""
    from oracle import data_utils as OD, f64_ops as F, transforms as OT
    rng = np.random.default_rng(SEED)
    x = F.span_values(rng, (64, 33, 6))
    val, bnd, exact = F.complex_to_magphase(x)
    got = OT.complex_to_magphase(x).astype(np.float32)
    m = F.magnitude_f32(x)
    assert np.array_equal(got[..., :3][exact].view(np.uint32), m[exact].view(np.uint32))
    val[..., :3][exact] = got[..., :3][exact]
    assert exact.sum() > 0 and _worst(got, val, bnd)[0] <= 1
    mono = x[..., :3]
    val, bnd, exact = F.complex_to_magphase(mono)
    got = np.concatenate([np.sqrt(mono[..., :1] ** 2 + mono[..., 1:] ** 2),
                          np.arctan2(mono[..., 1:], mono[..., :1])], -1)
    val[..., :2][exact] = got[..., :2][exact]
    assert _worst(got, val, bnd)[0] <= 1
    mp = np.concatenate([F.span_values(rng, (64, 33, 3), signed=False), F.span_values(rng, (64, 33, 3))], -1)
    assert _worst(OT.magphase_to_complex(mp), *F.magphase_to_complex(mp))[0] <= 1
    pos = F.span_values(rng, (64, 33, 6), signed=False)
    assert _worst(OT.log_magphase(pos, n_chan=3), *F.log_magphase(pos, 3))[0] <= 1
    assert _worst(OD.log_on_mel(pos), *F.log_eps(pos))[0] <= 1
    assert _worst(OD.multiply_label(0.25)(None, x)[1], *F.multiply(x, 0.25))[0] <= 1


def _mags(C, T=40, seed=0):
    """Magnitudes / phases [2, 257, T, 2C] of the structured signals (the bins of load_wav)."""
    from oracle import data_utils as OD, transforms as OT
    out = []
    for b, kind in enumerate(('brown', 'tones')):
        w = _sig(kind, C, 256 * (T - 1), seed + b)
        out.append(OT.complex_to_magphase(OD.load_wav_array(w)))
    return np.stack(out).astype(np.float32)


@pytest.mark.parametrize('n_mel,kw', [(80, {}), (40, {}), (128, dict(upper_edge_hertz=8000.0)),
                                      (80, dict(lower_edge_hertz=0.0))])
def test_mel_oracle_within_bound(n_mel, kw):
    from oracle import f64_ops as F, transforms as OT
    x = _mags(2)
    w = OT.linear_to_mel_weight_matrix(n_mel, 257, 16000, **kw)
    got = OT.magphase_to_mel(n_mel, **kw)(x)
    r, at = _worst(got, *F.mel_value_bound(x, w))
    print('mel %d %s: ratio %.3f at %s' % (n_mel, kw, r, at))
    assert r <= 1


def test_bitexact_forms_equal_the_oracle():
    """minmax, minmax_norm_magphase, the channel maps, to_frame_labels, label pooling, preprocess_labels and
    to_density_labels: the float32 oracle equals the kernel-order float32 form bit for bit."""
    from oracle import data_utils as OD, f64_ops as F, trainer as OTR, transforms as OT
    rng = np.random.default_rng(SEED)
    x = (rng.standard_normal((6, 80, 50, 2)) * 3).astype(np.float32)
    assert np.array_equal(F.minmax_f32(x), OD.minmax(x))
    assert np.array_equal(F.minmax_norm_magphase_f32(x), OT.minmax_norm_magphase(x))
    spec = rng.standard_normal((257, 20, 4)).astype(np.float32)
    assert np.array_equal(F.chan_map_f32(spec, 'stereo_mono'), OD.stereo_mono(spec))
    assert np.array_equal(F.chan_map_f32(spec, 'mono_chan'), OD.mono_chan(spec, 'y')[0])
    f = np.float32([0.3, 0.7, 0.123])
    assert np.array_equal(F.chan_map_f32(spec, 'merge_aug', f), OD.random_merge_aug(5)(spec, factor=f))
    y = (rng.random((3, 7, 40, 3)) < 0.2).astype(np.float32)
    assert np.array_equal(F.sum_voices_f32(y), OD.to_frame_labels(None, y)[1])
    for T, r in ((100, 7), (31, 32), (1, 4)):
        yy = (rng.random((5, T, 3)) < 0.5).astype(np.float32)
        assert np.array_equal(F.avg_pool_time_f32(yy, r, True)[:r], OD.label_downsample(r)(None, yy)[1])
    for T in (33, 34, 1):
        yy = (rng.random((4, T, 3)) < 0.3).astype(np.float32) * 3
        assert np.array_equal(F.preprocess_labels_f32(yy, 0.25), OTR.preprocess_labels(0.25)(None, yy)[1])
    assert np.array_equal(F.density_labels_f32(y), OTR.to_density_labels(None, y)[1])


def test_normalize_cos_sim_vocoder_oracle_within_bounds():
    from oracle import data_utils as OD, f64_ops as F, metrics as OM, transforms as OT
    for i, kind in enumerate(('pair80', 'burst_tail', 'pair100', 'tones')):
        w = _sig(kind, 2, 30001, i)
        assert _worst(OD.normalize(w), *F.normalize_value_bound(w))[0] <= 1, kind
    rng = np.random.default_rng(SEED)
    yt = (rng.random((16, 200, 8)) < 0.3).astype(np.float32)
    yt[3] = 0
    yp = np.clip(yt + rng.normal(0, 0.35, yt.shape), 0, 1).astype(np.float32)
    yp[4] = 0
    yp[5] *= np.float32(1e-8)
    assert _worst(OM.cos_sim(yt, yp), *F.cos_sim_value_bound(yt, yp))[0] <= 1
    x = OD.load_wav_array(_sig('tones', 3, 256 * 29, 1))
    for rate in (0.3, 0.7, 1.5, 3.0, 1.0001):
        pv = OT.phase_vocoder(x, rate)
        C = x.shape[-1] // 2
        r, at = _worst(np.hypot(pv[..., :C].astype(np.float64), pv[..., C:]), *F.vocoder_magnitude(x, rate))
        assert r <= 1, (rate, r, at)


def test_non_finite_values_fail():
    """NaN or inf where the reference is finite fails whatever the bound; a non-finite reference needs the same
    non-finite value; the bit-exact ratio fails on any bit (the sign of a zero included)."""
    from oracle import f64_ops as F
    ref = np.linspace(-1, 1, 24).reshape(4, 6)
    bnd = np.full(ref.shape, np.inf)
    for v in (np.nan, np.inf, -np.inf):
        got = ref.copy()
        got[1, 2] = v
        assert F.ratio(got, ref, bnd)[1, 2] == np.inf
    ref2 = ref.copy()
    ref2[0, 0] = -np.inf
    got = ref2.copy()
    assert F.ratio(got, ref2, 1e-9)[0, 0] == 0
    got[0, 0] = np.inf
    assert F.ratio(got, ref2, 1e-9)[0, 0] == np.inf
    got[0, 0] = -3.0
    assert F.ratio(got, ref2, 1e-9)[0, 0] == np.inf
    z = np.zeros(3, np.float32)
    assert F.bitexact_ratio(-z, z).min() == np.inf and F.bitexact_ratio(z, z).max() == 0


def test_phase_of_the_wrong_sign_at_the_branch_cut_fails():
    """atan2(+0, -1) = pi and atan2(-0, -1) = -pi: a phase of the other sign there (a circular difference would call
    it 0) fails the atan2f bound; fl(pi) against the exact pi passes."""
    from oracle import f64_ops as F
    x = np.float32([[-1.0, 0.0], [-1.0, -0.0], [-2.5, 0.0]])        # rows of [re, im]
    val, bnd, _ = F.complex_to_magphase(x)
    good = np.concatenate([np.hypot(x[:, :1], x[:, 1:]), np.arctan2(x[:, 1:], x[:, :1])], -1).astype(np.float32)
    assert F.ratio(good, val, bnd).max() <= 1
    bad = good.copy()
    bad[:, 1] = -bad[:, 1]
    assert (F.ratio(bad, val, bnd)[:, 1] > 1e6).all()


def test_mutations_fail_the_bounds():
    """Small defects planted in the float32 oracle break the per-cell bounds; the table records the normalised max
    error beside each and whether it passes the bar of the test that checks the operation today."""
    from oracle import data_utils as OD, f64_ops as F, metrics as OM, transforms as OT
    rows = []

    def record(name, got, val, bnd, bar, expect_caught=True):
        r, at = _worst(got, val, bnd)
        rows.append((name, r, at, nmax_err(got, val), bar, expect_caught))

    # resample: a quiet tail filtered with the wrong polyphase row; the last FIR tap dropped
    orig = 44100
    w = _sig('burst_tail', 2, 22050, 3)
    table = F.kaldi_table(orig, 16000)
    val, bnd = F.resample_value_bound(w, orig, 16000, table)
    ref32 = OD.resample_waveform(w, orig, 16000)
    first, wt, s, u_in, u_out = table
    rolled = (first, np.roll(wt, 1, 0), s, u_in, u_out)
    bad = ref32.copy()
    tail = np.arange(bad.shape[1]) > bad.shape[1] // 2
    bad[:, tail] = F.resample_value_bound(w, orig, 16000, rolled)[0][:, tail]
    record('resample: the quiet tail with the previous polyphase row', bad, val, bnd, 1e-5)
    cut = wt.copy()
    cut[:, -1] = 0
    record('resample: the last FIR tap dropped', F.resample_value_bound(w, orig, 16000, (first, cut, s, u_in, u_out))[0],
           val, bnd, 1e-5)
    # mel: one band's support shifted by one bin
    x = _mags(2)
    mw = OT.linear_to_mel_weight_matrix(80, 257, 16000)
    first = np.array([mw[np.argmax(mw[:, k] > 0), k] / mw[:, k].sum() for k in range(80)])
    m = int(np.argmin(first))           # rows [lo + 1, lo + len + 1) of band m: its first weight is lost
    sh = mw.copy()
    sh[np.argmax(mw[:, m] > 0), m] = 0
    got = np.tensordot(x[..., :2], sh, axes=[-3, 0]).astype(np.float32).transpose(0, 3, 1, 2)
    record('mel band %d support shifted up by one bin' % m, got, *F.mel_value_bound(x, mw), 1e-5)
    # load_wav: 1e-5 relative on a channel 80 dB below the others, in its own FFT pair (channel 2 of 3) -- and, as
    # a limit of what any bound can hold a packed FFT to, on the quiet member of a stereo pair
    w3 = _sig('brown', 3, 8000, 4)
    w3[2] *= np.float32(1e-4)
    got = OD.load_wav_array(w3)
    got[..., 2::3] *= np.float32(1 + 1e-5)
    record('load_wav: 1e-5 on a channel 80 dB down (own FFT pair)', got, *F.stft_value_bound(w3), 1e-4)
    w2 = _sig('pair80', 2, 8000, 5)
    got = OD.load_wav_array(w2)
    got[..., 1::2] *= np.float32(1 + 1e-5)
    record('load_wav: 1e-5 on the quiet member of an 80 dB stereo pair', got, *F.stft_value_bound(w2), 1e-4,
           expect_caught=False)
    # normalize with the mean over channel 0 only (channel 1 at 1.000002 x its RMS)
    wn = _sig('white', 2, 30000, 6).astype(np.float64)
    wn[1] *= np.sqrt(np.mean(wn[0] ** 2) / np.mean(wn[1] ** 2)) * (1 + 2e-6)
    wn = wn.astype(np.float32)
    import torch
    t = torch.as_tensor(wn)
    bad = (t / (torch.sqrt(torch.mean(t[:1] ** 2)) * 10)).numpy()
    record('normalize: the mean over channel 0 only', bad, *F.normalize_value_bound(wn), 2e-6)
    # complex_to_magphase: atan2 with its arguments swapped in the third quadrant
    rng = np.random.default_rng(7)
    xc = rng.standard_normal((257, 40, 4)).astype(np.float32)
    near = rng.random((257, 40, 2)) < 0.01                   # cells close to the diagonal
    xc[..., 2:][near] = xc[..., :2][near] * np.float32(1 + 3e-6)
    mp = OT.complex_to_magphase(xc)
    re, im = xc[..., :2], xc[..., 2:]
    q3 = (re < 0) & (im < 0)
    mp[..., 2:][q3 & near] = np.arctan2(re, im)[q3 & near]
    val, bnd, _ = F.complex_to_magphase(xc)
    record('complex_to_magphase: atan2(x, y) in quadrant 3, |x| ~ |y|', mp, val, bnd, 1e-5)
    # cos_sim without the 1e-12 floor, on a sample of predictions 1e-7 of the others
    rng = np.random.default_rng(8)
    yt = (rng.random((16, 200, 3)) < 0.3).astype(np.float32)
    yp = np.clip(yt + rng.normal(0, 0.35, yt.shape), 0, 1).astype(np.float32)
    yp[2] *= np.float32(2e-8)
    a, p = yt.astype(np.float64), yp.astype(np.float64)
    cs = -(a * p).sum(1) / np.sqrt(np.maximum((a * a).sum(1), 1e-12)) / np.sqrt((p * p).sum(1))
    occ = (a.sum(1) > 0).astype(np.float64)
    bad = (cs * occ / np.maximum(occ.sum(1, keepdims=True), 1e-8)).sum(1).astype(np.float32)
    record('cos_sim without the 1e-12 floor', bad, *F.cos_sim_value_bound(yt, yp), 2e-6)
    print('\n%-60s %12s %18s %10s  %s' % ('mutation', 'ratio/bound', 'at', 'nmax', 'bar of today\'s test'))
    for name, r, at, nm, bar, _ in rows:
        print('%-60s %12.3g %18s %10.2e  %s %.0e' % (name, r, str(at), nm, 'passes' if nm < bar else 'fails', bar))
    for name, r, at, nm, bar, caught in rows:
        assert (r > 1) == caught, (name, r)
    assert sum(nm < bar for _, _, _, nm, bar, c in rows if c) >= 4
