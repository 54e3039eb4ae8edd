"""The float64 reference and its per-cell error bounds (oracle/f64.py) on the CPU: the float32 oracle lies within
the bounds on every signal of the structured banks and every configuration it covers (this also re-measures the
ratios kappa is calibrated from), and each of a list of small defects planted in the float32 oracle breaks them --
some of which pass the normalised max-error bar of 1e-4 that the parity tests use."""
import numpy as np
import pytest

from conftest import nmax_err

TOL = 1e-4     # the normalised bar of the parity tests


def _banks(C, seed, fmt, white=False):
    """-> (fp32 banks for the oracle, float64 banks for the reference, labels, waveforms or None)."""
    from challenge_b200.synth import structured_banks, synthetic_banks
    from oracle import f64
    from oracle.chain import OracleBank
    if white:
        bgs, voices, labels, noises = synthetic_banks(seed, C, n_bg=2, n_voice=6, n_noise=3, bg_seconds=1.0,
                                                      lo_s=0.3, hi_s=1.0)
    else:
        bgs, voices, labels, noises = structured_banks(seed, C, n_voice=10, bg_seconds=1.5, hi_s=1.0)
    o = [OracleBank(x).specs for x in (bgs, voices, noises)]
    if fmt == 'spec':
        return o, [f64.bank_f64(x) for x in o], labels, None
    return o, [f64.bank_f64(x) for x in (bgs, voices, noises)], labels, (bgs, voices, noises)


def _draw(banks, B, T, seed, masks=True, merge_extra=0):
    from challenge_b200.plan import draw_batch
    fr = [np.array([s.shape[1] for s in x], np.int32) for x in banks]
    return draw_batch(np.random.default_rng(seed), B, T, fr[0], fr[1], fr[2], max_voices=4, max_noises=3, snr=-20,
                      min_ratio=2 / 3, n_time_masks=6 if masks else 0, time_mask_max=min(24, T),
                      n_freq_masks=1 if masks else 0, merge_extra=merge_extra)


def _complex32(o, labels, d, remap, n_out, stft_filter):
    """The float32 oracle's complex features (sj_train order: synthesis, masks, remap, stft_filter) and the keep
    flags it decided."""
    from oracle import chain, data_utils as OD
    if remap == 'mono_chan':
        x, y, _, keep = chain.dataset_batch(o[0], o[1], labels, o[2], d, mode='complex')
        x = np.stack([OD.mono_chan(xb, yb)[0] for xb, yb in zip(x, y)])
        if stft_filter:
            x = np.stack([OD.stft_filter(stft_filter)(xb) for xb in x])
    else:
        x, _, _, keep = chain.dataset_batch(o[0], o[1], labels, o[2], d, mode='complex', remap=remap,
                                            n_out_chan=n_out, stft_filter=stft_filter)
    return x.astype(np.float32), np.stack(keep)


def _post32(x, mode, mel_w=None, atan2=np.arctan2):
    """complex_to_magphase -> [log_magphase | mel -> [minmax] -> log_on_mel] of the float32 oracle."""
    from oracle import data_utils as OD, transforms as OT
    if mode == 'complex':
        return x
    n = x.shape[-1] // 2
    re, im = x[..., :n], x[..., n:]
    mag = np.sqrt(re ** 2 + im ** 2)
    mp = np.concatenate([mag, atan2(im, re).astype(np.float32)], -1)
    if mode == 'magphase':
        return mp
    if mode == 'log_magphase':
        return OT.log_magphase(mp, n_chan=mp.shape[-1] // 2)
    w = OT.linear_to_mel_weight_matrix(80, 257, 16000) if mel_w is None else mel_w
    mel = np.tensordot(mp[..., :mp.shape[-1] // 2], w, axes=[-3, 0]).astype(np.float32).transpose(0, 3, 1, 2)
    if mode == 'logmel_minmax':
        mel = OD.minmax(mel)
    return mel if mode == 'mel' else OD.log_on_mel(mel)


def _se32(o, labels, d, stft_filter):
    from oracle import chain, data_utils as OD, transforms as OT
    xs, vs, ns = [], [], []
    for b in range(d.batch):
        spec, (vtk, ov, on) = chain.synth_clip(o[0], o[1], labels, o[2], d, b, seperate_noise_voice=True)
        if d.time_masks is not None:
            spec = OT.mask(spec, axis=-2, max_mask_size=None, n_mask=d.time_masks.shape[1], draws=d.time_masks[b])
            spec = OT.mask(spec, axis=-3, max_mask_size=None, n_mask=d.freq_masks.shape[1], draws=d.freq_masks[b])
        if stft_filter:
            spec = OD.stft_filter(stft_filter)(spec)
        x, (_, v, n) = OD.speech_enhancement_preprocess(spec, (vtk, ov, on))
        xs.append(x)
        vs.append(v)
        ns.append(n)
    return [np.stack(a) for a in (xs, vs, ns)]


def _max_ratio(got, val, bound, mode):
    from oracle import f64
    return f64.worst(f64.ratio(got, val, bound, mode))


# (C, fmt, remap, n_out, stft_filter, masks, T, B)
CASES = [
    (2, 'wave', None, 0, 0, True, 64, 3), (2, 'wave', 'stereo_mono', 3, 3, False, 40, 2),
    (2, 'wave', 'merge_aug', 4, 0, True, 65, 2), (2, 'wave', 'mono_chan', 2, 3, True, 30, 2),
    (1, 'wave', None, 0, 3, False, 17, 3), (3, 'wave', None, 0, 0, True, 33, 2), (4, 'wave', None, 0, 0, False, 20, 2),
    (2, 'spec', None, 0, 3, True, 40, 2), (2, 'spec', 'merge_aug', 3, 0, False, 25, 2),
]
MODES = ('complex', 'magphase', 'log_magphase', 'mel', 'logmel', 'logmel_minmax')


def calibration_ratios(kappa_c=1.0):
    """-> (largest complex-cell ratio |oracle - f64| / bound at kappa_c, largest |fp32 mel - f64 mel| / (u mel)
    of the float32 mel on exact magnitudes) over the corpus: the numbers kappa_c / kappa_m are 4x of."""
    from oracle import f64
    from oracle import transforms as OT
    w = OT.linear_to_mel_weight_matrix(80, 257, 16000)
    rc, rm = 0.0, 0.0
    for i, (C, fmt, remap, n_out, filt, masks, T, B) in enumerate(CASES + [(2, 'wave', None, 0, 0, False, 50, 2)]):
        o, b64, labels, _ = _banks(C, 40 + i, fmt, white=i == len(CASES))
        d = _draw(o, B, T, i, masks, merge_extra=n_out - 2 if remap == 'merge_aug' else 0)
        x32, keep = _complex32(o, labels, d, remap, n_out, filt)
        val, bnd = f64.features(b64, labels, d, 'complex', fmt == 'spec', keep=keep, remap_kind=remap, n_out=n_out,
                                stft_filter=filt, gpu=False, kappa_c=kappa_c)
        rc = max(rc, _max_ratio(x32, val, bnd, 'complex')[0])
        n = val.shape[-1] // 2
        mag = np.hypot(val[..., :n], val[..., n:])
        mel64 = np.einsum('bftc,fm->bmtc', mag, w.astype(np.float64))
        mel32 = np.tensordot(mag.astype(np.float32), w, axes=[-3, 0]).astype(np.float32).transpose(0, 3, 1, 2)
        with np.errstate(divide='ignore', invalid='ignore'):
            r = np.where(mel64 > 0, np.abs(mel32 - mel64) / (f64.U * mel64), 0)
        rm = max(rm, float(r.max()))
    return rc, rm


def test_calibration_constants_hold():
    """kappa_c / kappa_m are 4x the ratios measured over the corpus; the written measurements are current."""
    from oracle import f64
    rc, rm = calibration_ratios()
    print('measured ratios: complex %.3f (written %.3f), mel %.3f (written %.3f)' %
          (rc, f64.MEASURED_RATIO_C, rm, f64.MEASURED_RATIO_M))
    assert rc <= f64.MEASURED_RATIO_C and rm <= f64.MEASURED_RATIO_M
    assert rc > 0.5 * f64.MEASURED_RATIO_C and rm > 0.5 * f64.MEASURED_RATIO_M     # not stale upwards either
    assert f64.KAPPA_C == 4 * f64.MEASURED_RATIO_C and f64.KAPPA_M == 4 * f64.MEASURED_RATIO_M


@pytest.mark.parametrize('case', range(len(CASES)))
def test_float32_oracle_within_the_bounds(case):
    """Every mode of the float32 oracle within the float64 bounds (no approximation terms: np.arctan2 / np.log are
    correctly rounded), SE blocks included where the configuration allows them."""
    from oracle import f64
    C, fmt, remap, n_out, filt, masks, T, B = CASES[case]
    o, b64, labels, _ = _banks(C, 40 + case, fmt)
    d = _draw(o, B, T, case, masks, merge_extra=n_out - 2 if remap == 'merge_aug' else 0)
    x32, keep = _complex32(o, labels, d, remap, n_out, filt)
    decided = 0
    for b in range(d.batch):        # the keep flags the float64 synthesis derives on its own
        if f64.keep_decidable(b64[1], d, b, fmt == 'spec'):
            assert f64.synth_index_level(b64[0], b64[1], labels, b64[2], d, b)[2] == list(keep[b]), b
            decided += 1
    assert decided
    kw = dict(remap_kind=remap, n_out=n_out, stft_filter=filt, mel_w=_mel_w(), gpu=False)
    for mode in MODES:
        got = _post32(x32, mode)
        val, bnd = f64.features(b64, labels, d, mode, fmt == 'spec', keep=keep, **kw)
        assert got.shape == val.shape, (mode, got.shape, val.shape)
        r, at = _max_ratio(got, val, bnd, mode)
        print('C=%d %s %s %s: ratio %.3f at %s' % (C, fmt, remap, mode, r, at))
        assert r <= 1, (mode, r, at)
    if C == 2 and remap is None:
        got = _se32(o, labels, d, filt)
        for g, (val, bnd) in zip(got, f64.features(b64, labels, d, 'se', fmt == 'spec', keep=keep, **kw)):
            assert f64.worst(f64.ratio(g, val, bnd, 'se'))[0] <= 1


def test_non_finite_outputs_fail_the_bounds():
    """A NaN or an infinity in any cell fails, also where the bound is unconstrained (inf) or 0, and in the phase
    columns; equal values and finite values under an unconstrained bound pass."""
    from oracle import f64
    ref = np.linspace(-1, 1, 2 * 5 * 3 * 4).reshape(2, 5, 3, 4)
    bound = np.full(ref.shape, 1e-6)
    bound[0, 0, 0] = np.inf
    bound[1, 1, 1] = 0.0
    for mode in ('mel', 'magphase'):
        assert f64.worst(f64.ratio(ref.copy(), ref, bound, mode))[0] == 0
        for at in ((0, 0, 0, 0), (1, 1, 1, 1), (1, 2, 2, 3), (0, 4, 2, 2)):
            for v in (np.nan, np.inf, -np.inf):
                got = ref.copy()
                got[at] = v
                r, where = f64.worst(f64.ratio(got, ref, bound, mode))
                assert r == np.inf and where == at, (mode, at, v)
        got = ref.copy()
        got[0, 0, 0] += 5.0                       # unconstrained cells: any finite value
        assert f64.worst(f64.ratio(got, ref, bound, mode))[0] == 0


def _mel_w():
    from oracle import transforms as OT
    return OT.linear_to_mel_weight_matrix(80, 257, 16000)


def _bank32(waves, window, left_pad):
    """The float32 oracle's load_wav with a different analysis window / left padding."""
    import torch
    from oracle import data_utils as OD
    out = []
    for w in waves:
        x = OD.normalize(w)
        pad = np.concatenate([np.pad(x, ((0, 0), (256, 0)), mode=left_pad)[:, :256], x,
                              np.pad(x, ((0, 0), (0, 256)), mode='reflect')[:, -256:]], 1)
        s = torch.stft(torch.from_numpy(np.ascontiguousarray(pad, np.float32)), 512, hop_length=256,
                       window=window, center=False, return_complex=True).numpy()
        out.append(OD.spec_layout(s))
    return out


def test_mutations_fail_the_bounds():
    """Small defects planted in the float32 oracle must break the per-cell bounds; the table records whether each
    one would have passed the normalised bar of 1e-4.  A 1e-4 gain on a band of bins passes that bar: the gap the
    per-cell bounds close.  A dropped mel tap of 8.7e-4 of its filter's weight is just visible to it (1e-4 .. 7e-4
    on brown .. white noise) and far outside the per-cell bounds.  The 80 dB pair runs on spectrogram banks, where no packed FFT
    ties the quiet channel's error to the loud one's."""
    import torch
    from oracle import f64
    w = _mel_w()
    rows = []

    def setup(white):
        o, b64, labels, waves = _banks(2, 77, 'wave', white=white)
        d = _draw(o, 3, 100, 5, masks=False)
        x32, keep = _complex32(o, labels, d, None, 0, 0)
        for mode in ('mel', 'complex', 'magphase'):      # the unmutated oracle passes
            val, bnd = bounds(mode, b64, d, labels, kp=keep)
            assert _max_ratio(_post32(x32, mode), val, bnd, mode)[0] <= 1, mode
        return o, b64, labels, waves, d, x32, keep

    def bounds(mode, banks, dd, labels, remap=None, spec=False, kp=None):
        return f64.features(banks, labels, dd, mode, spec, keep=kp, remap_kind=remap, n_out=2 if remap else 0,
                            mel_w=w, gpu=False)

    def record(name, got, mode, banks, dd, labels, **kw):
        val, bnd = bounds(mode, banks, dd, labels, **kw)
        r, at = _max_ratio(got, val, bnd, mode)
        rows.append((name, r, at, nmax_err(got, val)))

    # the two defects the normalised bar misses, on white noise (on the structured signals a tone or the chirp
    # in the band makes them visible to that bar as well)
    o, b64, labels, waves, d, x32, keep = setup(white=True)
    ctx = (b64, d, labels)
    s = w.sum(0)
    f, m = np.unravel_index(np.argmin(np.where(w > 0, w / s, np.inf)), w.shape)
    assert w[f, m] < 1e-3 * s[m]
    wd = w.copy()
    wd[f, m] = 0
    record('mel tap (%d, %d) of weight %.1e of its filter dropped' % (f, m, w[f, m] / s[m]),
           _post32(x32, 'mel', mel_w=wd), 'mel', *ctx, kp=keep)
    xb = x32.copy()
    xb[:, 60:68] *= np.float32(1 + 1e-4)
    record('bins 60-67 scaled by 1 + 1e-4', _post32(xb, 'mel'), 'mel', *ctx, kp=keep)
    o, b64, labels, waves, d, x32, keep = setup(white=False)
    ctx = (b64, d, labels)
    for name, window, pad in (('symmetric Hann window', torch.hann_window(512, periodic=False), 'reflect'),
                              ("'symmetric' padding at the start of a source", torch.hann_window(512), 'symmetric')):
        om = [_bank32(ws, window, pad) for ws in waves]
        record(name, _complex32(om, labels, d, None, 0, 0)[0], 'complex', *ctx, kp=keep)
    record('atan2 with 1e-5 rad error', _post32(x32, 'magphase', atan2=lambda y, x: np.arctan2(y, x) +
                                                1e-5 * np.cos(3 * np.arctan2(y, x))), 'magphase', *ctx, kp=keep)
    xm, km = _complex32(o, labels, d, 'mono_chan', 2, 0)
    xm[..., 2] = xm[..., 1]                          # re0 + im0 for both pseudo-channels
    record('mono_chan with im0 for both pseudo-channels', xm, 'complex', *ctx, remap='mono_chan', kp=km)
    from challenge_b200.synth import structured_source
    rng = np.random.default_rng(3)
    pair = [[structured_source(rng, 'pair80', 2, 16000)] for _ in range(3)]
    from oracle.chain import OracleBank
    op = [OracleBank(p).specs for p in pair]
    dp = _draw(op, 2, 40, 8, masks=False)
    xp, kpp = _complex32(op, np.eye(3, dtype=np.float32)[[0]], dp, None, 0, 0)
    xp[..., 1::2] *= np.float32(1 + 1e-5)            # re1 and im1: the quiet channel
    lab1 = np.eye(3, dtype=np.float32)[[0]]
    val, bnd = f64.features([f64.bank_f64(x) for x in op], lab1, dp, 'complex', True, keep=kpp, gpu=False)
    r, at = _max_ratio(xp, val, bnd, 'complex')
    rows.append(('1e-5 relative on the quiet channel of an 80 dB pair', r, at, nmax_err(xp, val)))
    print('\n%-56s %12s %22s %12s' % ('mutation', 'ratio/bound', 'at', 'nmax'))
    for name, r, at, nm in rows:
        print('%-56s %12.3g %22s %12.2e%s' % (name, r, str(at), nm, '  passes the 1e-4 bar' if nm < TOL else ''))
    for name, r, at, nm in rows:
        assert r > 1, ('mutation not caught', name, r)
    assert rows[1][3] < TOL, rows[1]
