"""Every feature kernel against the float64 reference of oracle/f64.py, cell by cell: |gpu - f64| within the per-cell
bound a correct float32 implementation is allowed there (kappa calibrated on the CPU, plus the stated budgets of
the kernels' approximations), on the structured signals of ``challenge_b200.synth.structured_banks`` -- quiet bins,
quiet frames, quiet channels, exact zeros -- where the normalised bar of the parity tests cannot see a defect.

A seeded sample of bank format x mode x remap x C x stft_filter x masks x T x B covers every (mode, remap, C,
format) cell; what the library refuses is compared with the list below.  The 2-channel mel kernels run in their
variants (generic epilogue, k_tiles tile lists, the all-bins mel matrix); features_select and iris_step once each;
bfloat16 / float16 features equal the float32 ones rounded.  Per configuration the largest ratio error / bound and
where it occurs is printed (profiles/r07_f64_bounds.txt)."""
import numpy as np
import pytest

from oracle import f64

pytestmark = pytest.mark.gpu

MODES = ('complex', 'magphase', 'log_magphase', 'mel', 'logmel', 'logmel_minmax', 'se')
REMAPS = ((None, 0), ('stereo_mono', 3), ('merge_aug', 3), ('merge_aug', 4), ('mono_chan', 2))
T_VALUES = (1, 2, 3, 17, 64, 65, 301)      # T = 1: the smallest the planner takes
B_VALUES = (1, 5, 24)


def refused(fmt, C, remap, mode):
    """What the library refuses: a channel remap of banks that are not 2-channel (data_utils.py:104 raises the
    same), and the 'se' batch of anything but 2-channel banks without a remap."""
    return (remap is not None and C != 2) or (mode == 'se' and (C != 2 or remap is not None))


EXPECTED_REFUSED = sorted((fmt, C, '%s%s' % (r, n if r == 'merge_aug' else ''), mode)
                          for fmt in ('wave', 'spec') for C in (1, 2, 3, 4) for r, n in REMAPS for mode in MODES
                          if refused(fmt, C, r, mode))


def _feat(mode):
    from challenge_b200 import _lib as L
    return {'complex': L.FEAT_COMPLEX, 'magphase': L.FEAT_MAGPHASE, 'log_magphase': L.FEAT_LOG_MAGPHASE,
            'mel': L.FEAT_MEL, 'logmel': L.FEAT_LOGMEL, 'logmel_minmax': L.FEAT_LOGMEL_MINMAX, 'se': L.FEAT_SE}[mode]


def _remap_id(remap):
    from challenge_b200 import _lib as L
    return {None: L.REMAP_NONE, 'stereo_mono': L.REMAP_STEREO_MONO, 'merge_aug': L.REMAP_MERGE_AUG,
            'mono_chan': L.REMAP_MONO_CHAN}[remap]


_banks = {}


def _register(engine, fmt, C):
    """Structured banks of C channels registered in format ``fmt`` -> (frames, float64 banks, labels)."""
    from challenge_b200 import _lib as L
    from challenge_b200.synth import structured_banks
    from oracle.chain import OracleBank
    key = (fmt, C)
    if key not in _banks:
        bgs, voices, labels, noises = structured_banks(700 + C, C)
        items = (bgs, voices, noises)
        if fmt == 'spec':
            items = tuple(OracleBank(x).specs for x in items)
        _banks[key] = (items, labels, [f64.bank_f64(x) for x in items])
    items, labels, b64 = _banks[key]
    frames = [engine.register_bank(L.BANK_BG, items[0]), engine.register_bank(L.BANK_VOICE, items[1], labels=labels),
              engine.register_bank(L.BANK_NOISE, items[2])]
    return frames, b64, labels


def _draw(frames, B, T, seed, masks, merge_extra=0):
    from challenge_b200.plan import draw_batch
    return draw_batch(np.random.default_rng(seed), B, T, frames[0], frames[1], frames[2], max_voices=4, max_noises=3,
                      snr=-20, min_ratio=2 / 3, n_time_masks=6 if masks else 0, time_mask_max=min(24, T),
                      n_freq_masks=1 if masks else 0, merge_extra=merge_extra)


def _np(t):
    return t.detach().float().cpu().numpy()


def _check(tag, got, ref, mode, report):
    """Every cell within its bound; one report line with the largest ratio and its (b, f|m, t, column)."""
    val, bnd = ref
    assert got.shape == val.shape, (tag, got.shape, val.shape)
    r, at = f64.worst(f64.ratio(got, val, bnd, mode))
    line = '%-62s ratio %8.3f at %s' % (tag, r, at)
    if mode == 'logmel_minmax':
        line += '  unconstrained %.2f %%' % (100 * float(np.isinf(bnd).mean()))
    report.append(line)
    print(line)
    assert r <= 1, (tag, r, at, float(got[at]), float(val[at]), float(bnd[at]))


def _exact_zeros(got, d, C, remap, fmt):
    """Masked / filtered cells are +-0; waveform banks: the DC and Nyquist imaginary parts are +0."""
    for b in range(d.batch):
        for size, off in (d.time_masks[b] if d.time_masks is not None else []):
            assert not got[b, :, off:off + size].any()
        for size, off in (d.freq_masks[b] if d.freq_masks is not None else []):
            assert not got[b, off:off + size].any()
    if fmt == 'wave' and remap != 'mono_chan':
        n = got.shape[-1] // 2
        for f in (0, 256):
            im = got[:, f, :, n:]
            assert not im.any() and not np.signbit(im).any()


def _matrix():
    """Sampled configurations; every mode runs on each.  A (format, C, remap) the library refuses gets one draw
    (refused at upload); every other gets two, the second with the stft_filter and masks of the first inverted.  T
    runs through a seeded shuffle of T_VALUES, so every T is drawn several times."""
    rng = np.random.default_rng(20261020)
    ts = [int(t) for t in np.concatenate([rng.permutation(T_VALUES) for _ in range(5)])]
    out = []
    for fmt in ('wave', 'spec'):
        for C in (1, 2, 3, 4):
            for remap, n_out in REMAPS:
                filt, masks = int(rng.choice([0, 3])), bool(rng.integers(2))
                if refused(fmt, C, remap, 'complex'):
                    out.append((fmt, C, remap, n_out, filt, masks, 64, 1))
                    continue
                for k in range(2):
                    T = ts.pop()
                    B = int(rng.choice(B_VALUES))
                    if T * B > 2000:            # keeps the float64 reference of the 301-frame clips to a few clips
                        B = 5
                    out.append((fmt, C, remap, n_out, filt if k == 0 else 3 - filt, masks != bool(k), T, B))
    return out


def test_feature_matrix_within_the_f64_bounds(engine):
    report, seen_refused, n_keep_checked = [], [], 0
    engine.set_mel(80)
    for i, (fmt, C, remap, n_out, filt, masks, T, B) in enumerate(_matrix()):
        frames, b64, labels = _register(engine, fmt, C)
        rname = '%s%s' % (remap, n_out if remap == 'merge_aug' else '')
        d = _draw(frames, B, T, 100 + i, masks, merge_extra=n_out - 2 if remap == 'merge_aug' else 0)
        try:
            engine.upload_plan(d, stft_filter=filt, chan_remap=_remap_id(remap), n_out_chan=n_out)
        except (ValueError, NotImplementedError):
            seen_refused += [(fmt, C, rname, mode) for mode in MODES]
            continue
        cache, keep = {}, None
        for mode in MODES:
            try:
                got = engine.features(_feat(mode))    # before iris_labels: tile lists from k_labels
            except (ValueError, NotImplementedError):
                seen_refused.append((fmt, C, rname, mode))
                continue
            if keep is None:
                keep = _np(engine.labels()[2]).astype(int)
                for b in range(B):      # the float64 synthesis derives the same flags where they are decidable
                    if f64.keep_decidable(b64[1], d, b, fmt == 'spec'):
                        assert f64.synth_index_level(b64[0], b64[1], labels, b64[2], d, b)[2] == list(keep[b]), \
                            ('keep flags', fmt, C, rname, b)
                        n_keep_checked += 1
            kw = dict(remap_kind=remap, n_out=n_out, stft_filter=filt, mel_w=engine.mel_matrix, keep=keep,
                      cache=cache)
            ref = f64.features(b64, labels, d, mode, fmt == 'spec', **kw)
            tag = '%s C=%d %s filt=%d masks=%d T=%d B=%d %s' % (fmt, C, rname, filt, masks, T, B, mode)
            if mode == 'se':
                for name, g, r in zip(('x', 'only_voice', 'only_noise'), got, ref):
                    _check(tag + ' ' + name, _np(g), r, mode, report)
            else:
                g = _np(got)
                _check(tag, g, ref, mode, report)
                if mode == 'complex':
                    _exact_zeros(g, d, C, remap, fmt)
    seen_refused = sorted(set(seen_refused))
    print('\n'.join(['refused: %s' % (r,) for r in seen_refused]))
    print('keep flags derived independently and equal on %d clips' % n_keep_checked)
    assert seen_refused == EXPECTED_REFUSED
    assert n_keep_checked > 0


def _stereo(engine, fmt, seed, B=6, T=120, filt=3):
    frames, b64, labels = _register(engine, fmt, 2)
    d = _draw(frames, B, T, seed, True)
    engine.upload_plan(d, stft_filter=filt)
    return d, b64, labels


@pytest.mark.parametrize('variant', ['fixed', 'IRIS_NO_FIXED_EPI', 'IRIS_NO_LABEL_TILES', 'all_bins'])
def test_two_channel_mel_variants(engine, monkeypatch, variant):
    """The 2-channel mel modes in each of their kernel variants: fixed vs generic epilogue, tile lists from k_labels
    vs k_tiles, and the all-bins mel matrix (80 bands to 7600 Hz)."""
    if variant.startswith('IRIS_'):
        monkeypatch.setenv(variant, '1')
    try:
        engine.set_mel(80, upper_edge_hertz=7600.0 if variant == 'all_bins' else 3800.0)
        d, b64, labels = _stereo(engine, 'wave', 41)
        cache = {}
        for mode in ('mel', 'logmel', 'logmel_minmax'):
            engine.upload_plan(d, stft_filter=3)          # features before labels: the k_labels tile lists
            got = _np(engine.features(_feat(mode)))
            keep = _np(engine.labels()[2]).astype(int)
            ref = f64.features(b64, labels, d, mode, False, keep=keep, stft_filter=3, mel_w=engine.mel_matrix,
                               cache=cache)
            _check('variant %s %s' % (variant, mode), got, ref, mode, [])
    finally:
        engine.set_mel(80)


def test_entry_points(engine):
    """features_select (only_voice) and iris_step against the float64 reference."""
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_config, uniforms_per_clip
    engine.set_mel(80)
    d, b64, labels = _stereo(engine, 'wave', 42, filt=0)
    engine.labels()
    got = _np(engine.features(L.FEAT_COMPLEX, select=L.SELECT_VOICES))
    keep = _np(engine.labels()[2]).astype(int)
    vals, bnds = [], []
    for b in range(d.batch):
        det = f64.synth_index_level(*[b64[0], b64[1], labels, b64[2]], d, b, keep=keep[b], detail=True)
        sv = f64.KAPPA_C * f64.U * f64.pair_scale(det['av'], False)
        vals.append(det['voice'])
        bnds.append(np.concatenate([sv, sv], -1) + f64.R_OUT * f64.U * np.abs(det['voice']))
    _check('features_select only_voice', got, (np.stack(vals), np.stack(bnds)), 'complex', [])
    B, T = 5, 90
    cfg = draw_config(B, T, 4, 3, -20, 2 / 3, 0.5, 6, 24, 1, 16)
    scfg = engine.step_config(cfg, L.FEAT_LOGMEL_MINMAX, stft_filter=3)
    x, _ = engine.step(scfg, np.random.default_rng(5).random((B, uniforms_per_clip(cfg))))
    torch.cuda.synchronize()
    x = _np(x)
    ds = engine.step_draws(scfg)
    engine.upload_plan(ds, stft_filter=3)
    keep = _np(engine.labels()[2]).astype(int)
    ref = f64.features(b64, labels, ds, 'logmel_minmax', False, keep=keep, stft_filter=3, mel_w=engine.mel_matrix)
    _check('iris_step logmel_minmax', x, ref, 'logmel_minmax', [])


@pytest.mark.parametrize('fmt', ['wave', 'spec'])
def test_half_features_are_rounded_float32(engine, fmt):
    """bfloat16 / float16 features of every mode equal the float32 ones converted with .to(dtype), on the
    structured signals (denormal-range and exactly-zero cells included)."""
    import torch
    engine.set_mel(80)
    _stereo(engine, fmt, 43)
    for mode in MODES[:-1]:
        ref = engine.features(_feat(mode))
        for dt in (torch.bfloat16, torch.float16):
            half = engine.features(_feat(mode), dtype=dt)
            assert torch.equal(half.view(torch.int16), ref.to(dt).view(torch.int16)), (fmt, mode, dt)
