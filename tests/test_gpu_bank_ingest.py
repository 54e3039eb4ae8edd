"""Waveform banks registered from audio at any sample rate (``iris_bank_register_audio``): the items are
resampled to 16 kHz on the device with load_wav's filter in one pass per bank, then registered as 16 kHz
banks are.  Checked against the per-item route (``Engine.resample`` of every item, then a 16 kHz bank) bit
for bit, against ``load_wav``'s spectrograms, through ``make_pipeline`` / ``merge_complex_specs``, and on
the error cases."""
import numpy as np
import pytest

from conftest import nmax_err

pytestmark = pytest.mark.gpu

RATES = (44100, 48000, 22050, 11025, 32000, 8000, 16000)


def _np(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope='module')
def mods(engine):
    import challenge_b200
    from challenge_b200 import data_utils, engine as E, pipeline, transforms
    E._engines[0] = engine
    challenge_b200.set_seed(0)
    return pipeline, transforms, data_utils


def _banks(seed, n_chan, rate, **kw):
    from challenge_b200.synth import synthetic_banks
    args = dict(n_bg=2, n_voice=6, n_noise=3, bg_seconds=3.0)
    args.update(kw)
    return synthetic_banks(seed, n_chan, sr=rate, **args)


def _register(engine, bgs, voices, labels, noises):
    """-> frames of the three banks, activity of every voice."""
    from challenge_b200 import _lib as L
    bf = engine.register_bank(L.BANK_BG, bgs)
    vf = engine.register_bank(L.BANK_VOICE, voices, labels=labels)
    nf = engine.register_bank(L.BANK_NOISE, noises)
    return (bf, vf, nf), [engine.voice_activity(i) for i in range(len(voices))]


def _outputs(engine, d, modes):
    """Frame labels, keep flags and the features of `modes` of plan `d` (host copies)."""
    engine.upload_plan(d)
    frame, _, keep = engine.labels()
    return [_np(frame), _np(keep)] + [_np(engine.features(m)) for m in modes]


def _per_item(engine, items, rates):
    """The route this replaces: Engine.resample of every item, back on the host."""
    return [_np(engine.resample(w, r)) for w, r in zip(items, rates)]


def _clip_frames(T, voice_frames):
    """The first clip length from T on that no voice has: a voice of exactly T frames leaves its offset the
    empty range the reference raises on (pipeline.py:68-69)."""
    while T in set(int(f) for f in voice_frames):
        T += 1
    return T


def _plan(seed, frames, B=4, T=90):
    from challenge_b200.plan import draw_batch
    bf, vf, nf = frames
    return draw_batch(np.random.default_rng(seed), B, _clip_frames(T, vf), bf, vf, nf, max_voices=4,
                      max_noises=2, n_time_masks=6, n_freq_masks=1)


def _bits_equal(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _check_against_per_item(engine, banks, rates):
    """Register `banks` from (wav, rate) items and from the per-item resampled arrays: same frame counts
    (1 + iris_resample_len // 256), same activity, same COMPLEX features bit for bit."""
    from challenge_b200 import _lib as L
    bgs, voices, labels, noises = banks
    r_bg, r_v, r_n = rates
    frames, act = _register(engine, list(zip(bgs, r_bg)), list(zip(voices, r_v)), labels, list(zip(noises, r_n)))
    for f, items, rs in zip(frames, (bgs, voices, noises), rates):
        want = [1 + int(engine.lib.iris_resample_len(w.shape[1], int(r), 16000)) // 256 for w, r in zip(items, rs)]
        assert f.tolist() == want
    d = _plan(int(sum(frames[0])), frames)
    got = _outputs(engine, d, (L.FEAT_COMPLEX,))
    frames2, act2 = _register(engine, _per_item(engine, bgs, r_bg), _per_item(engine, voices, r_v), labels,
                              _per_item(engine, noises, r_n))
    assert all(a.tolist() == b.tolist() for a, b in zip(frames, frames2))
    assert all(np.array_equal(a, b) for a, b in zip(act, act2))
    ref = _outputs(engine, d, (L.FEAT_COMPLEX,))
    assert all(_bits_equal(a, b) for a, b in zip(got, ref))


@pytest.mark.parametrize('n_chan', [1, 2, 3, 4])
@pytest.mark.parametrize('rate', RATES)
def test_bank_from_audio_is_the_per_item_route(engine, rate, n_chan):
    banks = _banks(rate + n_chan, n_chan, rate)
    _check_against_per_item(engine, banks, tuple([rate] * len(b) for b in (banks[0], banks[1], banks[3])))


def test_bank_of_mixed_rates_keeps_item_order(engine):
    """Five rates and 16 kHz items in one bank: each item gets its own filter, the bank keeps their order."""
    rng = np.random.default_rng(3)
    mix = (44100, 16000, 48000, 22050, 16000, 11025, 32000)
    bgs, voices, labels, noises = [], [], None, []
    for k, r in enumerate(mix):
        b, v, lab, n = _banks(100 + k, 2, r, n_bg=1, n_voice=2, n_noise=1)
        bgs += b
        voices += v
        noises += n
        labels = lab if labels is None else np.concatenate([labels, lab])
    order = rng.permutation(len(voices))        # interleave the rates inside the voice bank
    voices = [voices[i] for i in order]
    labels = labels[order]
    r_v = [mix[i // 2] for i in order]
    _check_against_per_item(engine, (bgs, voices, labels, noises), (list(mix), r_v, list(mix)))


def test_all_16k_audio_call_is_iris_bank_register(engine):
    """iris_bank_register_audio with every rate at 16000 registers what iris_bank_register does, bit for bit."""
    from challenge_b200 import _lib as L
    from challenge_b200.engine import pack_waveforms
    bgs, voices, labels, noises = _banks(9, 2, 16000)
    frames, act = _register(engine, bgs, voices, labels, noises)
    d = _plan(9, frames)
    ref = _outputs(engine, d, (L.FEAT_COMPLEX,))
    lab = np.ascontiguousarray(labels, np.float32)
    for kind, items in ((L.BANK_BG, bgs), (L.BANK_VOICE, voices), (L.BANK_NOISE, noises)):
        packed, offsets, rates, n_chan = pack_waveforms(items)
        assert (rates == 16000).all()
        L.check(engine.lib.iris_bank_register_audio(
            engine._ctx, kind, len(items), n_chan, packed.ctypes.data, offsets.ctypes.data, rates.ctypes.data,
            lab.ctypes.data if kind == L.BANK_VOICE else None, 3 if kind == L.BANK_VOICE else 0, 1,
            engine._stream()))
    for kind, f in zip((L.BANK_BG, L.BANK_VOICE, L.BANK_NOISE), frames):
        got = np.zeros(len(f), np.int32)
        L.check(engine.lib.iris_bank_info(engine._ctx, kind, None, None, got.ctypes.data))
        assert got.tolist() == f.tolist()
    assert all(np.array_equal(engine.voice_activity(i), a) for i, a in enumerate(act))
    got = _outputs(engine, d, (L.FEAT_COMPLEX,))
    assert all(_bits_equal(a, b) for a, b in zip(got, ref))


def test_bank_from_audio_agrees_with_load_wav(engine, mods):
    """The template of test_gpu_specbank.py::test_specbank_agrees_with_waveform_path at 44.1 kHz: a waveform
    bank of (wav, 44100) items through the fused FFT kernel, and the spectrogram bank of load_wav((wav, 44100))
    of the same items through the spectrogram-domain mix, under the same draws."""
    from challenge_b200 import _lib as L
    D = mods[2]
    engine.set_mel(80)
    bgs, voices, labels, noises = _banks(5, 2, 44100, n_bg=3, n_voice=8, n_noise=4, bg_seconds=4.0)
    tup = lambda xs: [(w, 44100) for w in xs]      # noqa: E731
    (bf, vf, nf), _ = _register(engine, tup(bgs), tup(voices), labels, tup(noises))
    d = _plan(12, (bf, vf, nf), B=6, T=200)
    modes = (L.FEAT_COMPLEX, L.FEAT_LOGMEL_MINMAX)
    frame_w, keep_w, *out_w = _outputs(engine, d, modes)
    spec = lambda xs: [_np(D.load_wav((w, 44100))) for w in xs]      # noqa: E731
    (bf2, _, _), _ = _register(engine, spec(bgs), spec(voices), labels, spec(noises))
    assert bf2.tolist() == bf.tolist()
    frame_s, keep_s, *out_s = _outputs(engine, d, modes)
    assert np.array_equal(frame_s, frame_w) and np.array_equal(keep_s, keep_w)
    for s, w, tol in zip(out_s, out_w, (2e-6, 1e-4)):
        assert nmax_err(s, w) <= tol


def test_make_pipeline_and_merge_complex_specs_take_audio_items(engine, mods):
    """make_pipeline with the sj_train chain on (wav, rate) banks yields, under the same seed, what it yields
    on the per-item resampled arrays; so does merge_complex_specs."""
    import torch
    from challenge_b200 import _ops as O
    P, TR, D = mods
    rates = (44100, 48000, 16000)
    bgs, voices, labels, noises = [], [], [], []
    for k, r in enumerate(rates):
        b, v, lab, n = _banks(40 + k, 2, r, n_bg=1, n_voice=4, n_noise=2, bg_seconds=4.0)
        bgs += [(w, r) for w in b]
        voices += [(w, r) for w in v]
        noises += [(w, r) for w in n]
        labels.append(lab)
    labels = np.concatenate(labels)
    arrays = [[_np(engine.resample(w, r)) for w, r in xs] for xs in (bgs, voices, noises)]
    T = _clip_frames(120, [1 + w.shape[1] // 256 for w in arrays[1]])

    def first_batches(banks):
        O.set_seed(21)
        ds = P.make_pipeline(banks[0], banks[1], labels, banks[2], n_frame=T, max_voices=4, max_noises=2,
                             min_ratio=1)
        ds = ds.map(D.to_frame_labels).map(D.augment).map(D.stft_filter(2)).batch(4).map(TR.complex_to_magphase)
        ds = ds.map(TR.magphase_to_mel(80)).map(D.minmax).map(D.log_on_mel)
        return [(x.clone(), y.clone()) for x, y in ds.take(2)]

    for (xa, ya), (xb, yb) in zip(first_batches((bgs, voices, noises)), first_batches(arrays)):
        assert torch.equal(xa, xb) and torch.equal(ya, yb)

    def merged(bg, vs, ns):
        O.set_seed(5)
        return P.merge_complex_specs(bg, (vs, labels[:3]), ns, n_frame=_clip_frames(60, [1 + w.shape[1] // 256
                                                                                       for w in arrays[1][:3]]))

    xa, ya = merged(bgs[0], voices[:3], noises[:2])
    xb, yb = merged(arrays[0][0], arrays[1][:3], arrays[2][:2])
    assert torch.equal(xa, xb) and torch.equal(ya, yb)


def test_bank_from_audio_errors(engine):
    from challenge_b200 import _lib as L
    rng = np.random.default_rng(1)
    w = (rng.standard_normal((2, 44100)) * 0.1).astype(np.float32)
    with pytest.raises(ValueError):
        engine.register_bank(L.BANK_BG, [(w, 44100), (w, 0)])
    with pytest.raises(NotImplementedError, match='filter bank above 32 MB'):
        engine.register_bank(L.BANK_BG, [(w, 1000003)])
    short = w[:, :700]                                  # 234 samples at 16 kHz
    assert engine.lib.iris_resample_len(700, 48000, 16000) <= 256
    with pytest.raises(ValueError, match='reflect padding'):
        engine.register_bank(L.BANK_BG, [(w, 48000), (short, 48000)])
    engine.register_bank(L.BANK_BG, [(w[:, :771], 48000)])   # 257 samples at 16 kHz: the shortest item
    with pytest.raises(AssertionError):
        engine.register_bank(L.BANK_BG, [(w, 44100), (w[:1], 44100)])
