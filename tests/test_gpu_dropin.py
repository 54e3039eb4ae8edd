"""GPU tests of the drop-in modules (challenge_b200.{pipeline,transforms,data_utils,metrics}):
the reference's own unit tests restated against the same function names (known answers in
tests/golden/reference_kats.json, transcribed from transforms_test.py / metrics_test.py /
pipeline_test.py), plus parity of every stand-alone stage with the CPU oracle."""
import json
import os

import numpy as np
import pytest

from conftest import nmax_err, phase_err

pytestmark = pytest.mark.gpu

KATS = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'reference_kats.json')))


def _np(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope='module')
def mods(engine):
    import challenge_b200
    from challenge_b200 import data_utils, engine as E, metrics, pipeline, transforms
    E._engines[0] = engine          # share the session engine
    challenge_b200.set_seed(0)
    return pipeline, transforms, data_utils, metrics


# ---- transforms_test.py ----
def test_mask(mods):
    _, TR, _, _ = mods
    for key in ('mask_axis0', 'mask_axis1'):
        k = KATS[key]
        got = TR.mask(np.array(k['org'], np.float32), axis=k['axis'],
                      max_mask_size=k['max_mask_size'], n_mask=k['n_mask'], draws=k['draws'])
        assert np.array_equal(_np(got), np.array(k['target'], np.float32))
    # random draws stay inside the reference's ranges and zero whole rows
    x = np.random.default_rng(0).standard_normal((257, 100, 4)).astype(np.float32)
    got = _np(TR.mask(x, axis=-2, max_mask_size=24, n_mask=6))
    cols = ~got.any(axis=(0, 2))
    assert cols.sum() < 6 * 24 and np.array_equal(got[:, ~cols], x[:, ~cols])


def test_random_shift(mods):
    _, TR, _, _ = mods
    k = KATS['random_shift']
    got = TR.random_shift(np.array(k['org'], np.float32), axis=k['axis'], width=k['width'],
                          offset=k['offset'])
    assert np.array_equal(_np(got), np.array(k['target'], np.float32))
    assert _np(TR.random_shift(np.ones((5, 3), np.float32), axis=1, width=2)).shape == (5, 3)


def test_magphase_to_mel(mods):
    from oracle import transforms as OT
    _, TR, _, _ = mods
    rng = np.random.default_rng(1)
    x = rng.random((4, 257, 100, 4), dtype=np.float32)
    got = _np(TR.magphase_to_mel(80)(x))
    assert got.shape == (4, 80, 100, 2)                       # transforms_test.py:45-55
    assert nmax_err(got, OT.magphase_to_mel(80)(x)) < 1e-5
    got = _np(TR.magphase_to_mel(80)(x[0]))
    assert got.shape == (80, 100, 2)
    assert nmax_err(got, OT.magphase_to_mel(80)(x[0])) < 1e-5
    # a matrix the fused epilogue does not take (wide filters) still projects
    got = _np(TR.magphase_to_mel(20, lower_edge_hertz=0.0, upper_edge_hertz=8000.0)(x))
    ref = OT.magphase_to_mel(20, lower_edge_hertz=0.0, upper_edge_hertz=8000.0)(x)
    assert nmax_err(got, ref) < 1e-5
    with pytest.raises(ValueError):
        TR.magphase_to_mel(80)(x[0, :, 0])


def test_log_magphase(mods):
    _, TR, _, _ = mods
    k = KATS['log_magphase']
    got = _np(TR.log_magphase(np.array(k['specs'], np.float32), n_chan=k['n_chan']))
    np.testing.assert_allclose(got, np.array(k['target'], np.float32), rtol=0, atol=1e-6)


def test_minmax_norm_magphase(mods):
    from oracle import transforms as OT
    _, TR, _, _ = mods
    x = np.random.default_rng(2).standard_normal((5, 257, 30, 4)).astype(np.float32) * 7
    got = _np(TR.minmax_norm_magphase(x))
    for half in (got[..., :2], got[..., 2:]):                  # transforms_test.py:64-77
        assert np.allclose(half.reshape(5, -1).min(1), 0) and np.allclose(half.reshape(5, -1).max(1), 1, atol=1e-6)
    assert np.array_equal(got, OT.minmax_norm_magphase(x))       # selections and one formula: bit exact


def test_complex_to_magphase_and_back(mods):
    _, TR, _, _ = mods
    k = KATS['complex_to_magphase']
    c = np.array(k['complex'], np.float32)
    mp = _np(TR.complex_to_magphase(c))
    np.testing.assert_allclose(mp, np.array(k['magphase'], np.float32), rtol=0, atol=1e-6)
    back = _np(TR.magphase_to_complex(np.array(k['magphase'], np.float32)))
    np.testing.assert_allclose(back, c, rtol=0, atol=1e-6)     # transforms_test.py:89-96
    x = np.random.default_rng(3).standard_normal((3, 257, 50, 8)).astype(np.float32)
    from oracle import transforms as OT
    got, ref = _np(TR.complex_to_magphase(x)), OT.complex_to_magphase(x)
    assert nmax_err(got[..., :4], ref[..., :4]) < 1e-6
    assert phase_err(ref[..., :4], got[..., 4:], ref[..., 4:]) < 1e-5
    x2, y = TR.complex_to_magphase(x, 'labels')
    assert y == 'labels'


def test_phase_vocoder_identity(mods):
    _, TR, _, _ = mods
    x = np.ones((257, 100, 6), np.float32)
    assert TR.phase_vocoder(x, rate=1.) is x                    # transforms_test.py:98-101


# ---- data_utils ----
def test_load_wav_and_feature_chain(mods):
    """metrics.evaluate's input side (metrics.py:41-54) on an in-memory waveform, incl. the
    per-mel-row min-max quirk of the unbatched call."""
    from oracle import data_utils as OD, transforms as OT
    _, TR, D, _ = mods
    wav = (np.random.default_rng(4).standard_normal((2, 48000)) * 0.1).astype(np.float32)
    spec = D.load_wav(wav)
    ref = OD.load_wav_array(wav)
    assert nmax_err(_np(spec), ref) < 1e-4
    x = D.stft_filter(16)(spec)
    x = TR.complex_to_magphase(x)
    x = TR.magphase_to_mel(80)(x)
    x = D.minmax(x)
    x = D.log_on_mel(x)
    r = OD.stft_filter(16)(ref)
    r = OT.complex_to_magphase(r)
    r = OT.magphase_to_mel(80)(r)
    r = OD.log_on_mel(OD.minmax(r))
    assert _np(x).shape == r.shape == (80, 188, 2)
    assert nmax_err(_np(x), r) < 1e-4


def test_normalize_runs_on_the_device(mods):
    """data_utils.normalize (data_utils.py:32-34) as iris_op_normalize: the RMS of the whole clip
    (all channels), squares summed in fp64 -- against the oracle's torch fp32 form and a float64 value."""
    from oracle import data_utils as OD
    _, _, D, _ = mods
    rng = np.random.default_rng(11)
    for shape in [(2, 160000), (4, 40001), (1, 300), (3, 7)]:
        wav = (rng.standard_normal(shape) * 0.1).astype(np.float32)
        got = _np(D.normalize(wav))
        assert got.shape == wav.shape
        assert nmax_err(got, OD.normalize(wav)) < 2e-6
        ref64 = wav.astype(np.float64) / (10 * np.sqrt(np.mean(wav.astype(np.float64) ** 2)))
        assert nmax_err(got, ref64) < 5e-7
        assert abs(float(np.sqrt(np.mean(got.astype(np.float64) ** 2))) - 0.1) < 1e-7


def test_minmax_log_labels_and_remaps(mods):
    from oracle import data_utils as OD
    _, _, D, _ = mods
    rng = np.random.default_rng(5)
    x = rng.random((6, 80, 50, 2), dtype=np.float32) * 3
    assert np.array_equal(_np(D.minmax(x)), OD.minmax(x))
    const = np.full((2, 4, 4), 2.5, np.float32)                 # max == min: safe_div path
    assert np.array_equal(_np(D.minmax(const)), OD.minmax(const))
    assert nmax_err(_np(D.log_on_mel(x)), OD.log_on_mel(x)) < 1e-6
    y = (rng.random((3, 7, 40, 3)) < 0.2).astype(np.float32)
    _, got = D.to_frame_labels(None, y)
    assert np.array_equal(_np(got), OD.to_frame_labels(None, y)[1])
    spec = rng.standard_normal((257, 20, 4)).astype(np.float32)
    assert np.array_equal(_np(D.stereo_mono(spec)), OD.stereo_mono(spec))
    got, lab = D.mono_chan(spec, 'y')
    assert lab == 'y' and np.array_equal(_np(got), OD.mono_chan(spec, 'y')[0])
    assert D.mono_chan(spec) is spec                            # no-op without labels (quirk)
    f = np.array([0.3, 0.7], np.float32)
    assert np.array_equal(_np(D.random_merge_aug(4)(spec, factor=f)),
                          OD.random_merge_aug(4)(spec, factor=f))
    assert _np(D.random_merge_aug(5)(spec)).shape == (257, 20, 10)
    with pytest.raises(ValueError):
        D.random_merge_aug(4)(np.zeros((257, 20, 8), np.float32))
    assert np.array_equal(_np(D.stft_filter(3)(spec)), OD.stft_filter(3)(spec))
    _, got = D.multiply_label(3.0)(None, y)
    assert np.array_equal(_np(got), y * 3)
    # speech_enhancement_preprocess (data_utils.py:139-148): values, incl. the quirk that the
    # only_voice / only_noise spectrograms are cut with the width of the ALREADY halved x
    x2 = D.speech_enhancement_preprocess(spec)
    assert _np(x2).shape == (256, 20, 2) and np.array_equal(_np(x2), OD.speech_enhancement_preprocess(spec))
    rng_se = np.random.default_rng(12)
    lab_v = (rng_se.random((5, 20, 3)) < 0.3).astype(np.float32)
    ov = rng_se.standard_normal(spec.shape).astype(np.float32)
    on = rng_se.standard_normal(spec.shape).astype(np.float32)
    gx, gy = D.speech_enhancement_preprocess(spec, (lab_v, ov, on))
    rx, ry = OD.speech_enhancement_preprocess(spec, (lab_v, ov, on))
    assert np.array_equal(_np(gx), rx)
    assert len(gy) == len(ry) == 3
    for g, r in zip(gy, ry):
        assert _np(g).shape == r.shape and np.array_equal(_np(g), r)
    assert ry[0].shape == (20, 3) and ry[1].shape == (256, 20, 1)
    specs, labels = D.augment(spec, 'y')
    assert labels == 'y' and _np(specs).shape == spec.shape


@pytest.mark.parametrize('T,r', [(626, 32), (512, 32), (100, 7), (31, 32), (64, 32)])
def test_label_downsample(mods, T, r):
    from oracle import data_utils as OD
    _, _, D, _ = mods
    rng = np.random.default_rng(T)
    y = (rng.random((40, T, 3)) < 0.5).astype(np.float32)
    _, got = D.label_downsample(r)(None, y)
    _, ref = OD.label_downsample(r)(None, y)
    assert np.array_equal(_np(got), ref) and ref.shape[0] == min(40, r)
    _, got = D.label_downsample(r)(None, (y, 'a', 'b'))
    assert got[1:] == ('a', 'b') and np.array_equal(_np(got[0]), ref)


@pytest.mark.parametrize('orig,n', [(44100, 22051), (48000, 30001), (8000, 9000), (22050, 12345),
                                    (32000, 4000), (16000, 700)])
def test_load_wav_resamples_like_kaldi(mods, orig, n):
    """data_utils.load_wav on audio that is not 16 kHz (data_utils.py:19-22): the kaldi resampler on
    the device against the oracle restatement, then the whole load_wav against the oracle chain."""
    from challenge_b200.engine import get_engine
    from oracle import data_utils as OD
    _, _, D, _ = mods
    rng = np.random.default_rng(orig)
    wav = (rng.standard_normal((2, n)) * 0.1).astype(np.float32)
    ref = OD.resample_waveform(wav, orig, 16000)
    got = _np(get_engine().resample(wav, orig, 16000))
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max()      # fp32 FIR, different summation order
    spec = _np(D.load_wav((wav, orig)))
    ref_spec = OD.load_wav_array(ref)
    assert spec.shape == ref_spec.shape
    assert np.abs(spec - ref_spec).max() <= 1e-4 * np.abs(ref_spec).max()


# ---- metrics_test.py ----
def test_er_score(mods):
    _, _, _, MT = mods
    k = KATS['er_score']
    g = np.zeros([k['batch'], k['frames'], k['classes']], np.float32)
    p = np.zeros_like(g)
    for c, s, e in k['gt']:
        g[:, s:e, c] = 1
    for c, t in k['predict']:
        p[:, t - 2:t + 2, c] = 1
    er = MT.er_score(smoothing=False)(g, p)
    assert float(_np(er).mean()) == np.float32(k['mean_er'])      # metrics_test.py:25
    assert _np(MT.er_counts(g, p)).tolist() == [[5, 5, 2], [5, 5, 2]]


@pytest.mark.parametrize('T', [20, 31, 626, 1000])
def test_er_score_smoothing_pooled_time_base(mods, T):
    """er_score(smoothing=True) (metrics.py:222-224): AveragePooling1D(31, 'same') has stride 31,
    so the predicted events live on ceil(T / 31) frames while the true events keep T; the
    reference matches them by raw frame index and so does iris_er_counts_pooled."""
    from oracle import metrics as OM
    _, _, _, MT = mods
    rng = np.random.default_rng(T)
    B = 24
    yt = np.zeros((B, T, 3), np.float32)
    for b in range(B):                       # a few events per class, some near frame 0 so that
        for c in range(3):                   # pooled midpoints (< ceil(T/31)) can fall inside them
            for _ in range(int(rng.integers(0, 4))):
                s = int(rng.integers(0, max(T // 4, 1)))
                yt[b, s:s + int(rng.integers(1, 30)), c] = 1
    yp = np.clip(yt + rng.normal(0, 0.3, yt.shape), 0, 1).astype(np.float32)
    got = _np(MT.er_score(smoothing=True)(yt, yp))
    ref = OM.er_score(smoothing=True)(yt, yp)
    nt, npd, co = OM.er_parts(yt, yp, 0.5, True)
    assert co.sum() > 0 or T <= 31
    np.testing.assert_array_equal(got, ref)


def test_f1_and_cos_sim(mods):
    from oracle import metrics as OM
    _, _, _, MT = mods
    rng = np.random.default_rng(6)
    yt = (rng.random((16, 200, 3)) < 0.3).astype(np.float32)
    yt[3] = 0                                                    # a sample with no class at all
    yt[5, :, 1] = 0
    yp = np.clip(yt + rng.normal(0, 0.35, yt.shape), 0, 1).astype(np.float32)
    f1, ref = MT.f1_score(), OM.f1_score()
    for _ in range(3):                                           # the state accumulates
        assert f1(yt, yp) == ref(yt, yp)
    assert f1((yt,), (yp,)) == ref((yt,), (yp,))
    got = _np(MT.cos_sim(yt, yp))
    np.testing.assert_allclose(got, OM.cos_sim(yt, yp), rtol=0, atol=2e-6)


# ---- pipeline_test.py ----
def _wave_banks(rng, n_bg, n_voice, n_noise, chan=2, n_classes=30):
    mk = lambda lo, hi: (rng.standard_normal((chan, int(rng.integers(lo, hi)))) * 0.1).astype(np.float32)
    bgs = [mk(2000, 6000) for _ in range(n_bg)]
    voices = [mk(1500, 5000) for _ in range(n_voice)]
    for v in voices[::2]:
        v[:, -v.shape[1] // 4:] = 0                              # zero tails (pipeline_test.py:21-24)
    labels = np.eye(n_classes, dtype=np.float32)[rng.integers(0, n_classes, n_voice)]
    noises = [mk(1500, 5000) for _ in range(n_noise)]
    return bgs, voices, labels, noises


def test_merge_complex_specs(mods):
    """pipeline_test.py:13-42: [257, n_frame, chan*2] and [n_voices, n_frame, n_classes];
    values against the oracle on the same draws."""
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    from oracle import chain
    P, _, _, _ = mods
    rng = np.random.default_rng(7)
    bgs, voices, labels, noises = _wave_banks(rng, 1, 4, 2)
    spec, label = P.merge_complex_specs(bgs[0], (voices, labels), noises, n_frame=10, n_classes=30)
    assert _np(spec).shape == (257, 10, 4) and _np(label).shape == (4, 10, 30)
    eng = mods[1].get_engine()
    frames = lambda ws: np.array([1 + w.shape[1] // 256 for w in ws], np.int32)
    d = draw_batch(np.random.default_rng(8), 1, 10, frames(bgs), frames(voices), frames(noises),
                   max_voices=4, max_noises=2)
    d.voice_id[:] = np.arange(4)
    d.noise_id[:] = np.arange(2)
    spec, label = P.merge_complex_specs(bgs[0], (voices, labels), noises, n_frame=10, n_classes=30,
                                        draws=d)
    ob, ov, on = chain.OracleBank(bgs), chain.OracleBank(voices), chain.OracleBank(noises)
    ref, ref_l = chain.synth_clip(ob, ov, labels, on, d, 0, n_classes=30)
    assert nmax_err(_np(spec), ref) < 1e-4
    assert np.array_equal(_np(label), ref_l)


def test_make_pipeline_and_dataset_chain(mods):
    """pipeline_test.py:44-74 shapes, then sj_train.make_dataset's chain (sj_train.py:107-123)
    fused vs the same functions applied one by one on the un-fused output."""
    import challenge_b200
    P, TR, D, _ = mods
    rng = np.random.default_rng(9)
    bgs, voices, labels, noises = _wave_banks(rng, 30, 40, 50, n_classes=30)
    ds = P.make_pipeline(bgs, voices, labels, noises, n_frame=30, max_voices=4, max_noises=4,
                         n_classes=30)
    for s, l in ds.take(2):
        assert _np(s).shape == (257, 30, 4) and _np(l).shape == (4, 30, 30)
    bgs, voices, labels, noises = _wave_banks(rng, 6, 20, 8, n_classes=3)

    def build(fuse):
        challenge_b200.set_seed(123)
        ds = P.make_pipeline(bgs, voices, labels, noises, n_frame=40, max_voices=4, max_noises=2,
                             n_classes=3, snr=-20, min_ratio=1)
        ds = ds.map(D.to_frame_labels)
        if fuse:
            ds = ds.batch(5).map(TR.complex_to_magphase).map(TR.magphase_to_mel(80))
            return ds.map(D.minmax).map(D.log_on_mel).prefetch(P.AUTOTUNE)
        ident = lambda x, y: (x, y)                              # breaks the fusion
        ds = ds.batch(5).map(ident).map(TR.complex_to_magphase).map(TR.magphase_to_mel(80))
        return ds.map(D.minmax).map(D.log_on_mel)

    fused, rest = build(True)._lower()
    assert rest == []
    assert len(build(False)._lower()[1]) == 5
    (xa, ya), = list(build(True).take(1))
    (xb, yb), = list(build(False).take(1))
    assert _np(xa).shape == (5, 80, 40, 2) and _np(ya).shape == (5, 40, 3)
    assert np.array_equal(_np(ya), _np(yb))
    assert nmax_err(_np(xa), _np(xb)) < 1e-4


# ---- trainer.py label variants + the legacy trainer's dataset chain (SURVEY.md 8f rank 4) ----
def test_trainer_label_variants(mods):
    from challenge_b200 import trainer as TRN
    from oracle import trainer as OT
    rng = np.random.default_rng(3)
    for T in (626, 300, 33, 1):
        y = (rng.random((4, T, 3)) < 0.3).astype(np.float32) * rng.integers(1, 4, (4, T, 3)).astype(np.float32)
        _, got = TRN.preprocess_labels(0.25)(None, y)
        _, ref = OT.preprocess_labels(0.25)(None, y)
        assert _np(got).shape == ref.shape and np.array_equal(_np(got), ref)
    lab = np.zeros((5, 7, 200, 3), np.float32)
    for b in range(5):
        for v in range(int(rng.integers(1, 7))):
            lo = int(rng.integers(0, 150))
            lab[b, v, lo:lo + int(rng.integers(1, 50)), int(rng.integers(0, 3))] = 1
    _, got = TRN.to_density_labels(None, lab)
    _, ref = OT.to_density_labels(None, lab)
    assert np.array_equal(_np(got), ref)
    assert np.allclose(_np(got).sum(axis=(1, 2)), (lab.sum(axis=(2, 3)) > 0).sum(axis=1))   # each voice integrates to 1
    _, got1 = TRN.to_density_labels(None, lab[0])                # unbatched element, as in the dataset map
    assert np.array_equal(_np(got1), ref[0])
    mel = rng.random((3, 80, 50, 2)).astype(np.float32)
    assert nmax_err(_np(TRN.minmax_log_on_mel(mel)), OT.minmax_log_on_mel(mel)) <= 1e-6


def test_trainer_make_dataset_on_pickled_banks(mods, tmp_path):
    """trainer.make_dataset (trainer.py:107-141) on banks written in the reference's file format
    (utils.load_data: pickled spectrogram lists, .npy integer labels with the `// 10` folding)."""
    import types
    from challenge_b200 import trainer as TRN, utils as U
    rng = np.random.default_rng(4)
    spec = lambda t: rng.standard_normal((257, t, 4)).astype(np.float32)
    U.save_bank(str(tmp_path / 'bg.pickle'), [spec(int(rng.integers(40, 90))) for _ in range(4)])
    U.save_bank(str(tmp_path / 'voice.pickle'), [spec(int(rng.integers(5, 30))) for _ in range(9)])
    U.save_bank(str(tmp_path / 'noise.pickle'), [spec(int(rng.integers(5, 30))) for _ in range(5)])
    np.save(str(tmp_path / 'labels.npy'), rng.integers(0, 3, 9) * 10 + rng.integers(0, 10, 9))
    assert len(U.load_data(str(tmp_path / 'bg.pickle'))) == 4
    with pytest.raises(ValueError):
        U.load_data(str(tmp_path / 'bank.txt'))
    cfg = types.SimpleNamespace(datapath=str(tmp_path), background_sounds='bg.pickle', voices='voice.pickle',
                                labels='labels.npy', noises='noise.pickle', n_classes=3, n_frame=64,
                                max_voices=4, max_noises=3, snr=-20, batch_size=3, n_mels=80, multiplier=10)
    ds = TRN.make_dataset(cfg, training=True)
    fused, rest = ds._lower()
    from challenge_b200 import _lib as L
    assert fused['mode'] == L.FEAT_LOGMEL_MINMAX and fused['augment']
    n = 0
    for x, y in ds.take(2):
        assert tuple(x.shape) == (3, 80, 64, 2) and tuple(y.shape) == (3, 2, 3)
        xs = _np(x)
        assert np.isfinite(xs).all() and xs.max() <= 1e-6 and xs.min() >= np.log(1e-8) - 1e-3
        assert np.all(_np(y) >= 0)
        n += 1
    assert n == 2


def test_phase_vocoder(mods):
    """transforms_test.py:98-109 restated (identity at rate 1, output shapes) plus values against
    the oracle restatement of transforms.py:137-195."""
    from oracle import transforms as OT
    _, TR, _, _ = mods
    rng = np.random.default_rng(8)
    n_freq, time, chan2 = 257, 100, 6
    spec = rng.standard_normal((n_freq, time, chan2)).astype(np.float32)
    assert TR.phase_vocoder(spec, 1.) is spec
    for rate in (1.2, 0.8, 2.0, 0.5):
        pv = _np(TR.phase_vocoder(spec, rate=rate))
        assert pv.shape == (n_freq, int(np.ceil(time / rate)), chan2)
        ref = OT.phase_vocoder(spec, rate)
        C = chan2 // 2
        # magnitudes are a plain interpolation: tight.  The accumulated phase of bin f grows by
        # ~pi * f per step (tf.cumsum in float32, transforms.py:186): at f = 256 it reaches 1e4..1e5
        # rad, where ONE float32 ulp is 1e-3..8e-3 rad, so a last-bit difference in any atan2 of the
        # chain is visible at that level in cos / sin of the sum -- in the reference itself too.
        # Bin 0 (small sums) must agree tightly, the whole tensor to two ulps of the largest
        # accumulated phase (pi * 256 * steps): once two float32 running sums differ in the last bit,
        # their later roundings are independent.
        assert nmax_err(np.hypot(pv[..., :C], pv[..., C:]), np.hypot(ref[..., :C], ref[..., C:])) <= 1e-6
        assert np.abs(pv[:1] - ref[:1]).max() <= 5e-5 * np.abs(ref).max()     # bin 0: no phase advance
        acc_max = np.pi * 256 * pv.shape[1]
        ulp = 2.0 ** (np.floor(np.log2(acc_max)) - 23)
        assert nmax_err(pv, ref) <= max(1e-4, 2 * ulp)
        assert np.median(np.abs(pv - ref)) <= 1e-5 * np.abs(ref).max()            # and typically far closer
