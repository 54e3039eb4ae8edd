"""The batch of the 'se' model (merge_complex_specs(seperate_noise_voice=True) -> speech_enhancement_preprocess,
sj_train.py:99-106) as one feature launch (IRIS_FEAT_SE), in both bank formats: x, only_voice and only_noise
against the CPU oracle (bit-identical for spectrogram banks), masks and stft_filter on x only, empty virtual
pairs, IrisDataset lowering (batched, partial last batch, unbatched, C = 4 kept on the old path), the ABI
rejections and the kernels of one step."""
import numpy as np
import pytest

from conftest import nmax_err

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().cpu().numpy()


def _spec_banks(seed, chan2=4, n_bg=4, n_voice=10, n_noise=5):
    rng = np.random.default_rng(seed)

    def spec(t, tail_zero=False):
        x = rng.standard_normal((257, t, chan2)).astype(np.float32)
        if tail_zero:       # silent frames exercise the activity mask
            x[:, t - int(rng.integers(0, max(t // 3, 1))):] = 0
        return x
    bgs = [spec(int(rng.integers(40, 160))) for _ in range(n_bg)]
    voices = [spec(int(rng.integers(5, 50)), True) for _ in range(n_voice)]
    labels = np.eye(3, dtype=np.float32)[rng.integers(0, 3, n_voice)]
    noises = [spec(int(rng.integers(5, 50))) for _ in range(n_noise)]
    return bgs, voices, labels, noises


def _banks(fmt, n_chan=2, seed=55):
    from challenge_b200.synth import synthetic_banks
    from oracle.chain import OracleBank
    if fmt == 'spec':
        bgs, voices, labels, noises = _spec_banks(seed, chan2=2 * n_chan)
        return (bgs, voices, labels, noises), (bgs, voices, noises)
    bgs, voices, labels, noises = synthetic_banks(seed, n_chan, n_bg=3, n_voice=8, n_noise=4, bg_seconds=3.0)
    return (bgs, voices, labels, noises), (OracleBank(bgs), OracleBank(voices), OracleBank(noises))


def _register(engine, banks, noises=True):
    from challenge_b200 import _lib as L
    bgs, voices, labels, ns = banks
    bf = engine.register_bank(L.BANK_BG, bgs)
    vf = engine.register_bank(L.BANK_VOICE, voices, labels=labels)
    nf = engine.register_bank(L.BANK_NOISE, ns) if noises else None
    return bf, vf, nf


def _oracle(obanks, labels, d, clips=None, stft_filter=0, noises=True):
    """[augment ->] [stft_filter ->] speech_enhancement_preprocess of every clip, stacked."""
    from oracle import chain, data_utils as OD, transforms as OT
    o_b, o_v, o_n = obanks
    xs, fl, vs, ns = [], [], [], []
    for b in (range(d.batch) if clips is None else clips):
        spec, (vtk, ov, on) = chain.synth_clip(o_b, o_v, labels, o_n if noises else None, d, b,
                                               seperate_noise_voice=True)
        if d.time_masks is not None:
            spec = OT.mask(spec, axis=-2, max_mask_size=None, n_mask=d.time_masks.shape[1], draws=d.time_masks[b])
        if d.freq_masks is not None:
            spec = OT.mask(spec, axis=-3, max_mask_size=None, n_mask=d.freq_masks.shape[1], draws=d.freq_masks[b])
        if stft_filter:
            spec = OD.stft_filter(stft_filter)(spec)
        x, (f, v, n) = OD.speech_enhancement_preprocess(spec, (vtk, ov, on))
        xs.append(x)
        fl.append(f)
        vs.append(v)
        ns.append(n)
    return np.stack(xs), np.stack(fl), np.stack(vs), np.stack(ns)


def _check(fmt, got, ref):
    x, v, n = (_np(t) for t in got)
    rx, rv, rn = ref
    assert x.shape == rx.shape and v.shape == rv.shape and n.shape == rn.shape, (x.shape, rx.shape, v.shape, rv.shape)
    if fmt == 'spec':
        assert np.array_equal(x, rx) and np.array_equal(v, rv) and np.array_equal(n, rn)
    else:
        # the bars of test_seperate_noise_voice: only_voice against the size of the mix
        mix = max(np.abs(rx).max(), np.abs(rn).max())
        assert nmax_err(x, rx) <= 1e-5
        assert np.abs(v - rv).max() <= 1e-5 * mix
        assert nmax_err(n, rn) <= 1e-5
        assert not v[rv == 0].any()       # frames no voice reaches: exact zeros (an empty virtual pair)


@pytest.mark.parametrize('fmt', ['spec', 'wave'])
@pytest.mark.parametrize('aug', [False, True])
def test_engine_se_against_the_oracle(engine, fmt, aug):
    """iris_features(IRIS_FEAT_SE): shapes, values, frame labels; with augment + stft_filter(3) x is masked and
    filtered while only_voice / only_noise keep their values, time-masked frames included."""
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    banks, obanks = _banks(fmt)
    bf, vf, nf = _register(engine, banks)
    B, T = 5, 90
    d = draw_batch(np.random.default_rng(13), B, T, bf, vf, nf, max_voices=4, max_noises=3,
                   n_time_masks=6 if aug else 0, n_freq_masks=1 if aug else 0)
    filt = 3 if aug else 0
    engine.upload_plan(d, stft_filter=filt)
    frame, _, _ = engine.labels()
    x, v, n = engine.features(L.FEAT_SE)
    assert tuple(x.shape) == (B, 256, T, 2) and tuple(v.shape) == (B, 256, T, 1) and tuple(n.shape) == (B, 256, T, 1)
    assert x.is_contiguous() and v.is_contiguous() and n.is_contiguous()
    rx, rf, rv, rn = _oracle(obanks, banks[2], d, stft_filter=filt)
    _check(fmt, (x, v, n), (rx, rv, rn))
    assert np.array_equal(_np(frame), rf)
    # only_voice / only_noise are the selected mixes of today's launches, bins 1..256, real part of channel 0
    sv = engine.features(L.FEAT_COMPLEX, select=L.SELECT_VOICES)[:, 1:, :, :1]
    sn = engine.features(L.FEAT_COMPLEX, select=L.SELECT_BG_NOISE)[:, 1:, :, :1]
    if fmt == 'spec':
        assert np.array_equal(_np(v), _np(sv)) and np.array_equal(_np(n), _np(sn))
    if aug:
        masked = [(b, int(o) + i) for b in range(B) for s, o in d.time_masks[b] for i in range(int(s))]
        assert masked
        for b, t in masked:
            assert not _np(x[b, :, t]).any()
        assert any(_np(n[b, :, t]).any() for b, t in masked)   # not masked where x is
        assert not _np(x[:, :filt]).any()                     # bins 1..3


@pytest.mark.parametrize('fmt', ['spec', 'wave'])
def test_empty_virtual_pairs_and_no_noises(engine, fmt):
    """Voices that lie outside the clip (min_ratio ~ 0 pads them by n_frame, offset 0) leave the voice pair
    without stages: only_voice is exactly zero and x is background + noises.  A plan without noises: only_noise
    is the background."""
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    banks, obanks = _banks(fmt, seed=56)
    bf, vf, nf = _register(engine, banks)
    d = draw_batch(np.random.default_rng(3), 4, 64, bf, vf, nf, max_voices=3, max_noises=2, min_ratio=1e-4)
    d.voice_offset[:] = 0
    engine.upload_plan(d)
    engine.labels()
    x, v, n = engine.features(L.FEAT_SE)
    assert not _np(v).any()
    rx, _, rv, rn = _oracle(obanks, banks[2], d)
    assert not rv.any()
    _check(fmt, (x, v, n), (rx, rv, rn))
    # no noise stream
    d = draw_batch(np.random.default_rng(4), 4, 64, bf, vf, None, max_voices=3)
    engine.upload_plan(d)
    engine.labels()
    got = engine.features(L.FEAT_SE)
    rx, _, rv, rn = _oracle(obanks, banks[2], d, noises=False)
    _check(fmt, got, (rx, rv, rn))


def _dataset(fmt, n_chan=2, seed=57):
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import make_pipeline
    banks, obanks = _banks(fmt, n_chan=n_chan, seed=seed)
    ds = make_pipeline(*banks, n_frame=64, max_voices=4, max_noises=3, seperate_noise_voice=True)
    return ds, banks, obanks, D


@pytest.mark.parametrize('fmt', ['spec', 'wave'])
def test_dataset_se_chain(fmt):
    """The sj_train 'se' chain, plain and with augment + stft_filter(3) in front, label_downsample(32) behind,
    a partial last batch (take before batch) and an unbatched dataset: one step per batch, values of the
    oracle on the step's draws."""
    from challenge_b200 import _lib as L
    from challenge_b200 import _ops as O
    from oracle import data_utils as OD
    O.set_seed(5)
    ds0, banks, obanks, D = _dataset(fmt)
    eng = ds0.engine
    chains = [(ds0.map(D.speech_enhancement_preprocess).batch(3).map(D.label_downsample(32)), 3, 0, 2),
              (ds0.map(D.augment).map(D.stft_filter(3)).map(D.speech_enhancement_preprocess).batch(3)
               .map(D.label_downsample(32)), 3, 3, 2),
              (ds0.map(D.speech_enhancement_preprocess).take(5).batch(3), 3, 0, None),
              (ds0.map(D.speech_enhancement_preprocess), None, 0, 2)]
    for ds, B, filt, take in chains:
        fused, rest = ds._lower()
        assert fused['mode'] == L.FEAT_SE
        sizes = []
        for x, y in (ds.take(take) if take else ds):
            b = x.shape[0] if B else 1
            sizes.append(b)
            d = eng.step_draws(ds._step_config(fused, b))
            rx, rf, rv, rn = _oracle(obanks, banks[2], d, stft_filter=filt)
            assert isinstance(y, tuple) and len(y) == 3
            if B is None:
                assert tuple(x.shape) == (256, 64, 2) and tuple(y[0].shape) == (64, 3)
                x, y = x[None], (y[0][None], y[1][None], y[2][None])
            _check(fmt, (x, y[1], y[2]), (rx, rv, rn))
            if any(getattr(st, '__name__', '') == '_label_downsample' for st in rest):
                _, ref_y = OD.label_downsample(32)(None, rf)
                assert np.array_equal(_np(y[0]), ref_y)
            else:
                assert np.array_equal(_np(y[0]), rf)
        assert sizes == ([3, 2] if take is None else [B or 1] * take)


def test_four_channel_banks_keep_the_old_path():
    """C = 4: the stage is not absorbed (FEAT_COMPLEX + the per-clip stage) and still matches the oracle; the
    library answers IRIS_FEAT_SE on such a plan with IRIS_ERR_UNSUPPORTED."""
    from challenge_b200 import _lib as L
    ds, banks, obanks, D = _dataset('spec', n_chan=4)
    ds = ds.map(D.speech_enhancement_preprocess).batch(2)
    fused, rest = ds._lower()
    assert fused['mode'] == L.FEAT_COMPLEX and len(rest) == 2
    eng = ds.engine
    for x, y in ds.take(1):
        assert tuple(x.shape) == (2, 256, 64, 4) and tuple(y[1].shape) == (2, 256, 64, 2)
        d = eng.step_draws(ds._step_config(fused, 2))
        rx, rf, rv, rn = _oracle(obanks, banks[2], d)
        _check('spec', (x, y[1], y[2]), (rx, rv, rn))
        assert np.array_equal(_np(y[0]), rf)
    with pytest.raises(NotImplementedError):
        eng.features(L.FEAT_SE)


def test_abi_rejections(engine):
    import torch
    from torch.utils.dlpack import to_dlpack
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    banks, _ = _banks('wave')
    bf, vf, nf = _register(engine, banks)
    d = draw_batch(np.random.default_rng(1), 2, 40, bf, vf, nf, max_voices=3, max_noises=2, merge_extra=2)
    engine.upload_plan(d, chan_remap=L.REMAP_MERGE_AUG, n_out_chan=4)
    with pytest.raises(NotImplementedError):            # a channel remap
        engine.features(L.FEAT_SE)
    engine.upload_plan(d)
    with pytest.raises(ValueError):                     # an IRIS_OUT_* flag
        engine.features(L.FEAT_SE, dtype=torch.bfloat16)
    buf = torch.zeros(2 * 256 * 40 * 4, device='cuda')
    for sel in (L.SELECT_VOICES, L.SELECT_BG_NOISE):
        rc = engine.lib.iris_features_select(engine._ctx, L.FEAT_SE, sel, engine._ptr(buf), engine._stream())
        assert rc == L.IRIS_ERR_INVALID
    for bytes_flag in (0, L.OUT_F16):
        bi, bo = L.C.c_int64(), L.C.c_int64()
        rc = engine.lib.iris_plan_bytes(engine._ctx, L.FEAT_SE | bytes_flag, None, L.C.byref(bi), L.C.byref(bo))
        assert rc == (L.IRIS_OK if not bytes_flag else L.IRIS_ERR_INVALID)
        if not bytes_flag:
            assert bo.value == buf.numel() * 4
    t = torch.full((2, 256, 40, 2), 7.0, device='cuda')
    rc = engine.lib.iris_features_dlpack(engine._ctx, L.FEAT_SE, L.dlpack_pointer(to_dlpack(t)), engine._stream())
    assert rc == L.IRIS_ERR_INVALID
    from challenge_b200.plan import draw_config
    scfg = engine.step_config(draw_config(2, 40, 3, 2, -20, 2 / 3, 0.5, 0, 24, 0, 16, 257, 0), L.FEAT_SE)
    u = np.random.default_rng(0).random((2, 64))
    rc = engine.lib.iris_step_dlpack(engine._ctx, L.C.byref(scfg), u.ctypes.data, None,
                                     L.dlpack_pointer(to_dlpack(t)), None, engine._stream())
    torch.cuda.synchronize()
    assert rc == L.IRIS_ERR_INVALID and bool((t == 7.0).all())


@pytest.mark.parametrize('fmt', ['spec', 'wave'])
def test_step_is_one_feature_launch(engine, fmt):
    """iris_step in IRIS_FEAT_SE: k_labels and one feature kernel (k_fused, whose tile lists k_labels built: no
    k_tiles; k_specmix for spectrogram banks), nothing per clip; the step's output is iris_features' on its draws."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_config, uniforms_per_clip
    banks, _ = _banks(fmt)
    _register(engine, banks)
    B, T = 12, 64
    scfg = engine.step_config(draw_config(B, T, 4, 3, -20, 2 / 3, 0.5, 6, 24, 1, 16, 257, 0), L.FEAT_SE,
                              stft_filter=3)
    u = np.random.default_rng(2).random((B, uniforms_per_clip(scfg.draw)))
    (x, v, n), frame = engine.step(scfg, u)
    torch.cuda.synchronize()
    got = [t.clone() for t in (x, v, n, frame)]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        engine.step(scfg, u)
        torch.cuda.synchronize()
    kernels = [e.key for e in prof.key_averages() if e.device_type.name == 'CUDA' and 'emcpy' not in e.key
               and 'emset' not in e.key]
    counts = {e.key: e.count for e in prof.key_averages() if e.key in kernels}
    feat = 'k_fused' if fmt == 'wave' else 'k_specmix'
    assert len(kernels) == 2, kernels
    assert sum(c for k, c in counts.items() if 'k_labels' in k) == 1, counts
    assert sum(c for k, c in counts.items() if feat in k) == 1, counts
    assert not any('k_tiles' in k for k in kernels), kernels
    d = engine.step_draws(scfg)
    engine.upload_plan(d, stft_filter=3)
    f2, _, _ = engine.labels()
    again = engine.features(L.FEAT_SE)
    assert all(torch.equal(a, b) for a, b in zip(again, got[:3])) and torch.equal(f2, got[3])
