"""Mel features behind a channel remap (stereo_mono / random_merge_aug(n)), fused into the feature
kernels of both bank formats: values against the CPU oracle (oracle.chain.dataset_batch), bfloat16 /
float16 as the rounded float32 output, the fused path against the old composition on the same plan,
iris_step with the metric leg, DLPack shapes and IrisDataset."""
import numpy as np
import pytest

from conftest import nmax_err

pytestmark = pytest.mark.gpu

TOL = 1e-4          # MEL / LOGMEL: normalised max error (DESIGN.md §5)
MINMAX_TOL = 2e-4   # LOGMEL_MINMAX: absolute
REMAPS = [('stereo_mono', 3), ('merge_aug', 3), ('merge_aug', 4), ('merge_aug', 5), ('merge_aug', 8),
          ('merge_aug', 16)]
MODES = [('FEAT_MEL', 'mel'), ('FEAT_LOGMEL', 'logmel'), ('FEAT_LOGMEL_MINMAX', 'logmel_minmax')]


def _remap_kw(remap, n):
    from challenge_b200 import _lib as L
    return dict(chan_remap=L.REMAP_STEREO_MONO if remap == 'stereo_mono' else L.REMAP_MERGE_AUG, n_out_chan=n)


def _check(got, ref, name):
    assert got.shape == ref.shape, (got.shape, ref.shape)
    if name == 'logmel_minmax':
        err = float(np.abs(got.astype(np.float64) - ref).max())
        assert err < MINMAX_TOL, err
    elif name == 'logmel':     # compared in the linear domain like the other log features
        assert nmax_err(np.exp(got), np.exp(ref)) < TOL
    else:
        assert nmax_err(got, ref) < TOL


def _rounded_equal(half, f32):
    import torch
    return half.shape == f32.shape and bool(torch.equal(half.view(torch.int16), f32.to(half.dtype).view(torch.int16)))


def _check_halves(engine, mode, ref32):
    import torch
    for dt in (torch.bfloat16, torch.float16):
        assert _rounded_equal(engine.features(mode, dtype=dt), ref32), (mode, dt)


@pytest.mark.parametrize('upper', [3800.0, 7600.0])   # NJ = 4 and NJ = 8 instances
@pytest.mark.parametrize('remap,n', REMAPS)
def test_waveform_banks_against_the_oracle(engine, workload_factory, remap, n, upper):
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    from oracle import chain, transforms as OT
    w = workload_factory(2)
    d = draw_batch(np.random.default_rng(n), 3, 300, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=5,
                   max_noises=2, snr=-20, min_ratio=2 / 3, n_time_masks=6, n_freq_masks=1, merge_extra=n - 2)
    try:
        engine.set_mel(80, upper_edge_hertz=upper)
        assert engine.mel_fusable()
        engine.upload_plan(d, stft_filter=3, **_remap_kw(remap, n))
        engine.labels()
        for mode, name in MODES:
            got = engine.features(getattr(L, mode))
            assert tuple(got.shape) == (3, 80, 300, n)
            ref = chain.dataset_batch(w.o_bg, w.o_voice, w.labels, w.o_noise, d, mode=name, remap=remap,
                                      n_out_chan=n, stft_filter=3,
                                      mel_fn=OT.magphase_to_mel(80, upper_edge_hertz=upper))[0]
            _check(got.cpu().numpy(), ref, name)
            _check_halves(engine, getattr(L, mode), got)
    finally:
        engine.set_mel(80)


def _spec_banks(seed, chan2=4, n_bg=4, n_voice=10, n_noise=5):
    rng = np.random.default_rng(seed)

    def spec(t):
        return rng.standard_normal((257, t, chan2)).astype(np.float32)
    bgs = [spec(int(rng.integers(40, 160))) for _ in range(n_bg)]
    voices = [spec(int(rng.integers(5, 50))) for _ in range(n_voice)]
    labels = np.eye(3, dtype=np.float32)[rng.integers(0, 3, n_voice)]
    noises = [spec(int(rng.integers(5, 50))) for _ in range(n_noise)]
    return bgs, voices, labels, noises


@pytest.mark.parametrize('remap,n', REMAPS)   # c_out = 16 takes the many-channel fallback
def test_spectrogram_banks_against_the_oracle(engine, remap, n):
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    from oracle import chain
    engine.set_mel(80)
    bgs, voices, labels, noises = _spec_banks(60 + n)
    bf = engine.register_bank(L.BANK_BG, bgs)
    vf = engine.register_bank(L.BANK_VOICE, voices, labels=labels)
    nf = engine.register_bank(L.BANK_NOISE, noises)
    d = draw_batch(np.random.default_rng(n), 4, 64, bf, vf, nf, max_voices=4, max_noises=3, min_ratio=2 / 3,
                   n_time_masks=6, n_freq_masks=1, merge_extra=n - 2)
    engine.upload_plan(d, stft_filter=3, **_remap_kw(remap, n))
    engine.labels()
    for mode, name in MODES:
        got = engine.features(getattr(L, mode))
        ref = chain.dataset_batch(bgs, voices, labels, noises, d, mode=name, remap=remap, n_out_chan=n,
                                  stft_filter=3)[0]
        _check(got.cpu().numpy(), ref, name)
        _check_halves(engine, getattr(L, mode), got)


@pytest.mark.parametrize('chan2', [6, 8, 26])   # 3, 4 and 13 channels: all in the fused k_specmix<FM_MEL>
def test_spectrogram_banks_without_a_remap_keep_their_channels(engine, chan2):
    """Without a remap c_out is the bank's channel count: a bank of more than 2 channels (more than one input
    pair) parks and projects its own channels only."""
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    from oracle import chain
    engine.set_mel(80)
    bgs, voices, labels, noises = _spec_banks(90 + chan2, chan2=chan2)
    bf = engine.register_bank(L.BANK_BG, bgs)
    vf = engine.register_bank(L.BANK_VOICE, voices, labels=labels)
    nf = engine.register_bank(L.BANK_NOISE, noises)
    d = draw_batch(np.random.default_rng(chan2), 4, 64, bf, vf, nf, max_voices=4, max_noises=3, min_ratio=2 / 3,
                   n_time_masks=6, n_freq_masks=1)
    engine.upload_plan(d, stft_filter=3)
    engine.labels()
    for mode, name in MODES:
        got = engine.features(getattr(L, mode))
        assert tuple(got.shape) == (4, 80, 64, chan2 // 2)
        ref = chain.dataset_batch(bgs, voices, labels, noises, d, mode=name, stft_filter=3)[0]
        _check(got.cpu().numpy(), ref, name)
        _check_halves(engine, getattr(L, mode), got)


def _old_chain(engine, mode):
    """The composition that ran before the remap was fused: MAGPHASE with the remap -> stand-alone mel
    (iris_op_mel) -> stand-alone min-max -> log, the drop-in stages of data_utils."""
    import torch
    from challenge_b200 import _lib as L, _ops as O
    from challenge_b200 import data_utils as D
    mp = engine.features(L.FEAT_MAGPHASE)
    B, _, T, C2 = mp.shape
    mel = torch.empty((B, engine.n_mel, T, C2 // 2), device='cuda')
    L.check(engine.lib.iris_op_mel(engine._ctx, O.ptr(mp), O.ptr(mel), B, T, C2 // 2, engine._stream()))
    if mode == L.FEAT_LOGMEL_MINMAX:
        mel = D.minmax(mel)
    return mel if mode == L.FEAT_MEL else D.log_on_mel(mel)


@pytest.mark.parametrize('remap,n', [('stereo_mono', 3), ('merge_aug', 4)])
def test_fused_matches_the_old_composition(engine, workload_factory, remap, n):
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    engine.set_mel(80)
    w = workload_factory(2)
    d = draw_batch(np.random.default_rng(5), 8, 626, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=7,
                   max_noises=2, snr=-20, min_ratio=1.0, n_time_masks=6, n_freq_masks=1, merge_extra=n - 2)
    engine.upload_plan(d, stft_filter=3, **_remap_kw(remap, n))
    engine.labels()
    for mode in (L.FEAT_MEL, L.FEAT_LOGMEL_MINMAX):
        new = engine.features(mode).cpu().numpy()
        old = _old_chain(engine, mode).cpu().numpy()
        if mode == L.FEAT_MEL:
            assert nmax_err(new, old) <= 1e-5
        else:
            assert nmax_err(np.exp(new), np.exp(old)) <= 1e-5


def test_step_with_the_metric_leg_and_its_kernels(engine, workload_factory):
    """iris_step with stereo_mono + LOGMEL_MINMAX: features as iris_features on the step's draws, labels and
    counts bit-exact against the same step without a remap, and no stand-alone mel / min-max kernel."""
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_config, uniforms_per_clip
    engine.set_mel(80)
    workload_factory(2)
    B, T = 8, 626
    cfg = draw_config(B, T, 7, 2, -20, 1.0, 0.5, 6, 24, 1, 16)
    u = np.random.default_rng(3).random((B, uniforms_per_clip(cfg)))
    y_pred = torch.rand((B, T, 3), device='cuda', generator=torch.Generator('cuda').manual_seed(5))
    res = {}
    for remap in (L.REMAP_NONE, L.REMAP_STEREO_MONO):
        scfg = engine.step_config(cfg, L.FEAT_LOGMEL_MINMAX, stft_filter=3, chan_remap=remap,
                                  n_out_chan=3 if remap else 0)
        triples = torch.zeros((B, 3), dtype=torch.int32, device='cuda')
        counts = torch.zeros(6, dtype=torch.int64, device='cuda')
        x, frame = engine.step(scfg, u, y_pred=y_pred, triples=triples, counts=counts)
        engine.counts_wait(0)
        torch.cuda.synchronize()
        res[remap] = (x.clone(), frame.clone(), triples.clone(), counts.clone())
    x, f, t, c = res[L.REMAP_STEREO_MONO]
    x0, f0, t0, c0 = res[L.REMAP_NONE]
    assert tuple(x.shape) == (B, 80, T, 3)
    assert torch.equal(f, f0) and torch.equal(t, t0) and torch.equal(c, c0)
    # the step's features are those of iris_features on the step's draws
    d = engine.step_draws(scfg)
    engine.upload_plan(d, stft_filter=3, chan_remap=L.REMAP_STEREO_MONO, n_out_chan=3)
    engine.labels()
    assert torch.equal(engine.features(L.FEAT_LOGMEL_MINMAX), x)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        engine.step(scfg, u)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    assert any('k_fused' in k for k in names), names
    assert not any('mel_project' in k or 'minmax' in k for k in names), names


def test_dlpack_takes_the_remapped_mel_shape(engine, workload_factory):
    import torch
    from torch.utils.dlpack import to_dlpack
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    engine.set_mel(80)
    w = workload_factory(2)
    d = draw_batch(np.random.default_rng(8), 4, 300, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=5,
                   max_noises=2, snr=-20, min_ratio=2 / 3, n_time_masks=6, n_freq_masks=1)
    engine.upload_plan(d, stft_filter=3, chan_remap=L.REMAP_STEREO_MONO, n_out_chan=3)
    engine.labels()
    ref = engine.features(L.FEAT_LOGMEL_MINMAX).clone()
    good = torch.full((4, 80, 300, 3), 7.0, device='cuda')
    engine.features_dlpack(L.FEAT_LOGMEL_MINMAX, to_dlpack(good))
    assert torch.equal(good, ref)
    bad = torch.full((4, 80, 300, 2), 7.0, device='cuda')
    cap = to_dlpack(bad)
    rc = engine.lib.iris_features_dlpack(engine._ctx, L.FEAT_LOGMEL_MINMAX, L.dlpack_pointer(cap), engine._stream())
    torch.cuda.synchronize()
    assert rc == L.IRIS_ERR_INVALID and bool((bad == 7.0).all())


@pytest.mark.parametrize('remap', ['stereo_mono', 'merge_aug'])
def test_iris_dataset_remap_chain(remap):
    """make_pipeline + the INTEGRATION.md §2 chain with a remap + cast_features(torch.bfloat16): one step per
    batch; features match the oracle on the step's draws and labels are exact."""
    import torch
    from challenge_b200 import _ops as O
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import make_pipeline
    from challenge_b200.synth import synthetic_banks
    from oracle import chain
    from oracle.chain import OracleBank
    bgs, voices, labels, noises = synthetic_banks(8, 2, n_bg=3, n_voice=12, n_noise=4, bg_seconds=4.0)
    O.set_seed(77)
    ds = make_pipeline(bgs, voices, labels, noises, n_frame=120, max_voices=4, max_noises=2, min_ratio=1)
    ds = ds.map(D.to_frame_labels).map(D.augment)
    ds = ds.map(D.stereo_mono if remap == 'stereo_mono' else D.random_merge_aug(4))
    ds = ds.map(D.stft_filter(3)).batch(4).map(TR.complex_to_magphase).map(TR.magphase_to_mel(80))
    ds = ds.map(D.minmax).map(D.log_on_mel).map(D.cast_features(torch.bfloat16))
    fused, rest = ds._lower()
    assert rest == []
    eng = ds.engine
    n = 3 if remap == 'stereo_mono' else 4
    for x, y in ds.take(2):
        assert x.dtype == torch.bfloat16 and tuple(x.shape) == (4, 80, 120, n)
        d = eng.step_draws(ds._step_config(fused, 4))
        ref, ref_y, _, _ = chain.dataset_batch(OracleBank(bgs), OracleBank(voices), labels, OracleBank(noises), d,
                                               mode='logmel_minmax', remap=remap, n_out_chan=n, stft_filter=3)
        assert np.array_equal(y.cpu().numpy(), ref_y)
        # bfloat16 keeps 8 significant bits: half an ulp of the value on top of the float32 bar
        got = x.float().cpu().numpy().astype(np.float64)
        assert (np.abs(got - ref) <= 2.0 ** -8 * np.abs(ref) + MINMAX_TOL).all()
