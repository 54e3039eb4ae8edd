"""bfloat16 / float16 features (IRIS_OUT_BF16 / IRIS_OUT_F16): every launch with a flag must give,
bit for bit, the float32 output of the same plan rounded to nearest even (``fp32.to(dtype)``) -- every
mode, channel count and remap, masks and stft_filter, both k_fused epilogue forms, with and without
the tile lists of k_labels, both bank formats (spectrogram banks fused and through the many-channel
fallback), only_voice, iris_step with its metric leg, DLPack and IrisDataset's cast_features."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ['FEAT_COMPLEX', 'FEAT_MAGPHASE', 'FEAT_LOG_MAGPHASE', 'FEAT_MEL', 'FEAT_LOGMEL', 'FEAT_LOGMEL_MINMAX']
DTYPES = ['bfloat16', 'float16']


def _rounded_equal(half, f32):
    """``half`` holds exactly ``f32.to(half.dtype)`` (compared as bit patterns: -0, inf and NaN included)."""
    import torch
    assert half.dtype in (torch.bfloat16, torch.float16) and f32.dtype == torch.float32
    return half.shape == f32.shape and bool(torch.equal(half.view(torch.int16), f32.to(half.dtype).view(torch.int16)))


def _check_modes(engine, modes, select=None):
    """features(mode) in fp32, then in bf16 and f16 on the same uploaded plan."""
    import torch
    from challenge_b200 import _lib as L
    sel = L.SELECT_ALL if select is None else select
    for name in modes:
        m = getattr(L, name)
        ref = engine.features(m, select=sel).clone()
        assert ref.dtype == torch.float32
        for dt in DTYPES:
            got = engine.features(m, select=sel, dtype=getattr(torch, dt))
            assert _rounded_equal(got, ref), (name, dt)


def _plan(w, B, T, V=5, M=2, seed=1, masks=True, merge_extra=0):
    from challenge_b200.plan import draw_batch
    return draw_batch(np.random.default_rng(seed), B, T, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=V,
                      max_noises=M, snr=-20, min_ratio=2 / 3, n_time_masks=6 if masks else 0,
                      n_freq_masks=1 if masks else 0, merge_extra=merge_extra)


@pytest.mark.parametrize('n_chan', [2, 4, 1])
def test_waveform_banks_every_mode_is_the_rounded_fp32_output(engine, workload_factory, n_chan):
    """2 channels (fixed mel epilogues), 4 (spectrogram pair merge), 1 (odd C, generic epilogue); masks and
    stft_filter on; only_voice."""
    from challenge_b200 import _lib as L
    engine.set_mel(80)
    w = workload_factory(n_chan)
    engine.upload_plan(_plan(w, 5, 300, seed=n_chan), stft_filter=3)
    engine.labels()
    _check_modes(engine, MODES)
    _check_modes(engine, ['FEAT_COMPLEX'], select=L.SELECT_VOICES)


@pytest.mark.parametrize('remap', ['stereo_mono', 'merge_aug'])
def test_waveform_channel_remaps_are_the_rounded_fp32_output(engine, workload_factory, remap):
    from challenge_b200 import _lib as L
    w = workload_factory(2)
    n_out = 3 if remap == 'stereo_mono' else 5
    engine.upload_plan(_plan(w, 4, 300, seed=7, merge_extra=n_out - 2 if remap == 'merge_aug' else 0), stft_filter=16,
                       chan_remap=L.REMAP_STEREO_MONO if remap == 'stereo_mono' else L.REMAP_MERGE_AUG,
                       n_out_chan=n_out)
    engine.labels()
    _check_modes(engine, MODES[:3])


@pytest.mark.parametrize('switch', ['IRIS_NO_FIXED_EPI', 'IRIS_NO_LABEL_TILES'])
def test_generic_epilogue_and_k_tiles_paths(engine, workload_factory, monkeypatch, switch):
    """The generic mel epilogue (NJ = 4) instead of the fixed ones, and tile lists built by k_tiles instead
    of k_labels."""
    engine.set_mel(80)
    w = workload_factory(2)
    monkeypatch.setenv(switch, '1')
    engine.upload_plan(_plan(w, 5, 300, seed=11))
    engine.labels()
    _check_modes(engine, MODES)


def test_mel_matrix_above_bin_128_uses_the_wide_instances(engine, workload_factory):
    """A mel matrix reaching bin 191 runs the NJ = 8 mel instances.  (Every filter of this matrix has a
    non-zero weight: the fused epilogue does not write the row of an all-zero filter.)"""
    w = workload_factory(2)
    engine.set_mel(96, upper_edge_hertz=6000.0)
    try:
        assert engine.mel_fusable() and (engine.mel_matrix != 0).any(1).nonzero()[0].max() > 128
        engine.upload_plan(_plan(w, 4, 300, seed=13))
        engine.labels()
        _check_modes(engine, MODES[3:])
    finally:
        engine.set_mel(80)


def _spec_banks(seed, chan2, n_bg=4, n_voice=10, n_noise=5):
    rng = np.random.default_rng(seed)

    def spec(t):
        return rng.standard_normal((257, t, chan2)).astype(np.float32)
    bgs = [spec(int(rng.integers(40, 160))) for _ in range(n_bg)]
    voices = [spec(int(rng.integers(5, 50))) for _ in range(n_voice)]
    labels = np.eye(3, dtype=np.float32)[rng.integers(0, 3, n_voice)]
    noises = [spec(int(rng.integers(5, 50))) for _ in range(n_noise)]
    return bgs, voices, labels, noises


@pytest.mark.parametrize('chan2', [4, 2, 32])   # 2, 1 and 16 channels
def test_spectrogram_banks_every_mode_is_the_rounded_fp32_output(engine, chan2):
    """k_specmix stores the half type itself; 16 channels take the many-channel mel fallback (magnitudes and
    the stand-alone mel / min-max passes in fp32, the last pass converts)."""
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    engine.set_mel(80)
    bgs, voices, labels, noises = _spec_banks(40 + chan2, chan2)
    bf = engine.register_bank(L.BANK_BG, bgs)
    vf = engine.register_bank(L.BANK_VOICE, voices, labels=labels)
    nf = engine.register_bank(L.BANK_NOISE, noises)
    d = draw_batch(np.random.default_rng(chan2), 4, 64, bf, vf, nf, max_voices=4, max_noises=3, min_ratio=2 / 3,
                   n_time_masks=6, n_freq_masks=1)
    engine.upload_plan(d, stft_filter=2)
    engine.labels()
    _check_modes(engine, MODES)
    _check_modes(engine, ['FEAT_COMPLEX'], select=L.SELECT_VOICES)
    if chan2 != 4:   # stereo_mono / merge_aug need 2 channels
        return
    for remap, n_out in ((L.REMAP_STEREO_MONO, 3), (L.REMAP_MERGE_AUG, 4)):
        d = draw_batch(np.random.default_rng(9), 4, 64, bf, vf, nf, max_voices=4, max_noises=3, min_ratio=2 / 3,
                       n_time_masks=6, n_freq_masks=1, merge_extra=n_out - 2 if remap == L.REMAP_MERGE_AUG else 0)
        engine.upload_plan(d, stft_filter=2, chan_remap=remap, n_out_chan=n_out)
        engine.labels()
        _check_modes(engine, MODES[:3])


@pytest.mark.parametrize('dtype', DTYPES)
def test_step_with_a_flag_and_the_metric_leg(engine, workload_factory, dtype):
    """iris_step with IRIS_OUT_*: the features are the rounded fp32 step's, and frame labels, per-clip
    triples and accumulated counts of the metric leg are those of the fp32 step with the same uniforms."""
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_config, uniforms_per_clip
    engine.set_mel(80)
    workload_factory(2)
    B, T = 8, 626
    dt = getattr(torch, dtype)
    cfg = draw_config(B, T, 7, 2, -20, 1.0, 0.5, 6, 24, 1, 16)
    u = np.random.default_rng(3).random((B, uniforms_per_clip(cfg)))
    y_pred = torch.rand((B, T, 3), device='cuda', generator=torch.Generator('cuda').manual_seed(5))
    for mode in (L.FEAT_LOGMEL_MINMAX, L.FEAT_MEL, L.FEAT_COMPLEX):
        res = {}
        for out in (torch.float32, dt):
            scfg = engine.step_config(cfg, mode, out_dtype=out)
            triples = torch.zeros((B, 3), dtype=torch.int32, device='cuda')
            counts = torch.zeros(6, dtype=torch.int64, device='cuda')
            x, frame = engine.step(scfg, u, y_pred=y_pred, triples=triples, counts=counts)
            engine.counts_wait(0)
            torch.cuda.synchronize()
            assert x.dtype == out and frame.dtype == torch.float32
            res[out] = (x.clone(), frame.clone(), triples.clone(), counts.clone())
        (x32, f32, t32, c32), (xh, fh, th, ch) = res[torch.float32], res[dt]
        assert _rounded_equal(xh, x32), mode
        assert torch.equal(fh, f32) and torch.equal(th, t32) and torch.equal(ch, c32), mode


def test_dlpack_half_tensors_and_refusals(engine, workload_factory):
    """bf16 / f16 tensors are filled in place through DLPack (the flag follows the tensor's dtype); a dtype
    that does not match the flag, or both flags at once, is IRIS_ERR_INVALID and leaves the buffer as it
    was."""
    import torch
    from torch.utils.dlpack import to_dlpack
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_config, uniforms_per_clip
    engine.set_mel(80)
    w = workload_factory(2)
    engine.upload_plan(_plan(w, 4, 626, seed=21))
    engine.labels()
    mode = L.FEAT_LOGMEL_MINMAX
    ref = engine.features(mode).clone()
    lib, ctx = engine.lib, engine._ctx
    stream = engine._stream()
    for dt, flag, other in ((torch.bfloat16, L.OUT_BF16, torch.float16), (torch.float16, L.OUT_F16, torch.bfloat16)):
        t = torch.full(ref.shape, 7.0, dtype=dt, device='cuda')
        ptr = t.data_ptr()
        engine.features_dlpack(mode, to_dlpack(t))                     # flag from the dtype
        assert t.data_ptr() == ptr and _rounded_equal(t, ref)
        t.fill_(7.0)
        cap = to_dlpack(t)                  # the capsule owns the DLManagedTensor: keep it alive over the call
        L.check(lib.iris_features_dlpack(ctx, mode | flag, L.dlpack_pointer(cap), stream))
        assert _rounded_equal(t, ref)
        # refusals leave the buffer untouched
        for bad_mode, tensor in ((mode | flag, torch.full(ref.shape, 7.0, dtype=other, device='cuda')),
                                 (mode | flag, torch.full(ref.shape, 7.0, device='cuda')),
                                 (mode, torch.full(ref.shape, 7.0, dtype=dt, device='cuda')),
                                 (mode | L.OUT_BF16 | L.OUT_F16, torch.full(ref.shape, 7.0, dtype=dt, device='cuda')),
                                 (mode | 0x400, torch.full(ref.shape, 7.0, dtype=dt, device='cuda'))):
            cap = to_dlpack(tensor)
            rc = lib.iris_features_dlpack(ctx, bad_mode, L.dlpack_pointer(cap), stream)
            torch.cuda.synchronize()
            assert rc == L.IRIS_ERR_INVALID, (bad_mode, tensor.dtype)
            assert bool((tensor == 7.0).all())
    # both flags through the pointer entry points and iris_step
    buf = torch.full(ref.shape, 7.0, dtype=torch.bfloat16, device='cuda')
    assert lib.iris_features(ctx, mode | L.OUT_BF16 | L.OUT_F16, ctypes.c_void_p(buf.data_ptr()), stream) == \
        L.IRIS_ERR_INVALID
    cfg = draw_config(4, 626, 7, 2, -20, 1.0, 0.5, 6, 24, 1, 16)
    u = np.random.default_rng(4).random((4, uniforms_per_clip(cfg)))
    bad = engine.step_config(cfg, mode | L.OUT_BF16 | L.OUT_F16)
    cap = to_dlpack(buf)
    rc = lib.iris_step_dlpack(ctx, ctypes.byref(bad), u.ctypes.data, None, L.dlpack_pointer(cap), None, stream)
    torch.cuda.synchronize()
    assert rc == L.IRIS_ERR_INVALID
    assert bool((buf == 7.0).all())
    # the whole step through DLPack into a bf16 tensor
    scfg = engine.step_config(cfg, mode)
    x, y = engine.step(scfg, u)
    fx, fy = torch.empty(x.shape, dtype=torch.bfloat16, device='cuda'), torch.empty_like(y)
    engine.step_dlpack(scfg, u, to_dlpack(fx), to_dlpack(fy))
    assert _rounded_equal(fx, x) and torch.equal(fy, y)


def test_iris_dataset_cast_features_is_the_rounded_fp32_chain():
    """make_pipeline + the sj_train chain + cast_features(torch.bfloat16) yields, under the same seed, the
    fp32 chain's x.to(torch.bfloat16) bit for bit and the same labels -- the cast absorbed into the step."""
    import torch
    from challenge_b200 import _ops as O
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import make_pipeline
    from challenge_b200.synth import synthetic_banks
    bgs, voices, labels, noises = synthetic_banks(8, 2, n_bg=3, n_voice=12, n_noise=4, bg_seconds=4.0)

    def chain(cast):
        ds = make_pipeline(bgs, voices, labels, noises, n_frame=120, max_voices=4, max_noises=2, min_ratio=1)
        ds = ds.map(D.to_frame_labels).map(D.augment).map(D.stft_filter(2)).batch(4).map(TR.complex_to_magphase)
        ds = ds.map(TR.magphase_to_mel(80)).map(D.minmax).map(D.log_on_mel)
        return ds.map(D.cast_features(torch.bfloat16)) if cast else ds

    out = {}
    for cast in (False, True):
        O.set_seed(77)
        ds = chain(cast)
        if cast:
            fused, rest = ds._lower()
            assert rest == [] and fused['out_flag'] != 0
        out[cast] = [(x.clone(), y.clone()) for x, y in ds.take(2)]
    for (x32, y32), (xh, yh) in zip(out[False], out[True]):
        assert xh.dtype == torch.bfloat16 and _rounded_equal(xh, x32)
        assert torch.equal(yh, y32)
