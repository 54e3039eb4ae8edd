"""sj_train's n_chan = 1 chain (mono_chan in front of complex_to_magphase -> mel -> minmax -> log_on_mel) fused
into the feature kernels of both bank formats (IRIS_REMAP_MONO_CHAN): every mode against the oracle composition
OD.mono_chan -> OD.stft_filter -> OT.complex_to_magphase -> ... on the same draws, half-precision features as the
rounded float32 ones, IrisDataset against the un-fused path, iris_step / DLPack shapes, the kernels of one step,
and the stand-alone complex_to_magphase of mono_chan's 3 columns."""
import numpy as np
import pytest

from conftest import nmax_err, phase_err, rel_err_gated

pytestmark = pytest.mark.gpu

TOL = 1e-4          # normalised max error (DESIGN.md §5)
PHASE_TOL = 2e-4    # rad, cells with |X| > 1e-3 max|X|
MINMAX_TOL = 2e-4   # LOGMEL_MINMAX through bfloat16: absolute, on top of half an ulp
MODES = ['complex', 'magphase', 'log_magphase', 'mel', 'logmel', 'logmel_minmax']


def _feat(name):
    from challenge_b200 import _lib as L
    return {'complex': L.FEAT_COMPLEX, 'magphase': L.FEAT_MAGPHASE, 'log_magphase': L.FEAT_LOG_MAGPHASE,
            'mel': L.FEAT_MEL, 'logmel': L.FEAT_LOGMEL, 'logmel_minmax': L.FEAT_LOGMEL_MINMAX}[name]


def _oracle(bg, voices, labels, noises, d, mode, stft_filter=3, mel_fn=None):
    """make_pipeline -> to_frame_labels -> augment -> mono_chan -> stft_filter -> batch -> features, on the CPU."""
    from oracle import chain, data_utils as OD, transforms as OT
    spec, y, _, _ = chain.dataset_batch(bg, voices, labels, noises, d, mode='complex')   # masked, 2 channels
    xs = []
    for b in range(d.batch):
        x = OD.mono_chan(spec[b], y[b])[0]
        xs.append(OD.stft_filter(stft_filter)(x) if stft_filter else x)
    x = np.stack(xs).astype(np.float32)
    if mode == 'complex':
        return x, y
    x = OT.complex_to_magphase(x)
    if mode == 'magphase':
        return x, y
    if mode == 'log_magphase':
        return OT.log_magphase(x, n_chan=2), y
    x = (mel_fn or OT.magphase_to_mel(80))(x)
    if mode == 'logmel_minmax':
        x = OD.minmax(x)
    return (x if mode == 'mel' else OD.log_on_mel(x)), y


def _check(got, ref, name, spec_banks):
    assert got.shape == ref.shape, (got.shape, ref.shape)
    if name == 'complex':
        if spec_banks:    # masks, sums and filter in the reference's order and rounding
            assert np.array_equal(got, ref)
        else:
            assert nmax_err(got, ref) < TOL
    elif name in ('magphase', 'log_magphase'):
        mag_ref = ref[..., :2] if name == 'magphase' else np.exp(ref[..., :2])
        mag = got[..., :2] if name == 'magphase' else np.exp(got[..., :2])
        assert nmax_err(mag, mag_ref) < (1e-6 if spec_banks else TOL)
        assert phase_err(mag_ref, got[..., 2:], ref[..., 2:]) < PHASE_TOL
    elif name in ('logmel', 'logmel_minmax'):   # compared in the linear domain like the other log features
        assert nmax_err(np.exp(got), np.exp(ref)) < TOL
        assert nmax_err(got, ref) < TOL
    else:
        assert nmax_err(got, ref) < TOL
        assert rel_err_gated(got, ref) < TOL


def _check_halves(engine, mode, ref32):
    import torch
    for dt in (torch.bfloat16, torch.float16):
        half = engine.features(mode, dtype=dt)
        assert half.shape == ref32.shape
        assert torch.equal(half.view(torch.int16), ref32.to(dt).view(torch.int16)), (mode, dt)


def _spec_banks(seed, n_bg=4, n_voice=10, n_noise=5):
    rng = np.random.default_rng(seed)

    def spec(t):
        return rng.standard_normal((257, t, 4)).astype(np.float32)
    bgs = [spec(int(rng.integers(40, 160))) for _ in range(n_bg)]
    voices = [spec(int(rng.integers(5, 50))) for _ in range(n_voice)]
    labels = np.eye(3, dtype=np.float32)[rng.integers(0, 3, n_voice)]
    noises = [spec(int(rng.integers(5, 50))) for _ in range(n_noise)]
    return bgs, voices, labels, noises


def _labels_exact(engine, ref_y):
    frame, _, _ = engine.labels()
    assert np.array_equal(frame.cpu().numpy(), ref_y)


@pytest.mark.parametrize('upper', [3800.0, 7600.0])   # NJ = 4 (fixed epilogues for the default shape) and NJ = 8
def test_waveform_banks_against_the_oracle(engine, workload_factory, upper):
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    from oracle import transforms as OT
    w = workload_factory(2)
    d = draw_batch(np.random.default_rng(31), 3, 300, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=5,
                   max_noises=2, snr=-20, min_ratio=2 / 3, n_time_masks=6, n_freq_masks=1)
    try:
        engine.set_mel(80, upper_edge_hertz=upper)
        assert engine.mel_fusable()
        engine.upload_plan(d, stft_filter=3, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
        for name in MODES:
            ref, ref_y = _oracle(w.o_bg, w.o_voice, w.labels, w.o_noise, d, name,
                                 mel_fn=OT.magphase_to_mel(80, upper_edge_hertz=upper))
            _labels_exact(engine, ref_y)
            got = engine.features(_feat(name))
            _check(got.cpu().numpy(), ref, name, spec_banks=False)
            _check_halves(engine, _feat(name), got)
    finally:
        engine.set_mel(80)


def test_spectrogram_banks_against_the_oracle(engine):
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    engine.set_mel(80)
    bgs, voices, labels, noises = _spec_banks(71)
    bf = engine.register_bank(L.BANK_BG, bgs)
    vf = engine.register_bank(L.BANK_VOICE, voices, labels=labels)
    nf = engine.register_bank(L.BANK_NOISE, noises)
    d = draw_batch(np.random.default_rng(6), 4, 64, bf, vf, nf, max_voices=4, max_noises=3, min_ratio=2 / 3,
                   n_time_masks=6, n_freq_masks=1)
    engine.upload_plan(d, stft_filter=3, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
    for name in MODES:
        ref, ref_y = _oracle(bgs, voices, labels, noises, d, name)
        _labels_exact(engine, ref_y)
        got = engine.features(_feat(name))
        _check(got.cpu().numpy(), ref, name, spec_banks=True)
        _check_halves(engine, _feat(name), got)
    x = engine.features(L.FEAT_COMPLEX).cpu().numpy()
    assert np.all(x[:, 1:4] == 0)                          # stft_filter(3) on the sums


def test_plan_checks_and_shapes(engine, workload_factory):
    """n_out_chan must be 2 and the banks 2-channel; feature, plan-bytes, iris_step and DLPack shapes follow
    include/iris.h (COMPLEX [B,257,T,3], MAGPHASE [B,257,T,4], mel [B,n_mel,T,2])."""
    import torch
    from torch.utils.dlpack import to_dlpack
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch, draw_config, uniforms_per_clip
    engine.set_mel(80)
    w = workload_factory(2)
    B, T = 4, 200
    d = draw_batch(np.random.default_rng(9), B, T, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=5,
                   max_noises=2, snr=-20, min_ratio=2 / 3, n_time_masks=6, n_freq_masks=1)
    for n_out in (0, 3):
        with pytest.raises(ValueError):
            engine.upload_plan(d, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=n_out)
    engine.upload_plan(d, stft_filter=3, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
    want = {'complex': (B, 257, T, 3), 'magphase': (B, 257, T, 4), 'log_magphase': (B, 257, T, 4),
            'mel': (B, 80, T, 2), 'logmel': (B, 80, T, 2), 'logmel_minmax': (B, 80, T, 2)}
    feats = {}
    for name, shape in want.items():
        feats[name] = engine.features(_feat(name)).clone()
        assert tuple(feats[name].shape) == shape
        _, bo = engine.plan_bytes(_feat(name))
        assert bo == int(np.prod(shape)) * 4
        _, bo = engine.plan_bytes(_feat(name) | L.OUT_BF16)
        assert bo == int(np.prod(shape)) * 2
    # iris_features_dlpack: the right shape is written, a 2C' = 4 COMPLEX tensor is refused untouched
    good = torch.full(want['complex'], 7.0, device='cuda')
    engine.features_dlpack(L.FEAT_COMPLEX, to_dlpack(good))
    assert torch.equal(good, feats['complex'])
    bad = torch.full((B, 257, T, 4), 7.0, device='cuda')
    rc = engine.lib.iris_features_dlpack(engine._ctx, L.FEAT_COMPLEX, L.dlpack_pointer(to_dlpack(bad)),
                                         engine._stream())
    torch.cuda.synchronize()
    assert rc == L.IRIS_ERR_INVALID and bool((bad == 7.0).all())
    # iris_step and iris_step_dlpack
    cfg = draw_config(B, T, 5, 2, -20, 2 / 3, 0.5, 6, 24, 1, 16)
    u = np.random.default_rng(4).random((B, uniforms_per_clip(cfg)))
    for name, shape in want.items():
        scfg = engine.step_config(cfg, _feat(name), stft_filter=3, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
        x, _ = engine.step(scfg, u)
        assert tuple(x.shape) == shape
        x = x.clone()
        t = torch.full(shape, 7.0, device='cuda')
        engine.step_dlpack(scfg, u, to_dlpack(t))
        torch.cuda.synchronize()
        assert torch.equal(t, x), name
    scfg = engine.step_config(cfg, L.FEAT_COMPLEX, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
    bad = torch.full((B, 257, T, 4), 7.0, device='cuda')
    rc = engine.lib.iris_step_dlpack(engine._ctx, L.C.byref(scfg), u.ctypes.data, None,
                                     L.dlpack_pointer(to_dlpack(bad)), None, engine._stream())
    torch.cuda.synchronize()
    assert rc == L.IRIS_ERR_INVALID and bool((bad == 7.0).all())


def test_four_channel_banks_refuse_the_remap(engine, workload_factory):
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    w = workload_factory(4, seed=20203, n_bg=2, n_voice=16, n_noise=4)
    d = draw_batch(np.random.default_rng(2), 2, 100, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=4,
                   max_noises=2, snr=-20, min_ratio=2 / 3)
    with pytest.raises(ValueError):
        engine.upload_plan(d, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)


def _step_kernels(fmt):
    """CUDA kernels (name -> launches, memcpy / memset left out) of one iris_step of the min-max log-mel mono chain
    on a fresh engine, and whether the step's features equal iris_features' on its draws."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from challenge_b200 import _lib as L
    from challenge_b200.engine import Engine
    from challenge_b200.plan import draw_config, uniforms_per_clip
    from challenge_b200.synth import synthetic_banks
    engine = Engine(0)
    engine.set_mel(80)
    if fmt == 'wave':
        bgs, voices, labels, noises = synthetic_banks(8, 2, n_bg=3, n_voice=12, n_noise=4, bg_seconds=4.0)
    else:
        bgs, voices, labels, noises = _spec_banks(72)
    engine.register_bank(L.BANK_BG, bgs)
    engine.register_bank(L.BANK_VOICE, voices, labels=labels)
    engine.register_bank(L.BANK_NOISE, noises)
    B, T = 12, 64
    scfg = engine.step_config(draw_config(B, T, 4, 3, -20, 2 / 3, 0.5, 6, 24, 1, 16), L.FEAT_LOGMEL_MINMAX,
                              stft_filter=3, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
    u = np.random.default_rng(2).random((B, uniforms_per_clip(scfg.draw)))
    x, _ = engine.step(scfg, u)
    torch.cuda.synchronize()
    got = x.clone()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        engine.step(scfg, u)
        torch.cuda.synchronize()
    counts = {e.key: e.count for e in prof.key_averages() if e.device_type.name == 'CUDA'
              and 'emcpy' not in e.key and 'emset' not in e.key}
    d = engine.step_draws(scfg)
    engine.upload_plan(d, stft_filter=3, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
    engine.labels()
    return counts, bool(torch.equal(engine.features(L.FEAT_LOGMEL_MINMAX), got))


@pytest.mark.parametrize('fmt', ['wave', 'spec'])
def test_step_is_one_feature_launch(fmt):
    """iris_step of the min-max log-mel mono chain: k_labels, one feature kernel (k_fused without k_tiles, or
    k_specmix) and k_logmel_post; no stand-alone op.  The profile is taken in a process of its own, so that this
    test adds no profiler session to the test process."""
    import json
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    code = ('import json, sys; sys.path[:0] = [%r, %r]; import test_gpu_mono_chain as T; '
            'c, same = T._step_kernels(%r); print(json.dumps([c, same]))' % (os.path.dirname(here), here, fmt))
    flags = ['-s'] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable] + flags + ['-c', code], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    counts, same = json.loads(r.stdout.strip().splitlines()[-1])
    feat = 'k_fused' if fmt == 'wave' else 'k_specmix'
    assert sum(c for k, c in counts.items() if 'k_labels' in k) == 1, counts
    assert sum(c for k, c in counts.items() if feat in k) == 1, counts
    assert sum(c for k, c in counts.items() if 'k_logmel_post' in k) == 1, counts
    assert len(counts) == 3, counts
    assert same


def test_iris_dataset_mono_chain_matches_the_unfused_path():
    """make_pipeline + sj_train's n_chan = 1 chain + cast_features(torch.bfloat16): one step per batch.  The same
    chain with mono_chan hidden from the lowering (so that it and every stage behind it run un-fused, per element
    and stand-alone) gets the same draws: labels are identical, both feature sets match the oracle."""
    import torch
    from challenge_b200 import _ops as O
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import make_pipeline
    from challenge_b200.synth import synthetic_banks
    from oracle.chain import OracleBank
    bgs, voices, labels, noises = synthetic_banks(8, 2, n_bg=3, n_voice=12, n_noise=4, bg_seconds=4.0)

    def dataset(mono):
        O.set_seed(78)
        ds = make_pipeline(bgs, voices, labels, noises, n_frame=120, max_voices=4, max_noises=2, min_ratio=1)
        ds = ds.map(D.to_frame_labels).map(D.augment).map(mono).map(D.stft_filter(3)).batch(4)
        ds = ds.map(TR.complex_to_magphase).map(TR.magphase_to_mel(80)).map(D.minmax).map(D.log_on_mel)
        return ds.map(D.cast_features(torch.bfloat16))

    # one dataset after the other: both draw from the seeded host generator in the same order
    fused_ds = dataset(D.mono_chan)
    fused, rest = fused_ds._lower()
    assert rest == []
    batches = []
    for x, y in fused_ds.take(2):
        batches.append((x.clone(), y.clone(), fused_ds.engine.step_draws(fused_ds._step_config(fused, 4))))
    plain_ds = dataset(lambda x, y: D.mono_chan(x, y))
    _, plain_rest = plain_ds._lower()
    assert len(plain_rest) == 8
    plain = [(x.clone(), y.clone()) for x, y in plain_ds.take(2)]
    assert len(batches) == len(plain) == 2
    ob, ov, on = OracleBank(bgs), OracleBank(voices), OracleBank(noises)
    for (x, y, d), (xp, yp) in zip(batches, plain):
        assert x.dtype == torch.bfloat16 and tuple(x.shape) == (4, 80, 120, 2) and xp.shape == x.shape
        assert torch.equal(y, yp)
        ref, ref_y = _oracle(ob, ov, labels, on, d, 'logmel_minmax')
        assert np.array_equal(y.cpu().numpy(), ref_y)
        for got in (x, xp):   # bfloat16 keeps 8 significant bits: half an ulp of the value on top of the bar
            got = got.float().cpu().numpy().astype(np.float64)
            assert (np.abs(got - ref) <= 2.0 ** -8 * np.abs(ref) + MINMAX_TOL).all()


def test_standalone_complex_to_magphase_broadcasts_width_3(engine):
    """transforms.complex_to_magphase of mono_chan's [re, im0, im1] rows: TF's broadcast, [mag0, mag1, ph0, ph1];
    the other odd widths stay errors."""
    import torch
    from challenge_b200 import transforms as TR
    from oracle import transforms as OT
    x = np.random.default_rng(3).standard_normal((257, 50, 3)).astype(np.float32)
    x[5] = 0.0
    x[6, :, 0] = -0.0
    got = TR.complex_to_magphase(x).cpu().numpy()
    ref = OT.complex_to_magphase(x)
    assert got.shape == ref.shape == (257, 50, 4)
    assert np.array_equal(got[..., :2], ref[..., :2])            # sqrt(real**2 + img**2), same rounding
    assert float(np.abs(got[..., 2:] - ref[..., 2:]).max()) <= 1e-6
    assert np.array_equal(np.signbit(got[5:7, :, 2:]), np.signbit(ref[5:7, :, 2:]))
    for width in (5, 7):
        with pytest.raises(ValueError):
            TR.complex_to_magphase(torch.zeros((4, width), device='cuda'))
