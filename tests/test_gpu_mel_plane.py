"""2-channel mel features from the STFT bin planes of the waveform banks (k_fused EPI_PLANE): the stored bins
themselves, every mel mode in float32 and bfloat16 with and without mono_chan and stft_filter, banks registered
from 44.1 kHz audio, and the launch rule (a mel support reaching bin 128 or beyond keeps the FFT path)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import f64

pytestmark = pytest.mark.gpu

_banks = {}


def _register(engine):
    from challenge_b200 import _lib as L
    from challenge_b200.synth import structured_banks
    if 'b' not in _banks:
        bgs, voices, labels, noises = structured_banks(702, 2)
        _banks['b'] = ((bgs, voices, noises), labels, [f64.bank_f64(x) for x in (bgs, voices, noises)])
    items, labels, b64 = _banks['b']
    frames = [engine.register_bank(L.BANK_BG, items[0]), engine.register_bank(L.BANK_VOICE, items[1], labels=labels),
              engine.register_bank(L.BANK_NOISE, items[2])]
    return frames, b64, labels


def _draw(frames, B, T, seed, masks, voices=True):
    from challenge_b200.plan import draw_batch
    return draw_batch(np.random.default_rng(seed), B, T, frames[0], frames[1] if voices else None,
                      frames[2] if voices else None, max_voices=4 if voices else 0, max_noises=3 if voices else 0,
                      snr=-20, min_ratio=2 / 3, n_time_masks=6 if masks else 0, time_mask_max=min(24, T),
                      n_freq_masks=1 if masks else 0)


def _np(t):
    return t.detach().float().cpu().numpy()


def _check(tag, got, ref, mode):
    val, bnd = ref
    assert got.shape == val.shape, (tag, got.shape, val.shape)
    r, at = f64.worst(f64.ratio(got, val, bnd, mode))
    print('%-50s ratio %8.3f at %s' % (tag, r, at))
    assert r <= 1, (tag, r, at, float(got[at]), float(val[at]), float(bnd[at]))


def _remap(name):
    from challenge_b200 import _lib as L
    return {None: L.REMAP_NONE, 'mono_chan': L.REMAP_MONO_CHAN}[name]


@pytest.mark.parametrize('remap', [None, 'mono_chan'])
def test_plane_bins_through_an_identity_mel_matrix(engine, remap):
    """A 128-band matrix that picks bin m for band m: the mel features are |X| (mono_chan: |re0 + re1 + i (re0 +
    im_j)|, which needs re and im of both channels) of the mixed stored bins 0..127, cell by cell within the
    float64 bound -- background alone (the plane rows of the items at gain 1) and the full mix."""
    from challenge_b200 import _lib as L
    W = np.zeros((257, 128), np.float32)
    W[np.arange(128), np.arange(128)] = 1.0
    try:
        engine.set_mel(128, mel_matrix=W)
        frames, b64, labels = _register(engine)
        for voices in (False, True):
            d = _draw(frames, 6, 120, 51, False, voices=voices)
            engine.upload_plan(d, chan_remap=_remap(remap), n_out_chan=2 if remap else 0)
            got = _np(engine.features(L.FEAT_MEL))
            keep = _np(engine.labels()[2]).astype(int) if voices else None
            ref = f64.features(b64, labels, d, 'mel', False, keep=keep, remap_kind=remap, n_out=2 if remap else 0,
                               mel_w=W)
            _check('identity %s voices=%d' % (remap, voices), got, ref, 'mel')
    finally:
        engine.set_mel(80)


@pytest.mark.parametrize('filt', [0, 3])
@pytest.mark.parametrize('remap', [None, 'mono_chan'])
def test_mel_modes_from_the_plane(engine, monkeypatch, remap, filt):
    """mel / logmel / logmel_minmax with masks against the float64 reference; bfloat16 features are the float32
    ones rounded; the fixed-shape and the generic instance agree bit for bit."""
    import torch
    from challenge_b200 import _lib as L
    engine.set_mel(80)
    frames, b64, labels = _register(engine)
    d = _draw(frames, 7, 150, 60 + filt, True)
    cache = {}
    for mode, feat in (('mel', L.FEAT_MEL), ('logmel', L.FEAT_LOGMEL), ('logmel_minmax', L.FEAT_LOGMEL_MINMAX)):
        engine.upload_plan(d, stft_filter=filt, chan_remap=_remap(remap), n_out_chan=2 if remap else 0)
        got = engine.features(feat)          # before labels: the tile lists of k_labels
        keep = _np(engine.labels()[2]).astype(int)
        ref = f64.features(b64, labels, d, mode, False, keep=keep, remap_kind=remap, n_out=2 if remap else 0,
                           stft_filter=filt, mel_w=engine.mel_matrix, cache=cache)
        _check('%s %s filt=%d' % (remap, mode, filt), _np(got), ref, mode)
        half = engine.features(feat, dtype=torch.bfloat16)
        assert torch.equal(half.view(torch.int16), got.to(torch.bfloat16).view(torch.int16)), mode
        monkeypatch.setenv('IRIS_NO_FIXED_EPI', '1')
        generic = engine.features(feat)
        monkeypatch.delenv('IRIS_NO_FIXED_EPI')
        assert torch.equal(generic, got), mode


def test_plane_of_a_bank_registered_from_44k_audio(engine):
    """A bank registered from 44.1 kHz items builds its plane from the resampled audio: its features equal those
    of the same bank registered from the device-resampled 16 kHz waveforms, bit for bit."""
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200.synth import structured_banks
    engine.set_mel(80)
    rng = np.random.default_rng(44)
    bgs = [rng.standard_normal((2, n)).astype(np.float32) for n in (441000, 300000, 200017)]
    _, voices, labels, noises = structured_banks(702, 2)
    feats = []
    for items in ([(x, 44100) for x in bgs], [engine.resample(x, 44100).cpu().numpy() for x in bgs]):
        bg_frames = engine.register_bank(L.BANK_BG, items)
        vf = engine.register_bank(L.BANK_VOICE, voices, labels=labels)
        nf = engine.register_bank(L.BANK_NOISE, noises)
        d = _draw([bg_frames, vf, nf], 6, 200, 7, True)
        engine.upload_plan(d, stft_filter=3)
        feats.append(engine.features(L.FEAT_LOGMEL_MINMAX).clone())
        engine.labels()
    assert torch.equal(feats[0], feats[1])
    assert torch.isfinite(feats[0]).all()


def test_support_reaching_bin_191_keeps_the_fft_path(engine):
    """A mel matrix whose support reaches bin 191 (upper edge 6 kHz) needs bins a plane row does not hold: the
    launch takes the NJ = 8 FFT instance, within the float64 bound; the default matrix takes the plane."""
    from challenge_b200 import _lib as L
    try:
        engine.set_mel(80, upper_edge_hertz=6000.0)
        assert 128 <= np.nonzero(engine.mel_matrix.any(1))[0].max() <= 191
        frames, b64, labels = _register(engine)
        d = _draw(frames, 5, 100, 71, True)
        engine.upload_plan(d, stft_filter=3)
        got = _np(engine.features(L.FEAT_LOGMEL))
        keep = _np(engine.labels()[2]).astype(int)
        ref = f64.features(b64, labels, d, 'logmel', False, keep=keep, stft_filter=3, mel_w=engine.mel_matrix)
        _check('support to bin 191 logmel', got, ref, 'logmel')
    finally:
        engine.set_mel(80)


_KERNELS = r"""
import json, sys
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
from challenge_b200 import _lib as L
from challenge_b200.engine import Engine
from challenge_b200.plan import draw_batch
from challenge_b200.synth import structured_banks
eng = Engine(0)
bgs, voices, labels, noises = structured_banks(702, 2)
fr = [eng.register_bank(L.BANK_BG, bgs), eng.register_bank(L.BANK_VOICE, voices, labels=labels),
      eng.register_bank(L.BANK_NOISE, noises)]
d = draw_batch(np.random.default_rng(3), 6, 100, fr[0], fr[1], fr[2], max_voices=4, max_noises=3, snr=-20,
               min_ratio=2 / 3, n_time_masks=6, time_mask_max=24, n_freq_masks=1)
out = {}
for name, mel_kw, remap, mode in (('default logmel_minmax', {}, L.REMAP_NONE, L.FEAT_LOGMEL_MINMAX),
                                  ('default mel mono_chan', {}, L.REMAP_MONO_CHAN, L.FEAT_MEL),
                                  ('to 6 kHz logmel', dict(upper_edge_hertz=6000.0), L.REMAP_NONE, L.FEAT_LOGMEL)):
    eng.set_mel(80, **mel_kw)
    eng.upload_plan(d, stft_filter=3, chan_remap=remap, n_out_chan=2 if remap else 0)
    eng.labels()
    eng.features(mode)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.features(mode)
        torch.cuda.synchronize()
    out[name] = sorted({e.key for e in prof.key_averages() if 'k_fused<' in e.key})
print('KERNELS ' + json.dumps(out))
"""


def test_launch_rule_picks_the_plane_instances():
    """The k_fused instances the launches run (torch.profiler, in a process of its own): the default matrix takes
    the fixed plane instances (EPI_PLANE | EPI_C2 | ..., with EPI_MONO for mono_chan), a matrix reaching bin 191
    the NJ = 8 FFT instance."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, '-c', _KERNELS], capture_output=True, text=True, cwd=root, timeout=600)
    line = [x for x in r.stdout.splitlines() if x.startswith('KERNELS ')]
    assert r.returncode == 0 and line, r.stdout + r.stderr
    got = json.loads(line[0][8:])
    print(got)
    assert got['default logmel_minmax'] == ['void iris::k_fused<3, 4, %d, float>(iris::FusedParams)' % (32 | 4 | 1)]
    assert got['default mel mono_chan'] == ['void iris::k_fused<3, 4, %d, float>(iris::FusedParams)' % (32 | 16 | 4)]
    assert got['to 6 kHz logmel'] == ['void iris::k_fused<3, 8, 0, float>(iris::FusedParams)']
