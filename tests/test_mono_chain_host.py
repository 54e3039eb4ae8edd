"""Host-side lowering of sj_train's n_chan = 1 chain (mono_chan in front of the feature stages): IrisDataset
absorbs mono_chan as a channel remap for 2-channel banks and keeps it a per-element stage otherwise (no GPU
needed)."""
import pytest


def _chain(n_chan=2, cast=None, batch=12):
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import IrisDataset
    ds = IrisDataset({'n_chan': n_chan}).map(D.to_frame_labels).map(D.augment).map(D.mono_chan)
    ds = ds.map(D.stft_filter(3)).batch(batch)
    ds = ds.map(TR.complex_to_magphase).map(TR.magphase_to_mel(80)).map(D.minmax).map(D.log_on_mel)
    return ds.map(D.cast_features(cast)) if cast is not None else ds


def test_header_constant():
    import os
    import re
    from challenge_b200 import _lib as L
    h = open(os.path.join(os.path.dirname(__file__), '..', 'include', 'iris.h')).read()
    assert int(re.search(r'IRIS_REMAP_MONO_CHAN\s*=\s*(\d+)', h).group(1)) == L.REMAP_MONO_CHAN == 3


@pytest.mark.parametrize('cast', [None, 'bfloat16', 'float16'])
def test_mono_chain_lowers_to_one_step(cast):
    import torch
    from challenge_b200 import _lib as L
    fused, rest = _chain(cast=getattr(torch, cast) if cast else None)._lower()
    assert rest == []
    assert fused['mode'] == L.FEAT_LOGMEL_MINMAX and fused['remap'] == L.REMAP_MONO_CHAN and fused['n_out'] == 2
    assert fused['filt'] == 3 and fused['augment'] and fused['frame_labels'] and fused['n_mels'] == 80
    assert fused['out_flag'] == {None: 0, 'bfloat16': L.OUT_BF16, 'float16': L.OUT_F16}[cast]


def test_stage_order_of_the_spectrogram_chains():
    """mono_chan sits in the remap slot: after augment, before stft_filter; the feature stages behind the batch
    fold in as they do for the other remaps."""
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import IrisDataset
    src = {'n_chan': 2}
    fused, rest = IrisDataset(src).map(D.augment).map(D.mono_chan).map(D.stft_filter(5)).batch(4)._lower()
    assert rest == [] and fused['mode'] == L.FEAT_COMPLEX and fused['remap'] == L.REMAP_MONO_CHAN
    assert fused['filt'] == 5
    fused, rest = IrisDataset(src).map(D.mono_chan).batch(4).map(TR.complex_to_magphase)._lower()
    assert rest == [] and fused['mode'] == L.FEAT_MAGPHASE and fused['remap'] == L.REMAP_MONO_CHAN
    # unbatched, mono_chan the only stage
    fused, rest = IrisDataset(src).map(D.mono_chan)._lower()
    assert rest == [] and fused['remap'] == L.REMAP_MONO_CHAN
    # out of order: stft_filter is absorbed, the mono_chan behind it is not (nor is anything after it)
    fused, rest = IrisDataset(src).map(D.stft_filter(3)).map(D.mono_chan).batch(4)._lower()
    assert fused['remap'] == L.REMAP_NONE and fused['filt'] == 3 and rest[0] is D.mono_chan
    # one remap per chain: a second remap stage stays per element
    fused, rest = IrisDataset(src).map(D.mono_chan).map(D.stereo_mono).batch(4)._lower()
    assert fused['remap'] == L.REMAP_MONO_CHAN and rest[0] is D.stereo_mono


@pytest.mark.parametrize('n_chan', [1, 4, None])
def test_other_channel_counts_keep_the_stage(n_chan):
    """mono_chan of 1- or 4-channel banks (or a source that does not say) is not fused: it runs per element as
    before, and the stages behind it are not absorbed."""
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D
    fused, rest = _chain(n_chan=n_chan)._lower()
    assert fused['remap'] == L.REMAP_NONE and fused['mode'] == L.FEAT_COMPLEX
    assert fused['augment'] and fused['filt'] == 0
    assert rest[0] is D.mono_chan and len(rest) == 7


def test_wide_mel_fallback_keeps_mono_chan_and_the_standalone_mel():
    """_lower(allow_mel=False) (a mel matrix wider than the fused epilogue takes): magnitude + phase of the two
    pseudo-channels fused, the mel stage and everything behind it stand-alone."""
    import torch
    from challenge_b200 import _lib as L
    fused, rest = _chain(cast=torch.bfloat16)._lower(allow_mel=False)
    assert fused['mode'] == L.FEAT_MAGPHASE and fused['remap'] == L.REMAP_MONO_CHAN and fused['n_out'] == 2
    assert fused['out_flag'] == 0 and len(rest) == 4
    assert getattr(rest[0], '_iris_stage', (None,))[0] == 'mel'
    assert getattr(rest[3], '_iris_stage', (None,))[0] == 'cast'
