"""Host-side lowering of the sj_train chain with a channel remap (stereo_mono / random_merge_aug(n)) in
front of the mel stage: IrisDataset absorbs the whole chain into one step (no GPU needed)."""
import pytest


def _chain(remap, n=4, cast=None):
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import IrisDataset
    ds = IrisDataset({}).map(D.to_frame_labels).map(D.augment)
    ds = ds.map(D.stereo_mono if remap == 'stereo_mono' else D.random_merge_aug(n))
    ds = ds.map(D.stft_filter(3)).batch(12)
    ds = ds.map(TR.complex_to_magphase).map(TR.magphase_to_mel(80)).map(D.minmax).map(D.log_on_mel)
    return ds.map(D.cast_features(cast)) if cast is not None else ds


@pytest.mark.parametrize('remap,n', [('stereo_mono', 3), ('merge_aug', 3), ('merge_aug', 4), ('merge_aug', 16)])
def test_remap_chain_lowers_to_one_step(remap, n):
    import torch
    from challenge_b200 import _lib as L
    want = L.REMAP_STEREO_MONO if remap == 'stereo_mono' else L.REMAP_MERGE_AUG
    fused, rest = _chain(remap, n, cast=torch.bfloat16)._lower()
    assert rest == []
    assert fused['mode'] == L.FEAT_LOGMEL_MINMAX and fused['out_flag'] == L.OUT_BF16
    assert fused['remap'] == want and fused['n_out'] == n and fused['filt'] == 3 and fused['n_mels'] == 80
    fused, rest = _chain(remap, n)._lower()                 # without the cast
    assert rest == [] and fused['mode'] == L.FEAT_LOGMEL_MINMAX and fused['out_flag'] == 0 and fused['remap'] == want


def test_wide_mel_fallback_keeps_the_remap_and_the_standalone_mel():
    """_lower(allow_mel=False) (a mel matrix wider than the fused epilogue takes): magnitude + phase with the
    remap fused, the mel stage and everything behind it stand-alone."""
    import torch
    from challenge_b200 import _lib as L
    fused, rest = _chain('stereo_mono', cast=torch.bfloat16)._lower(allow_mel=False)
    assert fused['mode'] == L.FEAT_MAGPHASE and fused['remap'] == L.REMAP_STEREO_MONO and fused['n_out'] == 3
    assert fused['out_flag'] == 0 and len(rest) == 4
    assert getattr(rest[0], '_iris_stage', (None,))[0] == 'mel'
