"""Host-side lowering of the 'se' chain (speech_enhancement_preprocess behind make_pipeline(...,
seperate_noise_voice=True)): IrisDataset absorbs the stage into one IRIS_FEAT_SE step exactly where it may
(no GPU needed)."""
import pytest


def _src(separate=True, n_chan=2):
    return {'separate': separate, 'n_chan': n_chan}


def _mode(ds):
    from challenge_b200 import _lib as L
    fused, rest = ds._lower()
    return fused['mode'] == L.FEAT_SE, fused, rest


def test_header_constant():
    import os
    import re
    from challenge_b200 import _lib as L
    h = open(os.path.join(os.path.dirname(__file__), '..', 'include', 'iris.h')).read()
    assert int(re.search(r'IRIS_FEAT_SE\s*=\s*(\d+)', h).group(1)) == L.FEAT_SE == 6


@pytest.mark.parametrize('front', ['', 'augment', 'filter', 'augment+filter'])
def test_se_chain_lowers_to_one_step(front):
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import IrisDataset
    ds = IrisDataset(_src())
    if 'augment' in front:
        ds = ds.map(D.augment)
    if 'filter' in front:
        ds = ds.map(D.stft_filter(3))
    ds = ds.map(D.speech_enhancement_preprocess).batch(12).map(D.label_downsample(32))
    se, fused, rest = _mode(ds.map(D.cast_features(torch.bfloat16)))
    assert se and fused['augment'] == ('augment' in front) and fused['filt'] == (3 if 'filter' in front else 0)
    # label_downsample and the cast stay stages of their own: the cast is not folded into FEAT_SE
    assert fused['out_flag'] == 0 and len(rest) == 2 and rest[1]._iris_stage[0] == 'cast'
    # unbatched, as the only stage
    se, _, rest = _mode(IrisDataset(_src()).map(D.speech_enhancement_preprocess))
    assert se and rest == []


def test_ineligible_chains_keep_the_stage():
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import IrisDataset
    se_ = D.speech_enhancement_preprocess
    cases = [
        IrisDataset(_src(separate=False)).map(se_).batch(4),           # labels are not (label, voice, noise)
        IrisDataset(_src(n_chan=4)).map(se_).batch(4),                 # C != 2
        IrisDataset(_src(n_chan=1)).map(se_).batch(4),
        IrisDataset(_src()).map(D.stereo_mono).map(se_).batch(4),      # a remap in front
        IrisDataset(_src()).map(D.random_merge_aug(4)).map(se_).batch(4),
        IrisDataset(_src()).map(D.to_frame_labels).map(se_).batch(4),  # to_frame_labels in front
        IrisDataset(_src()).map(lambda x, y: (x, y)).map(se_).batch(4),   # another stage in front
        IrisDataset(_src()).batch(4).map(se_),                        # after the batch point
        IrisDataset(_src()).map(se_).map(D.label_downsample(32)),     # unbatched with a stage behind
        IrisDataset({}).map(se_).batch(4),
    ]
    for ds in cases:
        se, fused, rest = _mode(ds)
        assert not se and fused['mode'] == L.FEAT_COMPLEX
        assert se_ in rest


def test_no_pre_batch_stage_is_absorbed_behind_it():
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import IrisDataset
    ds = IrisDataset(_src()).map(D.speech_enhancement_preprocess).map(D.stft_filter(3)).batch(4)
    se, fused, rest = _mode(ds)
    assert se and fused['filt'] == 0 and len(rest) == 2
