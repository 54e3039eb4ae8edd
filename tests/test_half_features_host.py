"""Host-side tests of bfloat16 / float16 feature output: the IRIS_OUT_* flags of the C ABI and how
IrisDataset lowers data_utils.cast_features (no GPU needed)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sj_train_chain(ds, batch=12):
    from challenge_b200 import data_utils as D, transforms as TR
    ds = ds.map(D.to_frame_labels).map(D.augment).map(D.stft_filter(3)).batch(batch)
    return ds.map(TR.complex_to_magphase).map(TR.magphase_to_mel(80)).map(D.minmax).map(D.log_on_mel)


@pytest.mark.parametrize('dtype,flag_name', [('bfloat16', 'OUT_BF16'), ('float16', 'OUT_F16'), ('float32', None)])
def test_cast_after_the_sj_train_chain_is_absorbed_into_the_step_flag(dtype, flag_name):
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import IrisDataset
    flag = getattr(L, flag_name) if flag_name else 0
    for dt in (getattr(torch, dtype), dtype):          # a torch dtype or its name
        fused, rest = _sj_train_chain(IrisDataset({})).map(D.cast_features(dt))._lower()
        assert rest == [] and fused['mode'] == L.FEAT_LOGMEL_MINMAX and fused['out_flag'] == flag
    # the plain complex features of make_pipeline(...).batch(n) too
    fused, rest = IrisDataset({}).map(D.to_frame_labels).batch(4).map(D.cast_features(dtype))._lower()
    assert rest == [] and fused['mode'] == L.FEAT_COMPLEX and fused['out_flag'] == flag


def test_cast_stays_a_trailing_stage_behind_an_unabsorbed_stage():
    import torch
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import IrisDataset
    cast = D.cast_features(torch.bfloat16)
    # behind label_downsample (not absorbed) and behind a user lambda
    for other in (D.label_downsample(32), lambda x, y: (x, y)):
        fused, rest = _sj_train_chain(IrisDataset({})).map(other).map(cast)._lower()
        assert fused['out_flag'] == 0 and rest == [other, cast]
    # before .batch(): a per-element stage, never absorbed
    fused, rest = IrisDataset({}).map(D.to_frame_labels).map(cast).batch(4)._lower()
    assert fused['out_flag'] == 0 and rest[0] is cast
    # the wide-mel fallback of _prepare lowers without the mel stage: the cast trails the stand-alone mel
    fused, rest = _sj_train_chain(IrisDataset({})).map(cast)._lower(allow_mel=False)
    assert fused['out_flag'] == 0 and rest[-1] is cast and len(rest) == 4
    # only the first of two casts is absorbed (bf16 -> f16 is not fp32 -> f16)
    second = D.cast_features(torch.float16)
    fused, rest = _sj_train_chain(IrisDataset({})).map(cast).map(second)._lower()
    assert rest == [second]


@pytest.mark.parametrize('bad', ['float64', 'int8', 'half', None, 3])
def test_cast_features_rejects_other_dtypes_when_the_stage_is_built(bad):
    import torch
    from challenge_b200 import data_utils as D
    with pytest.raises(ValueError):
        D.cast_features(bad)
    with pytest.raises(ValueError):
        D.cast_features(torch.float64)


def test_output_flag_constants_match_the_header():
    from challenge_b200 import _lib as L
    text = open(os.path.join(ROOT, 'include', 'iris.h')).read()
    got = dict((k, int(v, 16)) for k, v in re.findall(r'\b(IRIS_OUT_[A-Z0-9]+)\s*=\s*(0x[0-9a-fA-F]+)', text))
    assert got == {'IRIS_OUT_BF16': L.OUT_BF16, 'IRIS_OUT_F16': L.OUT_F16}
    assert L.OUT_BF16 & L.MODE_MASK == 0 and L.OUT_F16 & L.MODE_MASK == 0
    assert max(L.FEAT_COMPLEX, L.FEAT_LOGMEL_MINMAX) <= L.MODE_MASK
    dl = open(os.path.join(ROOT, 'include', 'iris_dlpack.h')).read()
    assert re.search(r'\bkDLBfloat\s*=\s*4\b', dl)
