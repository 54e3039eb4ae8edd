"""Host side of waveform banks at any sample rate (no GPU): how bank items are classified and packed for
iris_bank_register / iris_bank_register_audio, and the frame counts the resampled lengths give."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _wav(n_chan, n, seed=0):
    return np.random.default_rng(seed).standard_normal((n_chan, n)).astype(np.float32)


def test_bank_item_forms():
    from challenge_b200.engine import bank_item
    w = _wav(2, 1000)
    a, r = bank_item(w)
    assert r == 16000 and a is w
    a, r = bank_item((w.astype(np.float64), np.int64(44100)))
    assert r == 44100 and type(r) is int and a.dtype == np.float32 and np.array_equal(a, w)
    a, r = bank_item((w[:, ::2], 8000))                 # a strided view becomes contiguous
    assert a.flags['C_CONTIGUOUS'] and np.array_equal(a, w[:, ::2]) and r == 8000


def test_classification_of_bank_items():
    from challenge_b200.engine import is_spec_bank
    from challenge_b200.pipeline import _is_waveform_bank
    w, s = _wav(2, 1000), np.zeros((257, 10, 4), np.float32)
    for items, spec in (([w], False), ([(w, 44100)], False), ([(w, 16000), w], False), ([s], True),
                        (np.stack([s, s]), True), ([w.tolist()], False)):
        assert is_spec_bank(items) is spec
        assert _is_waveform_bank(items) is (not spec)


def test_packing_keeps_order_lengths_and_rates():
    from challenge_b200.engine import pack_waveforms
    items = [(_wav(3, 900, 1), 44100), _wav(3, 500, 2), (_wav(3, 700, 3), 8000), (_wav(3, 300, 4), 16000)]
    packed, offsets, rates, n_chan = pack_waveforms(items)
    assert n_chan == 3 and packed.dtype == np.float32 and rates.dtype == np.int32 and offsets.dtype == np.int64
    assert offsets.tolist() == [0, 900, 1400, 2100, 2400]       # per-channel samples at each item's own rate
    assert rates.tolist() == [44100, 16000, 8000, 16000]
    for i, it in enumerate(items):
        w = it[0] if isinstance(it, tuple) else it
        assert np.array_equal(packed[3 * offsets[i]:3 * offsets[i + 1]].reshape(3, -1), w)   # [C, len_i] blocks


def test_packing_rejects_mixed_channel_counts():
    from challenge_b200.engine import pack_waveforms
    with pytest.raises(AssertionError):
        pack_waveforms([(_wav(2, 500), 44100), (_wav(1, 500), 44100)])
    with pytest.raises(AssertionError):
        pack_waveforms([_wav(2, 500), np.zeros(500, np.float32)])


@pytest.mark.parametrize('rate', [44100, 48000, 22050, 11025, 32000, 8000])
def test_frames_of_resampled_items(rate):
    """A registered item has 1 + n16 // 256 frames, n16 = iris_resample_len(n, rate, 16000), the length
    load_wav's resampler gives (host arithmetic of the library, checked against the oracle's count)."""
    from challenge_b200 import _lib
    from oracle.data_utils import _lr_num_output_samples
    lib = _lib.load()
    for n in (700, 771, 22051, 44100 * 3 + 17):
        n16 = lib.iris_resample_len(n, rate, 16000)
        assert n16 == _lr_num_output_samples(n, rate, 16000)
        assert abs(n16 - n * 16000 / rate) <= 1


def test_audio_entry_point_is_declared_and_optional():
    """iris_bank_register_audio is in include/iris.h and the binding, under ABI version 2; the loader treats
    it as optional, so a library that predates it still loads (callers probe with hasattr)."""
    from challenge_b200 import _lib
    text = open(os.path.join(ROOT, 'include', 'iris.h')).read()
    assert 'int iris_bank_register_audio(' in text and '#define IRIS_ABI_VERSION 2' in text
    assert 'iris_bank_register_audio' in _lib.OPTIONAL and 'iris_bank_register_audio' in _lib.SIGNATURES
    assert len(_lib.SIGNATURES['iris_bank_register_audio'][1]) == 11
    assert hasattr(_lib.load(), 'iris_bank_register_audio')
