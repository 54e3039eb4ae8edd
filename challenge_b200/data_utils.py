"""Drop-in mirror of the reference's ``data_utils.py`` on the GPU (libiris C ABI).

Same names, argument meaning and quirks as /root/reference/data_utils.py (the broadcast in
``mono_chan``, the batch-axis ``[:resolution]`` slice in ``label_downsample``); tensors are
torch CUDA tensors.  ``load_wav`` takes a file name (decoded by torchaudio, as in the
reference) or an in-memory ``(waveform [chan, samples], sample_rate)`` / waveform: the kaldi
resampler to 16 kHz (``iris_resample``), normalize, STFT and the ``[freq, time, chan*2]`` layout
all run on the device.
"""
import numpy as np

from . import _lib as L
from . import _ops as O
from .engine import get_engine
from .transforms import mask, draw_masks

EPSILON = 1e-8  # utils.py:6


def load_wav(wav_fname):
    '''
    OUTPUT
    complex_specs: complex spectrogram of shape [freq, time, chan*2]
    (data_utils.py:9-29: normalize + Spectrogram(512, power=None) + relayout)
    '''
    r = 16000
    if isinstance(wav_fname, (str, bytes)):
        import torchaudio
        wav, r = torchaudio.load(wav_fname)
        wav = wav.numpy()
    elif isinstance(wav_fname, tuple):
        wav, r = wav_fname
    else:
        wav = wav_fname
    eng = get_engine()
    if int(r) != 16000:
        wav = eng.resample(wav, int(r), 16000)     # kaldi.resample_waveform (data_utils.py:20-21)
    return eng.stft(wav, normalize=True)


def normalize(wav):
    """data_utils.py:32-34 -- a scalar RMS of the whole clip (``iris_op_normalize``: the arithmetic
    of the bank registration, which applies it on the fused path)."""
    t = O.dev(wav)
    out = O.empty(t.shape)
    O.call('iris_op_normalize', O.ptr(t), O.ptr(out), t.numel())
    return out


def minmax(x, y=None):
    """data_utils.py:37-47 -- per-sample (axis 0) global min-max with safe_div."""
    t = O.dev(x)
    out = O.empty(t.shape)
    n = int(t.shape[0])
    O.call('iris_op_minmax', 0, O.ptr(t), O.ptr(out), n, t.numel() // max(n, 1), 1)
    if y is not None:
        return out, y
    return out


def log_on_mel(mel, labels=None):
    """data_utils.py:50-55."""
    t = O.dev(mel)
    out = O.empty(t.shape)
    O.call('iris_op_pointwise', L.PW_LOG_ON_MEL, O.ptr(t), O.ptr(out), t.numel(), 1, 0, 0.0)
    if labels is not None:
        return out, labels
    return out


def augment(specs, labels, time_axis=-2, freq_axis=-3, *, time_draws=None, freq_draws=None):
    """data_utils.py:58-61 -- 6 time masks (< 24) then 1 frequency mask (< 16)."""
    specs = mask(specs, axis=time_axis, max_mask_size=24, n_mask=6, draws=time_draws)
    specs = mask(specs, axis=freq_axis, max_mask_size=16, draws=freq_draws)
    return specs, labels


def to_frame_labels(x, y):
    """
    :param y: [..., n_voices, n_frames, n_classes]
    :return: [..., n_frames, n_classes]
    (data_utils.py:64-70)
    """
    t = O.dev(y)
    shape = tuple(t.shape)
    outer = int(np.prod(shape[:-3], dtype=np.int64))
    V, inner = int(shape[-3]), int(shape[-2] * shape[-1])
    out = O.empty(shape[:-3] + shape[-2:])
    O.call('iris_op_sum_voices', O.ptr(t), O.ptr(out), outer, V, inner)
    return x, out


def _chan_map(kind, x, w_out, factor=None, n_samples=1, rows_per_sample=None):
    t = O.dev(x)
    w_in = int(t.shape[-1])
    rows = t.numel() // w_in
    out = O.empty(tuple(t.shape[:-1]) + (w_out,))
    fp = None
    if factor is not None:
        factor, fp = O.f32_host(factor)
    O.call('iris_op_chan_map', kind, O.ptr(t), O.ptr(out), rows, w_in, w_out, fp, int(n_samples),
           int(rows_per_sample or rows))
    return out


def mono_chan(x, y=None):
    """data_utils.py:73-76 -- ``x[..., :1] + x[..., 1:]`` (broadcast quirk kept); a no-op when
    ``y is None``, like the reference."""
    if y is not None:
        return _chan_map(L.MAP_MONO_CHAN, x, int(x.shape[-1]) - 1), y
    return x


def stereo_mono(x, y=None):
    """data_utils.py:79-82."""
    out = _chan_map(L.MAP_STEREO_MONO, x, 6)
    if y is None:
        return out
    return out, y


def label_downsample(resolution=32):
    """data_utils.py:85-97 -- AveragePooling1D(r, r, 'same'), ``>= 0.5``, then the
    reference's ``[:resolution]`` on the BATCH axis."""
    def _pool(y_):
        t = O.dev(y_)
        B, T, K = (int(s) for s in t.shape)
        out = O.empty((B, -(-T // resolution), K))
        O.call('iris_op_avg_pool_time', O.ptr(t), O.ptr(out), B, T, K, int(resolution), 1)
        return out[:resolution]

    def _label_downsample(x, y):
        if isinstance(y, (list, tuple)):
            y = (_pool(y[0]),) + tuple([*y[1:]])
        else:
            y = _pool(y)
        return x, y
    return _label_downsample


def random_merge_aug(number):
    """data_utils.py:100-117 -- ``factor ~ U(0.1, 0.9)`` of shape ``(1, 1, number - chan)``,
    one draw per call (per sample: the map runs before ``batch``); ``factor=`` passes it."""
    def _random_merge_aug(x, y=None, *, factor=None):
        chan = x.shape[-1] // 2
        if chan != 2:
            raise ValueError('This augment can be used in 2 channel audio')
        if factor is None:
            factor = np.float32(0.1) + O.rng().random(number - chan, dtype=np.float32) * np.float32(0.8)
        out = _chan_map(L.MAP_MERGE_AUG, x, 2 * number, factor=np.asarray(factor, np.float32).reshape(-1),
                        n_samples=1)
        if y is not None:
            return out, y
        return out
    _random_merge_aug._iris_stage = ('merge_aug', number)
    return _random_merge_aug


def multiply_label(multiply_factor):
    """data_utils.py:120-123."""
    def _multiply_label(x, y):
        t = O.dev(y)
        out = O.empty(t.shape)
        O.call('iris_op_pointwise', L.PW_MULTIPLY, O.ptr(t), O.ptr(out), t.numel(), 1, 0,
               float(multiply_factor))
        return x, out
    return _multiply_label


def stft_filter(filter_num):
    """data_utils.py:126-136 -- bins 1..filter_num times 0 (axis 0 = frequency)."""
    def _stft_filter(x, y=None):
        t = O.dev(x)
        out = O.empty(t.shape)
        n_bins = int(t.shape[0])
        O.call('iris_op_stft_filter', O.ptr(t), O.ptr(out), n_bins, t.numel() // n_bins, int(filter_num))
        if y is None:
            return out
        return out, y
    _stft_filter._iris_stage = ('stft_filter', filter_num)
    return _stft_filter


def cast_features(dtype):
    """Not a reference function: the drop-in form of ``.map(lambda x, y: (tf.cast(x, dtype), y))``,
    e.g. for a trainer that runs in bfloat16 / float16.  ``dtype``: torch.bfloat16, torch.float16,
    torch.float32 or their names; anything else raises ValueError here.  Mapped after ``.batch()``
    behind stages the fused launch absorbs, it is absorbed too: the feature kernels store that dtype
    (the float32 features rounded to nearest even, bit for bit ``x.to(dtype)``).  Anywhere else it
    runs ``x.to(dtype)``.  Labels are not touched."""
    from .engine import out_flag
    import torch
    flag = out_flag(dtype)
    dt = {0: torch.float32, L.OUT_BF16: torch.bfloat16, L.OUT_F16: torch.float16}[flag]

    def _cast_features(x, y=None):
        x = x.to(dt) if isinstance(x, torch.Tensor) else O.dev(x).to(dt)
        if y is None:
            return x
        return x, y
    _cast_features._iris_stage = ('cast', flag)
    return _cast_features


def to_waveform(x, y=None, *, length=None):
    """Not a reference function: complex spectrograms back to audio, ``[257, T, 2C]`` -> ``[C, L]`` or
    ``[B, 257, T, 2C]`` -> ``[B, C, L]`` (``iris_istft``: ``torch.istft`` with ``load_wav``'s STFT parameters,
    ``L = 256 (T - 1)`` unless ``length`` is given).  The inverse of ``load_wav`` up to its normalisation.
    As a dataset stage (``.map(to_waveform)``) it converts ``x`` and, for a ``seperate_noise_voice=True``
    source, the ``only_voice`` / ``only_noise`` members of ``y = (labels, only_voice, only_noise)``; labels
    pass through."""
    from .engine import istft_shape
    parts = [x] + ([y[1], y[2]] if isinstance(y, tuple) and len(y) == 3 else [])
    for p in parts:   # shapes are checked before anything reaches the device
        istft_shape(np.shape(p), length)
    eng = get_engine()
    x = eng.istft(x, length)
    if y is None:
        return x
    if isinstance(y, tuple) and len(y) == 3:
        y = (y[0], eng.istft(y[1], length), eng.istft(y[2], length))
    return x, y


def speech_enhancement_preprocess(x, y=None):
    """
    :param y: ([..., n_voices, n_frames, n_classes], ..., ...)
    :return: [..., n_frames, n_classes]
    (data_utils.py:139-148 -- slices only: drop the DC bin, keep the real half)
    """
    x = O.dev(x)
    x = x[1:, ..., :x.shape[-1] // 2].contiguous()
    if y is None:
        return x
    _, y0 = to_frame_labels(None, y[0])
    y = (y0, O.dev(y[1])[1:, ..., :x.shape[-1] // 2].contiguous(),
         O.dev(y[2])[1:, ..., :x.shape[-1] // 2].contiguous())
    return x, y


augment._iris_stage = ('augment',)
to_frame_labels._iris_stage = ('to_frame_labels',)
speech_enhancement_preprocess._iris_stage = ('se',)
stereo_mono._iris_stage = ('stereo_mono',)
mono_chan._iris_stage = ('mono_chan',)
minmax._iris_stage = ('minmax',)
log_on_mel._iris_stage = ('log_on_mel',)
