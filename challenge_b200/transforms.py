"""Drop-in mirror of the reference's ``transforms.py`` on the GPU (libiris C ABI).

Same names, argument meaning and error behaviour as /root/reference/transforms.py; tensors
are torch CUDA tensors (DLPack-exportable).  Random draws the reference takes from
``tf.random`` are made on the host (``challenge_b200.set_seed``) or passed explicitly with the
keyword-only ``draws=`` / ``offset=`` arguments, so a caller -- and the parity tests -- can
feed the GPU and the reference identical randomness.
"""
import numpy as np

from . import _lib as L
from . import _ops as O
from .engine import default_mel_matrix, get_engine

EPSILON = 1e-8                       # transforms.py:6
LOG_EPSILON = float(np.log(EPSILON))  # transforms.py:7


# ---- FEATURE INDEPENDENT AUGMENTATIONS ----
def draw_masks(total, max_mask_size=None, n_mask=1, rng=None):
    """The draws of ``mask`` in the reference's order (transforms.py:25-26): per mask
    ``size in [0, max_mask_size)`` then ``offset in [0, total - size)``."""
    rng = rng or O.rng()
    if max_mask_size is None:
        max_mask_size = total
    out = np.zeros((n_mask, 2), np.int32)
    for i in range(n_mask):
        size = int(rng.integers(0, max_mask_size))
        if total - size <= 0:
            from .errors import InvalidArgumentError
            raise InvalidArgumentError('mask: empty offset range (transforms.py:26)')
        out[i] = (size, int(rng.integers(0, total - size)))
    return out


def mask(specs, axis, max_mask_size=None, n_mask=1, *, draws=None):
    """transforms.py:12-40 -- ``n_mask`` multiplicative 0/1 masks along ``axis``."""
    x = O.dev(specs)
    axis = O.norm_axis(axis, x.dim())
    total = x.shape[axis]
    if draws is None:
        draws = draw_masks(total, max_mask_size, n_mask)
    d, dp = O.i32_host(np.asarray(draws).reshape(-1, 2))
    assert d.shape[0] == n_mask, 'need n_mask (size, offset) pairs'
    outer, n, inner = O.split_axis(x.shape, axis)
    out = O.empty(x.shape)
    O.call('iris_op_mask', O.ptr(x), O.ptr(out), outer, n, inner, dp, int(n_mask))
    return out


def random_shift(specs, axis=0, width=16, *, offset=None):
    """transforms.py:43-47 -- zero-pad ``width`` both sides of ``axis``, random crop."""
    x = O.dev(specs)
    axis = O.norm_axis(axis, x.dim())
    if offset is None:
        offset = int(O.rng().integers(0, 2 * width + 1))     # tf.image.random_crop: inclusive
    outer, n, inner = O.split_axis(x.shape, axis)
    out = O.empty(x.shape)
    O.call('iris_op_random_shift', O.ptr(x), O.ptr(out), outer, n, inner, int(width), int(offset))
    return out


# ---- MAGNITUDE-PHASE SPECTROGRAM ----
def magphase_to_mel(num_mel_bins=80, num_spectrogram_bins=257, sample_rate=16000, **kwargs):
    """transforms.py:51-77 -- the matrix is ``tf.signal.linear_to_mel_weight_matrix`` rebuilt
    op-for-op in fp32 (``engine.default_mel_matrix``); kwargs as in TF
    (``lower_edge_hertz``, ``upper_edge_hertz``)."""
    mel_matrix = default_mel_matrix(num_mel_bins, num_spectrogram_bins, sample_rate, **kwargs)

    def _magphase_to_mel(x, y=None):
        '''
        x: [batch_size, freq, time, chan2]

        output: [batch_size, mel_freq, time, chan]
        '''
        t = O.dev(x)
        if t.dim() not in (3, 4):
            raise ValueError('len(x.shape) must be 3 or 4')
        eng = get_engine()
        cur = getattr(eng, 'mel_matrix', None)
        if cur is None or cur.shape != mel_matrix.shape or not np.array_equal(cur, mel_matrix):
            eng.set_mel(mel_matrix=mel_matrix)
        shape = t.shape if t.dim() == 4 else (1,) + tuple(t.shape)
        B, F, T, C2 = (int(s) for s in shape)
        if F != num_spectrogram_bins:
            raise ValueError('x has %d frequency bins, the mel matrix %d' % (F, num_spectrogram_bins))
        C = C2 // 2
        out = O.empty((B, num_mel_bins, T, C))
        L.check(eng.lib.iris_op_mel(eng._ctx, O.ptr(t), O.ptr(out), B, T, C, eng._stream()))
        if t.dim() == 3:
            out = out[0]
        if y is None:
            return out
        return out, y
    _magphase_to_mel._iris_stage = ('mel', num_mel_bins, mel_matrix)
    return _magphase_to_mel


def log_magphase(specs, labels=None, n_chan=2):
    """transforms.py:80-86."""
    x = O.dev(specs)
    out = O.empty(x.shape)
    width = int(x.shape[-1])
    O.call('iris_op_pointwise', L.PW_LOG_MAGPHASE, O.ptr(x), O.ptr(out), x.numel() // width, width,
           int(n_chan), 0.0)
    if labels is not None:
        return out, labels
    return out


def minmax_norm_magphase(specs, labels=None):
    """transforms.py:89-107 -- separate per-sample min-max of the magnitude and phase halves."""
    x = O.dev(specs)
    out = O.empty(x.shape)
    n = int(x.shape[0])
    O.call('iris_op_minmax', 1, O.ptr(x), O.ptr(out), n, x.numel() // max(n, 1), int(x.shape[-1]))
    if labels is not None:
        return out, labels
    return out


# ---- COMPLEX-SPECTROGRAMS ----
def complex_to_magphase(complex_tensor, y=None):
    """transforms.py:111-123."""
    x = O.dev(complex_tensor)
    width = int(x.shape[-1])
    # mono_chan's [re, im0, im1]: TF broadcasts re against both imaginary columns -> [mag0, mag1, ph0, ph1]
    out = O.empty(tuple(x.shape[:-1]) + (4 if width == 3 else width,))
    O.call('iris_op_pointwise', L.PW_C2MP, O.ptr(x), O.ptr(out), x.numel() // width, width, 0, 0.0)
    if y is None:
        return out
    return out, y


def magphase_to_complex(magphase):
    """transforms.py:126-134."""
    x = O.dev(magphase)
    out = O.empty(x.shape)
    width = int(x.shape[-1])
    O.call('iris_op_pointwise', L.PW_MP2C, O.ptr(x), O.ptr(out), x.numel() // width, width, 0, 0.0)
    return out


def phase_vocoder(complex_spec, rate=1.):
    """transforms.py:137-195 -- time-stretch by ``rate`` (magnitudes interpolated between
    neighbouring frames, phases advanced by the wrapped frame-to-frame difference).
    ``rate == 1`` returns the input, like the reference.  The time-step arithmetic
    (``tf.range(0, T, rate)`` in float32: ``ceil(T / rate)`` steps ``i * rate``) is done on the
    host, the per-row phase accumulation on the GPU."""
    if rate == 1:
        return complex_spec
    x = O.dev(complex_spec)
    if x.dim() != 3 or x.shape[-1] % 2:
        raise ValueError('phase_vocoder expects [freq, time, chan*2]')
    F, T, C2 = (int(v) for v in x.shape)
    f32 = np.float32
    n_steps = int(np.ceil(T / rate))
    steps = (f32(0) + np.arange(n_steps, dtype=np.float32) * f32(rate)).astype(np.float32)
    idx0, p0 = O.i32_host(steps.astype(np.int32))
    idx1, p1 = O.i32_host((steps + f32(1)).astype(np.int32))
    alpha, pa = O.f32_host(np.mod(steps, f32(1.)))
    out = O.empty((F, n_steps, C2))
    O.call('iris_op_phase_vocoder', O.ptr(x), O.ptr(out), F, T, C2 // 2, n_steps, p0, p1, pa)
    return out


complex_to_magphase._iris_stage = ('magphase',)
log_magphase._iris_stage = ('log_magphase',)
