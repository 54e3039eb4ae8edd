"""Float64 values and per-cell error bounds of the stand-alone drop-in operations (TEST INFRASTRUCTURE ONLY).

The functions of ``challenge_b200.{data_utils,transforms,metrics,trainer}`` run one stand-alone kernel each
(k_ops.cu, k_resample.cu, the STFT of ``iris_stft``, the inverse STFT of ``iris_istft``).  Their inputs are exact float32 values, so the error a correct
float32 implementation may make in an output cell is a forward-error bound of the operation's own arithmetic,
computed here next to the float64 value from the size of the terms that went into that cell:

n-term sum          gamma_n * sum |terms|, gamma_n = n u / (1 - n u), u = 2^-24
math functions      (k + 1) ulp of the float32-rounded result for a function of k ulp maximum error (CUDA C
                    Programming Guide, single-precision functions without --use_fast_math: atan2f 3, logf 1, sinf /
                    cosf / sincosf 2, rsqrtf 2; sqrtf and division are correctly rounded)
one rounding        u * |value|, plus TINY = 2^-149 where a product may land in the subnormal range

Operations whose result is decided by selections, 0 / 1 factors and a fixed order of float32 operations are
given as the float32 computation itself, in the kernel's order (``*_f32``): the kernel must match it bit for bit.

Only ``load_wav`` / ``Engine.stft`` and the inverse (``to_waveform`` / ``Engine.istft``, KAPPA_ISTFT and SUB_ISTFT
below) use calibrated constants.  The former is the 'complex' cell of oracle/f64.py with its own
KAPPA_LOAD, 4x the largest ratio |oracle - f64| / (u S_pair) the float32 oracle (float32 normalisation, torchaudio
FFT) reaches on the signals of tests/test_f64_ops_host.py, which re-measures it.  It is larger than oracle/f64.py's
KAPPA_C: these signals put exact-zero stretches, a -100 dB tail and pure DC / Nyquist tones into single frames,
which the bank corpus of that calibration does not.  Everything else is derived.  The product-defined float32 constants (the Kaldi filter
table, the mel matrix, the phase vocoder's steps) are built in float32 as the library builds them and promoted.
"""
import math

import numpy as np

from . import f64
from .data_utils import _lr_indices_and_weights, _lr_num_output_samples, stft_f64

U = f64.U
TINY = 2.0 ** -149
F32 = np.float32
EPS32 = float(F32(1e-8))          # the kernels' 1e-8f
FLOOR12 = float(F32(1e-12))       # k_cos_sim's 1e-12f
# maximum ulp errors of the CUDA single-precision functions (CUDA C Programming Guide, table of mathematical
# functions; the library is built without --use_fast_math)
ULP_ATAN2 = 3
ULP_LOG = 1
ULP_SINCOS = 2
ULP_RSQRT = 2
# The Kaldi table is computed twice, on the host in C (append_kaldi_table: libm cosf / sinf) and here in numpy; two
# float32 implementations of cos and sin that are each within 1 ulp of the exact value.  With w = h * s, h = 0.5 (1 +
# cos a) and s = sin(b) / (pi dt) / orig: |dh| <= 0.5 (2 ulp(1) + 2 half-ulps of 1 + cos) <= 3 u, and s (a sine and
# three roundings, each differently rounded in the two) <= 2 * 4 u relative; so |dw| <= A_TAB * u * |s| with
# A_TAB = 11.  tests/test_f64_ops_host.py checks numpy's table against the float64 one at half of that.
A_TAB = 11
# load_wav: largest |oracle - f64| / (u S_pair) measured over tests/test_f64_ops_host.py LOAD_CASES (5.09, the
# 'zeros' signal at a frame that straddles an exact-zero stretch); KAPPA_LOAD = 4x, as oracle/f64.py's kappas
MEASURED_RATIO_LOAD = 5.1
KAPPA_LOAD = 4 * MEASURED_RATIO_LOAD
# to_waveform: largest |float32 torch.istft - f64| / (u S) over tests/test_istft_host.py istft_cases (4.51, the
# 'clicks' signal, C = 3: a frame whose energy sits in a few samples); KAPPA_ISTFT = 4x, the same rule.  SUB_ISTFT:
# 4x the largest |float32 model of k_istft - f64| / (2^-149 G) on bins around 1e-40 and 1e-43 (0.997), where the
# samples are subnormal and their rounding is absolute; torch.istft cannot calibrate that one, its x w / w^2 rounds
# x w at the subnormal spacing before dividing by w^2 (1.1e4 times this bound past the last frame's centre)
MEASURED_RATIO_ISTFT = 4.6
KAPPA_ISTFT = 4 * MEASURED_RATIO_ISTFT
MEASURED_SUB_ISTFT = 1.0
SUB_ISTFT = 4 * MEASURED_SUB_ISTFT


def gamma(n):
    n = np.asarray(n, np.float64)
    return n * U / (1 - n * U)


def ulp32(y):
    """Spacing of float32 at |y| rounded to float32 (2^-149 at 0)."""
    a = np.abs(np.asarray(y, np.float64))
    with np.errstate(over='ignore'):
        return np.spacing(a.astype(np.float32)).astype(np.float64)


def fn_bound(y, k):
    """Bound of a float32 function of k ulp maximum error at the exact value y."""
    return (k + 1) * ulp32(y)


def ratio(got, ref, bound):
    """``f64.ratio`` with a plain (linear) difference in every column, phases included: for exact float32 inputs
    atan2f stays in [-fl(pi), fl(pi)], so a circular difference is not needed, and a linear one also fails a phase of
    the wrong sign at the branch cut (atan2(+-0, x < 0)).  Where the reference itself is not finite (a log of 0, an
    overflowed product of the reference's own float32 formula) the cell must be the identical non-finite value,
    else inf."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    bound = np.broadcast_to(np.asarray(bound, np.float64), ref.shape)
    fin = np.isfinite(ref)
    with np.errstate(invalid='ignore', over='ignore'):
        diff = np.abs(got - ref)
    with np.errstate(divide='ignore', invalid='ignore'):
        r = np.where(got == ref, 0.0, diff / bound)
    r[np.isnan(r) | (~np.isfinite(got) & fin)] = np.inf
    same = (np.isnan(got) & np.isnan(ref)) | (got == ref)
    r[~fin] = np.where(same[~fin], 0.0, np.inf)
    return r


def bitexact_ratio(got, ref):
    """0 where ``got`` is ``ref`` bit for bit (float32), inf elsewhere: the ratio of the bit-exact operations."""
    g = np.ascontiguousarray(got, np.float32).view(np.uint32)
    r = np.ascontiguousarray(ref, np.float32).view(np.uint32)
    assert g.shape == r.shape, (g.shape, r.shape)
    return np.where(g == r, 0.0, np.inf)


# ---- load_wav / Engine.stft (iris_stft: k_bank_prepare + k_fused<FM_COMPLEX>) ----
def stft_f64_frames(wav, t0, t1):
    """Frames [t0, t1) of ``stft_f64`` (centre reflect padding) -> [C, 257, t1 - t0], without padding the whole
    clip: long files are checked frame block by frame block."""
    wav = np.asarray(wav, np.float64)
    C, N = wav.shape
    idx = 256 * np.arange(t0, t1)[:, None] + np.arange(512)[None, :] - 256     # sample index of each tap
    idx = np.abs(idx)                                                           # reflect at the start
    idx = np.where(idx > N - 1, 2 * (N - 1) - idx, idx)                         # reflect at the end
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(512) / 512)
    return np.fft.rfft(wav[:, idx] * w, axis=-1).transpose(0, 2, 1)


def stft_value_bound(wav, normalize=True, frames=None, kappa=KAPPA_LOAD):
    """load_wav of ``wav [C, N]`` in float64 -> (value, bound) ``[257, T, 2C]`` (or frames [t0, t1) only).  The
    bound is the 'complex' cell of oracle/f64.py for one source of gain 1: kappa u times the L2 norm of the frame's
    bins over both channels of its FFT pair, plus R_OUT u |value|."""
    wav = np.asarray(wav, np.float64)
    if normalize:
        wav = f64.normalize_f64(wav)
    T = 1 + wav.shape[1] // 256
    t0, t1 = frames if frames is not None else (0, T)
    X = stft_f64(wav) if (t0, t1) == (0, T) and wav.shape[1] < 2_000_000 else stft_f64_frames(wav, t0, t1)
    val = np.concatenate([X.real, X.imag], 0).transpose(1, 2, 0)
    s = kappa * U * f64.pair_scale(np.abs(X).transpose(1, 2, 0), False)
    return val, np.concatenate([s, s], -1) + f64.R_OUT * U * np.abs(val)


# ---- to_waveform / Engine.istft (iris_istft: k_istft) ----
def istft_f64(spec, length=None):
    """torch.istft(n_fft=512, hop_length=256, periodic Hann, center=True, length) in float64 on the CPU of
    ``[.., 257, T, 2C]`` spectrograms in load_wav's layout (real parts, then imaginary parts) -> ``[.., C, L]``."""
    import warnings
    import torch
    x = torch.as_tensor(np.asarray(spec, np.float64))
    C = x.shape[-1] // 2
    z = torch.complex(x[..., :C], x[..., C:]).movedim(-1, -3)          # [.., C, 257, T]
    lead = z.shape[:-2]
    with warnings.catch_warnings():   # a length past the last frame is padded with zeros on purpose
        warnings.simplefilter('ignore', UserWarning)
        y = torch.istft(z.reshape(-1, 257, z.shape[-1]), 512, 256, window=torch.hann_window(512, dtype=torch.float64),
                        center=True, length=length)
    return y.reshape(*lead, y.shape[-1]).numpy()


def istft_weights(T, L):
    """The overlap-add weight of each covering frame, per output sample s = 256 h + r (r < 256) of ``L``:
    -> (hi [L], lo [L], h [L]).  Frame h contributes with ``hi`` (w[r + 256] / env[r] where frame h + 1 also covers
    s, 1 / w[r + 256] past the last frame's centre), frame h + 1 with ``lo`` (w[r] / env[r]); env[r] = w[r]^2 +
    w[r + 256]^2, w the periodic Hann window.  Both are 0 from s = 256 T on, where no frame covers s."""
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(512) / 512)
    s = np.arange(L)
    h, r = s // 256, s % 256
    env = w[r] ** 2 + w[r + 256] ** 2
    two = h + 1 < T
    hi = np.where(two, w[r + 256] / env, np.where(h < T, 1 / w[r + 256], 0.0))
    lo = np.where(two, w[r] / env, 0.0)
    return hi, lo, h


def istft_frame_norms(spec):
    """``[.., 257, T, 2C]`` -> ``[.., C, T]``: per channel, the L2 norm over bins 0 .. 256 of both channels of its
    channel pair (the complex FFT ``z = X_a + i X_b`` the kernel inverts), without the imaginary parts of bins 0
    and 256, which the inverse ignores."""
    x = np.asarray(spec, np.float64)
    C = x.shape[-1] // 2
    sq = x * x
    sq[..., [0, 256], :, C:] = 0
    e = sq[..., :C] + sq[..., C:]                                        # [.., 257, T, C]
    e = e.sum(-3)                                                        # [.., T, C]
    out = np.empty_like(e)
    for c0 in range(0, C, 2):
        out[..., c0:c0 + 2] = np.sqrt(e[..., c0:c0 + 2].sum(-1, keepdims=True))
    return np.swapaxes(out, -1, -2)


def istft_spread(per_frame, T, L):
    """Sum over the (at most two) frames covering each sample of the frame's weight times ``per_frame [.., T]``
    -> ``[.., L]``."""
    hi, lo, h = istft_weights(T, L)
    p = np.concatenate([per_frame, np.zeros(per_frame.shape[:-1] + (2,))], -1)
    hh = np.minimum(h, T)
    return hi * p[..., hh] + lo * p[..., hh + 1]


def istft_value_bound(spec, length=None):
    """to_waveform of ``[.., 257, T, 2C]`` -> (value, bound) ``[.., C, L]``.  The bound is KAPPA_ISTFT u S(s) +
    R_OUT u |value| + SUB_ISTFT 2^-149 G(s): S(s) sums, over the frames covering sample s, the frame's weight
    (istft_weights) times its channel pair's norm (istft_frame_norms) over sqrt(512); G(s) sums the weights of the
    covering frames whose pair is not all zero (rounding in the subnormal range, where u |x| no longer bounds it).
    A sample no frame covers, or only all-zero frames, has a bound of 0: it must be exactly 0."""
    x = np.asarray(spec, np.float64)
    T = x.shape[-2]
    L = 256 * (T - 1) if length is None else int(length)
    val = istft_f64(x, L)
    nrm = istft_frame_norms(x)
    S = istft_spread(nrm / math.sqrt(512), T, L)
    G = istft_spread((nrm > 0).astype(np.float64), T, L)
    return val, KAPPA_ISTFT * U * S + f64.R_OUT * U * np.abs(val) + SUB_ISTFT * TINY * G


def istft_carry(bound_spec, T, L):
    """How far an error of the spectrum, at most ``bound_spec [.., 257, T, 2C]`` per cell, moves the exact inverse
    -> ``[.., C, L]``: per frame and channel (|d0| + |d256| + 2 sum_{k=1}^{255} (|dRe_k| + |dIm_k|)) / 512 (the
    real inverse FFT; the imaginary parts of bins 0 and 256 are ignored), times the overlap-add weights."""
    b = np.asarray(bound_spec, np.float64)
    C = b.shape[-1] // 2
    e = b[..., 0, :, :C] + b[..., 256, :, :C] + 2 * (b[..., 1:256, :, :C] + b[..., 1:256, :, C:]).sum(-3)
    return istft_spread(np.swapaxes(e, -1, -2) / 512, T, L)


# ---- resample (k_resample) ----
def kaldi_table(orig, new):
    """The float32 filter table of orig -> new as append_kaldi_table / ``_lr_indices_and_weights`` build it ->
    (first [u_out] int64, weights [u_out, W] float32, sinc part |s| [u_out, W] float64, u_in, u_out)."""
    g = math.gcd(int(orig), int(new))
    u_in, u_out = orig // g, new // g
    cutoff = 0.99 * 0.5 * min(orig, new)
    width = 6 / (2.0 * cutoff)
    first, w = _lr_indices_and_weights(orig, new, u_out, width, cutoff, 6)
    t = np.arange(u_out, dtype=F32) / F32(new)
    dt = ((first.astype(F32)[:, None] + np.arange(w.shape[1], dtype=F32)[None, :]) / F32(orig) - t[:, None])
    dt = dt.astype(np.float64)
    with np.errstate(divide='ignore', invalid='ignore'):
        s = np.where(dt == 0, 2 * cutoff, np.abs(np.sin(2 * np.pi * cutoff * dt) / (np.pi * dt))) / orig
    return first, w, s, u_in, u_out


def resample_value_bound(wav, orig, new, table=None):
    """kaldi resample_waveform of ``wav [C, n_in]`` -> (value, bound) ``[C, n_out]``:
    value = sum_j w_ij x_k in float64 with the float32 table; bound = gamma_W sum_j |w_ij x_k| + u |y| +
    A_TAB u sum_j |s_ij x_k| (the two float32 tables, see A_TAB).  Local: a quiet stretch is held to its own
    scale."""
    wav = np.asarray(wav, np.float64)
    first, w, s, u_in, u_out = table if table is not None else kaldi_table(orig, new)
    C, n_in = wav.shape
    n_out = _lr_num_output_samples(n_in, orig, new)
    W = w.shape[1]
    n = np.arange(n_out)
    u, i = n // u_out, n % u_out
    k0 = first[i] + u * u_in
    val = np.zeros((C, n_out))
    aw = np.zeros((C, n_out))
    asx = np.zeros((C, n_out))
    w64 = w.astype(np.float64)
    for j in range(W):
        k = k0 + j
        ok = (k >= 0) & (k < n_in)
        x = np.where(ok, wav[:, np.clip(k, 0, n_in - 1)], 0.0)
        val += w64[i, j] * x
        aw += np.abs(w64[i, j] * x)
        asx += s[i, j] * np.abs(x)
    return val, gamma(W) * aw + U * np.abs(val) + A_TAB * U * asx + TINY


# ---- pointwise (k_pointwise) ----
def complex_to_magphase(x):
    """-> (value, bound, exact_cells) of ``complex_to_magphase`` on ``[..., 2C]`` (or mono_chan's 3 columns
    [re, im0, im1], re broadcast).  Magnitude: hypot, 3 u |m|; phase: arctan2, the atan2f bound.
    ``exact_cells``: the magnitude cells where the float32 ``a*a`` or ``b*b`` of the reference's formula under- or
    overflows; they are compared bit for bit with the float32 oracle (:func:`magnitude_f32`) instead."""
    x = np.asarray(x, np.float32)
    w = x.shape[-1]
    if w == 3:
        a, b = np.repeat(x[..., :1], 2, -1), x[..., 1:]
    else:
        a, b = x[..., :w // 2], x[..., w // 2:]
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    m = np.hypot(a64, b64)
    ph = np.arctan2(b64, a64)
    em = 3 * U * m
    eph = fn_bound(ph, ULP_ATAN2)
    with np.errstate(over='ignore', under='ignore'):
        aa, bb = a * a, b * b
    tiny = np.float32(np.finfo(np.float32).tiny)
    flow = lambda p, v: ~np.isfinite(p) | ((p < tiny) & (v != 0))
    exact = flow(aa, a) | flow(bb, b)
    return np.concatenate([m, ph], -1), np.concatenate([em, eph], -1), exact


def magnitude_f32(x):
    """The reference's float32 magnitude ``sqrt(re**2 + im**2)`` (transforms.py:111-123), broadcast for 3 columns."""
    x = np.asarray(x, np.float32)
    w = x.shape[-1]
    a, b = (np.repeat(x[..., :1], 2, -1), x[..., 1:]) if w == 3 else (x[..., :w // 2], x[..., w // 2:])
    with np.errstate(over='ignore', under='ignore'):
        return np.sqrt(a * a + b * b)


def magphase_to_complex(x):
    """``mag * cos(phase)``, ``mag * sin(phase)`` -> (value, bound): |mag| (cosf / sinf bound) + one rounding."""
    x = np.asarray(x, np.float32).astype(np.float64)
    n = x.shape[-1] // 2
    a, b = x[..., :n], x[..., n:]
    c, s = np.cos(b), np.sin(b)
    val = np.concatenate([a * c, a * s], -1)
    bnd = np.concatenate([np.abs(a) * fn_bound(c, ULP_SINCOS), np.abs(a) * fn_bound(s, ULP_SINCOS)], -1)
    return val, bnd + U * np.abs(val) + TINY


def log_eps(x):
    """``log(x + 1e-8f)`` -> (value, bound): the rounding of ``x + 1e-8f`` through the log, plus the logf bound."""
    v = np.asarray(x, np.float32).astype(np.float64) + EPS32
    with np.errstate(divide='ignore', invalid='ignore'):
        y = np.log(v)
        return y, f64.dlog(U * np.abs(v), v) + fn_bound(y, ULP_LOG)


def log_magphase(x, n_chan):
    """transforms.log_magphase: log(x + 1e-8) on the first ``n_chan`` columns, the rest passed through."""
    x = np.asarray(x, np.float32)
    y, e = log_eps(x)
    keep = np.arange(x.shape[-1]) >= n_chan
    return np.where(keep, x.astype(np.float64), y), np.where(keep, 0.0, e)


def multiply(x, scalar):
    """multiply_label: one correctly rounded product."""
    v = np.asarray(x, np.float32).astype(np.float64) * float(F32(scalar))
    return v, U * np.abs(v) + TINY


# ---- magphase_to_mel (k_mel_project) ----
def mel_value_bound(x, mel_w):
    """transforms.magphase_to_mel of ``[B, F, T, 2C]`` (or ``[F, T, 2C]``) with the float32 matrix promoted ->
    (value, bound) ``[B, n_mel, T, C]``: gamma_len[m] sum_f W |mag|, len[m] = the rows from the first to the last
    non-zero weight of band m (the kernel's fma chain)."""
    x = np.asarray(x, np.float32)
    w = np.asarray(mel_w, np.float32).astype(np.float64)
    squeeze = x.ndim == 3
    if squeeze:
        x = x[None]
    C = x.shape[-1] // 2
    mag = x[..., :C].astype(np.float64)
    nz = w != 0
    lo = np.argmax(nz, 0)
    hi = w.shape[0] - np.argmax(nz[::-1], 0)
    ln = np.where(nz.any(0), hi - lo, 0)
    val = np.einsum('bftc,fm->bmtc', mag, w)
    bnd = gamma(ln)[None, :, None, None] * np.einsum('bftc,fm->bmtc', np.abs(mag), w) + TINY
    return (val[0], bnd[0]) if squeeze else (val, bnd)


# ---- normalize (k_sumsq + k_rms_scale) ----
def normalize_value_bound(wav):
    """data_utils.normalize -> (value, bound): fp64 sum of squares (n u_64 relative), then float32 mean, sqrt,
    * 10 and the division: 4 u relative in all (0.5 u for the rounding of the mean through the sqrt)."""
    v = f64.normalize_f64(wav)
    return v, 4 * U * np.abs(v) + TINY


# ---- minmax / minmax_norm_magphase (k_minmax_reduce + k_minmax_apply): bit exact ----
def _total_order_key(x):
    u = np.ascontiguousarray(x, np.float32).view(np.uint32)
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def _extremum(x, axis, fn):
    """min / max under the IEEE total order (-0 < +0), the kernel's ordered-key reduction."""
    k = _total_order_key(x)
    i = fn(k, axis=axis, keepdims=True)
    return np.where(i & 0x80000000, i & 0x7fffffff, ~i).astype(np.uint32).view(np.float32)


def minmax_f32(x):
    """data_utils.minmax in the kernel's order: per sample (axis 0) ``(x - min) / max(max - min, 1e-8f)``, every
    operation one float32 rounding; the extrema are selections (-0 below +0)."""
    x = np.asarray(x, np.float32)
    ax = tuple(range(1, x.ndim))
    mn, mx = _extremum(x, ax, np.min), _extremum(x, ax, np.max)
    return ((x - mn) / np.maximum(mx - mn, F32(1e-8))).astype(np.float32)


def minmax_norm_magphase_f32(x):
    """transforms.minmax_norm_magphase in the kernel's order: magnitude half and phase half separately,
    ``(x - min) / ((max - min) + 1e-8f)``."""
    x = np.asarray(x, np.float32)
    n = x.shape[-1] // 2
    ax = tuple(range(1, x.ndim))
    out = []
    for h in (x[..., :n], x[..., n:]):
        mn, mx = _extremum(h, ax, np.min), _extremum(h, ax, np.max)
        out.append((h - mn) / ((mx - mn) + F32(1e-8)))
    return np.concatenate(out, -1).astype(np.float32)


# ---- cos_sim (k_cos_sim) ----
def cos_sim_value_bound(y_true, y_pred):
    """metrics.cos_sim -> (value, bound) ``[B]``.  Per class k: S = sum a p, A = sum a^2, P = sum p^2 (T terms,
    gamma_T each), cs_k = -S rsqrt(max(A, 1e-12)) rsqrt(max(P, 1e-12)) (two rsqrtf of (ULP_RSQRT + 1) ulp <= 6 u
    and half the relative error of A or P each, two products); then sum_k cs_k (occ_k / n_occ) over K terms
    (gamma_K, the quotient, the products)."""
    a = np.asarray(y_true, np.float32).astype(np.float64)
    p = np.asarray(y_pred, np.float32).astype(np.float64)
    B, T, K = a.shape
    S = (a * p).sum(1)
    eS = gamma(T) * np.abs(a * p).sum(1)
    A, P = (a * a).sum(1), (p * p).sum(1)
    rA, rP = 1 / np.sqrt(np.maximum(A, FLOOR12)), 1 / np.sqrt(np.maximum(P, FLOOR12))
    cs = -S * rA * rP
    rel = 2 * (0.5 * gamma(T) + 2 * (ULP_RSQRT + 1) * U) + 2 * U
    ecs = (eS * rA * rP + np.abs(cs) * rel) * (1 + 1e-6)
    occ = (a.sum(1) > 0).astype(np.float64)
    n = occ.sum(1, keepdims=True)
    wk = occ / np.maximum(n, float(F32(1e-8)))
    val = (cs * wk).sum(1)
    bnd = (ecs * wk).sum(1) + (gamma(K) + 2 * U) * np.abs(cs * wk).sum(1) + TINY
    return val, bnd


# ---- phase_vocoder (k_phase_vocoder): the magnitudes ----
def vocoder_steps(T, rate):
    """The host's tf.range(0, T, rate) arithmetic in float32 (challenge_b200/transforms.py) -> (i0, i1, alpha)."""
    n_steps = int(np.ceil(T / rate))
    steps = (F32(0) + np.arange(n_steps, dtype=F32) * F32(rate)).astype(F32)
    return steps.astype(np.int32), (steps + F32(1)).astype(np.int32), np.mod(steps, F32(1.))


def vocoder_magnitude(x, rate):
    """|output| of phase_vocoder ``[F, T, 2C]`` -> (value, bound) ``[F, T_out, C]``: the interpolation
    alpha n1 + (1 - alpha) n0 of the frame norms in float64 with the float32 alpha.  Bound: 2.5 u per norm
    (two products, a sum, sqrt), u for 1 - alpha and each of the three roundings of the interpolation, and the
    output's mag * cos / mag * sin: (ULP_SINCOS + 1) ulp of cos and sin (<= 6 u of the magnitude each) and the two
    products."""
    x = np.asarray(x, np.float32).astype(np.float64)
    F, T, C2 = x.shape
    C = C2 // 2
    i0, i1, al = vocoder_steps(T, rate)
    xp = np.concatenate([x, np.zeros((F, 2, C2))], 1)
    nrm = np.hypot(xp[..., :C], xp[..., C:])
    al = al.astype(np.float64)[None, :, None]
    t1, t0 = al * nrm[:, i1], (1 - al) * nrm[:, i0]
    val = t1 + t0
    bnd = (2.5 + 2) * U * t1 + (2.5 + 3) * U * t0 + (2 * 2 * (ULP_SINCOS + 1) + 2) * U * val
    return val, bnd * (1 + 1e-6) + TINY


# ---- bit-exact label / channel operations, numpy float32 in the kernel's order ----
def chan_map_f32(x, kind, factor=None):
    """k_chan_map: out = c0 * x[i0] (+ c1 * x[i1]); the products and the sum rounded separately.
    mono_chan ``x[..., :1] + x[..., 1:]``; stereo_mono ``[x0, x1, x0 + x1, x2, x3, x2 + x3]``; merge_aug(number)
    ``[re0, re1, f re0 + sqrt(1 - f) re1 ..., im0, im1, im0 + im1 ...]``."""
    x = np.asarray(x, np.float32)
    if kind == 'mono_chan':
        return (x[..., :1] + x[..., 1:]).astype(np.float32)
    if kind == 'stereo_mono':
        return np.concatenate([x[..., :2], x[..., :1] + x[..., 1:2], x[..., 2:4], x[..., 2:3] + x[..., 3:4]], -1)
    f = np.asarray(factor, np.float32).reshape(-1)
    c1 = np.sqrt(F32(1) - f)
    aug = [f[i] * x[..., 0:1] + c1[i] * x[..., 1:2] for i in range(f.size)]
    im = [x[..., 2:3] + x[..., 3:4] for _ in range(f.size)]
    return np.concatenate([x[..., :2]] + aug + [x[..., 2:4]] + im, -1).astype(np.float32)


def sum_voices_f32(y):
    """k_sum_axis (to_frame_labels): sum over the voice axis -3, voices in ascending order."""
    y = np.asarray(y, np.float32)
    acc = np.zeros(y.shape[:-3] + y.shape[-2:], np.float32)
    for v in range(y.shape[-3]):
        acc = acc + y[..., v, :, :]
    return acc


def avg_pool_time_f32(y, r, binarize):
    """k_avg_pool_time: Keras AveragePooling1D(r, r, 'same') on [B, T, K]; each window summed in ascending order,
    divided by its number of valid cells; ``binarize``: ``>= 0.5``."""
    y = np.asarray(y, np.float32)
    B, T, K = y.shape
    n = -(-T // r)
    left = max((n - 1) * r + r - T, 0) // 2
    out = np.zeros((B, n, K), np.float32)
    for i in range(n):
        lo, hi = max(i * r - left, 0), min(i * r - left + r, T)
        acc = np.zeros((B, K), np.float32)
        for t in range(lo, hi):
            acc = acc + y[:, t]
        out[:, i] = acc / F32(hi - lo)
    return (out >= F32(0.5)).astype(np.float32) if binarize else out


def sum_pool2_f32(y, scale):
    """k_sum_pool2 (one stage of preprocess_labels): ``((a + b) * 0.5) * 2`` per pair, a lone last cell ``a * 2``,
    then ``* scale`` unless scale is 1."""
    y = np.asarray(y, np.float32)
    B, T, K = y.shape
    n = (T + 1) // 2
    out = np.empty((B, n, K), np.float32)
    full = T // 2
    out[:, :full] = ((y[:, 0:2 * full:2] + y[:, 1:2 * full:2]) * F32(0.5)) * F32(2)
    if T % 2:
        out[:, full] = y[:, T - 1] * F32(2)
    return out if scale == 1 else (out * F32(scale)).astype(np.float32)


def preprocess_labels_f32(y, multiplier):
    for i in range(5):
        y = sum_pool2_f32(y, multiplier if i == 4 else 1.0)
    return y


def density_labels_f32(y):
    """k_density_labels (to_density_labels) on 0 / 1 labels ``[outer, V, T, K]``: each voice divided by max(its
    total, 1e-8) (an integer, exact in any order), then summed over the voices in ascending order."""
    y = np.asarray(y, np.float32)
    den = np.maximum(y.sum(axis=(-2, -1), dtype=np.float64).astype(np.float32), F32(1e-8))
    acc = np.zeros(y.shape[:-3] + y.shape[-2:], np.float32)
    for v in range(y.shape[-3]):
        acc = acc + y[..., v, :, :] / den[..., v, None, None]
    return acc


# ---- test signals ----
SIGNALS = ('white', 'pink', 'brown', 'tones', 'chirp', 'clicks', 'quiet', 'zeros', 'pair80', 'burst_tail', 'pair100',
           'dc_nyquist')


def signal(rng, kind, n_chan, n, sr=16000):
    """``challenge_b200.synth.structured_source`` kinds plus: ``burst_tail`` (white noise over the first fifth, then
    a tail 100 dB down), ``pair100`` (the odd channels at 1e-5 of their even partner), ``dc_nyquist`` (a DC level and
    an alternating-sign Nyquist tone, nothing else)."""
    from challenge_b200.synth import structured_source
    if kind in ('burst_tail', 'pair100', 'dc_nyquist'):
        if kind == 'burst_tail':
            x = rng.standard_normal((n_chan, n))
            x[:, max(n // 5, 1):] *= 1e-5
        elif kind == 'pair100':
            x = rng.standard_normal((n_chan, n))
            x[1::2] *= 1e-5
        else:
            x = 0.3 + 0.7 * (-1.0) ** np.arange(n)[None, :] * np.ones((n_chan, 1))
        x *= 0.1 / np.sqrt(np.mean(x * x))
        return x.astype(np.float32)
    return structured_source(rng, kind, n_chan, n, sr)


def span_values(rng, shape, signed=True):
    """float32 values spanning 1e-30 .. 1e18 in magnitude (log-uniform), with +-0, subnormals, the smallest
    normal and a few values whose square overflows, scattered over ``shape``."""
    v = 10.0 ** rng.uniform(-30, 18, size=shape)
    if signed:
        v *= rng.choice([-1.0, 1.0], size=shape)
    v = v.astype(np.float32).reshape(-1)
    special = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, 3e-39, np.finfo(np.float32).tiny, 1e19, -3e19, 1e-20,
                        1.0, -1.0, np.pi, 2 ** -75], np.float32)
    if not signed:
        special = np.abs(special)
        special[0] = 0.0
    pos = rng.choice(v.size, size=min(v.size, 4 * special.size), replace=False)
    v[pos] = np.resize(special, pos.size)
    return v.reshape(shape)
