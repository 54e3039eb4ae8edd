"""Float64 reference of the feature chain with a per-cell error bound (TEST INFRASTRUCTURE ONLY).

The chain -- sample synthesis, masks, channel remap, ``stft_filter``, magnitude / phase, log-magnitude, mel,
min-max + log, the 'se' blocks -- is computed in float64 from the same inputs and draws as the GPU.  Next to every
output value it computes the error a correct float32 implementation is allowed in that cell, from the size of the
terms that went into it rather than from the size of the clip:

complex cell     kappa_c * u * S, u = 2^-24.  Waveform banks: S is the L2 norm over the bins of one frame of the
                 un-mixed terms sum_s |g_s| |X_s|, over both channels of the channel pair that shares one complex
                 FFT (re = even channel, im = odd channel), so the quiet member of a pair is held to the loud
                 member's scale: an error of the FFT spreads over all bins of both channels.  Spectrogram banks run
                 no FFT: S is the cell's own term sum.
remapped channel the |coefficient|-weighted sum of the scales of its inputs (per real / imaginary column).
magnitude        hypot of the column scales; phase: that over |X|, plus A_ATAN (circular error).
log(x + 1e-8)    first-order -log1p(-dx / (x + 1e-8)), plus the ``__logf`` budget A_LOG_ABS + A_LOG_ULP ulp.
mel              sum_f W[f, m] * (magnitude scale of bin f) + kappa_m * u * mel.
min-max log-mel  propagated through (x - min) / (max - min) with the errors of the argmin / argmax cells (and of
                 every cell that could take their place); cells whose bound exceeds UNCONSTRAINED are reported as
                 unconstrained (bound = inf): near the clip minimum the log is ill-posed (SURVEY.md 7.3).
every output     plus R_OUT * u * |value|: the roundings of the value itself (sqrt, the last sum, the store).

kappa_c and kappa_m are calibrated on the CPU against the float32 oracle (torchaudio FFT, numpy mel) over the
signals of ``challenge_b200.synth.structured_banks`` and the white-noise banks: 4x the largest ratio measured
(tests/test_f64_bounds_host.py re-measures it).  The GPU is held to the same kappa plus the approximation terms.
"""
import numpy as np

from . import EPSILON
from .data_utils import stft_f64

U = 2.0 ** -24
# Largest |oracle - f64| / (u * S) over complex cells, and |fp32 mel - f64 mel| / (u * mel) of the fp32
# tensordot on exact magnitudes, measured over the calibration corpus of tests/test_f64_bounds_host.py.
MEASURED_RATIO_C = 1.1
MEASURED_RATIO_M = 2.8
KAPPA_C = 4 * MEASURED_RATIO_C
KAPPA_M = 4 * MEASURED_RATIO_M
R_OUT = 4
# fast_atan2f_mag_x2 (challenge_b200/csrc/iris_common.cuh): "|error| <= ~7e-7 rad"
A_ATAN = 7e-7
# __logf (MUFU.LG2 * ln 2; CUDA C Programming Guide, intrinsic functions): absolute error <= 2^-21.41 for x in
# [0.5, 2], otherwise <= 3 ulp
A_LOG_ABS = 2.0 ** -21.41
A_LOG_ULP = 3
UNCONSTRAINED = 1e-2


def normalize_f64(wav):
    """data_utils.py:32-34 in float64: ``wav / (10 * sqrt(mean(wav**2)))`` over all channels."""
    wav = np.asarray(wav, np.float64)
    return wav / (10.0 * np.sqrt(np.mean(wav * wav)))


def spec_f64(wav):
    """load_wav in float64: normalise, STFT, ``[F, T, 2C]`` layout (re | im)."""
    X = stft_f64(normalize_f64(wav))                    # [C, F, T]
    return np.concatenate([X.real, X.imag], 0).transpose(1, 2, 0).copy()


def bank_f64(items):
    """Waveforms ``[C, N]`` -> float64 spectra; spectrogram-bank items ``[F, T, 2C]`` promoted as they are."""
    return [np.asarray(x, np.float64) if np.ndim(x) == 3 else spec_f64(x) for x in items]


def _cmag(x):
    C = x.shape[-1] // 2
    return np.hypot(x[..., :C], x[..., C:])


def synth_index_level(bg, voices, vlabels, noises, d, b, K=3, keep=None, detail=False):
    """Independent restatement of sample synthesis from the INDEX-LEVEL semantics (SURVEY.md appendix
    A.2), frame by frame in float64, sharing no code with oracle/pipeline.py (which pads, slices and
    adds whole tensors like the reference does): out[f,t] = BG[f,(t+o_b) mod bgT] + sum over kept
    voices of g_v X_v[f, t+off_v-s_v] + sum over noises; labels and keep flags by the same indices.

    ``keep``: the keep flags to use instead of the ones derived here (the voice activity behind them is a
    ``> 0`` test on the spectrum, which rounding can decide differently for a frame of silence).
    ``detail``: return a dict with the mix ``x``, ``voice`` (kept voices) and ``noise`` (background +
    noises) ``[F, T, 2C]`` and their term sums ``ax`` / ``av`` / ``an`` = sum_s g_s |X_s| ``[F, T, C]``."""
    T = d.n_frame
    V, M = d.max_voices, d.max_noises
    BG = np.asarray(bg[int(d.bg_id[b])], np.float64)
    bgT = BG.shape[1]
    idx = (np.arange(T) + int(d.bg_offset[b])) % bgT
    noise = BG[:, idx].copy()
    an = _cmag(BG)[:, idx]
    voice = np.zeros_like(noise)
    av = np.zeros_like(an)
    label = np.zeros((V, T, K), np.float64)
    flags = [0] * V
    if V:
        ids = [int(i) for i in d.voice_id[b]]
        vP = max(voices[i].shape[1] for i in ids)                      # padded_batch: the group's longest
        pad = T - int(np.int32(np.float32(d.min_ratio) * np.float32(vP)))
        s = pad if pad > 0 else 0
        nv = int(d.n_voices[b]) if V > 1 else 1
        L = np.zeros((T, K), np.float64)
        for v in range(nv):
            X = np.asarray(voices[ids[v]], np.float64)
            kT = X.shape[1]
            act = (X.max(axis=(0, 2)) > 0)
            cand = np.zeros((T, K), np.float64)
            src = [t + int(d.voice_offset[b][v]) - s for t in range(T)]
            for t, k in enumerate(src):
                if 0 <= k < kT and act[k]:
                    cand[t] = np.asarray(vlabels[ids[v]], np.float64)
            ok = not ((L + cand) >= 2).any()
            if keep is not None:
                ok = bool(keep[v])
            flags[v] = int(ok)
            if ok:
                g = float(d.voice_gain[b][v])
                mag = _cmag(X)
                for t, k in enumerate(src):
                    if 0 <= k < kT:
                        voice[:, t] += g * X[:, k]
                        av[:, t] += g * mag[:, k]
                L += cand
                label[v] = cand
    if M:
        ids = [int(i) for i in d.noise_id[b]]
        nP = max(noises[i].shape[1] for i in ids)
        pad = T - int(np.int32(np.float32(d.min_noise_ratio) * np.float32(nP)))
        s = pad if pad > 0 else 0
        for n in range(int(d.n_noises[b])):
            X = np.asarray(noises[ids[n]], np.float64)
            mag = _cmag(X)
            g = float(d.noise_gain[b][n])
            for t in range(T):
                k = t + int(d.noise_offset[b][n]) - s
                if 0 <= k < X.shape[1]:
                    noise[:, t] += g * X[:, k]
                    an[:, t] += g * mag[:, k]
    if detail:
        return dict(x=voice + noise, voice=voice, noise=noise, ax=av + an, av=av, an=an, label=label, keep=flags)
    return voice + noise, label, flags


def activity_ambiguous(X, spec_banks):
    """Frames of a float64 voice spectrum ``[F, T, 2C]`` whose voice activity (``max > 0`` over the frame,
    pipeline.py:55) a correct float32 FFT may decide either way: the largest coefficient is not exactly 0 but
    within kappa_c * u * (L2 norm of the frame) of it.  Spectrogram banks hold the float32 values themselves:
    nothing is ambiguous there."""
    X = np.asarray(X, np.float64)
    if spec_banks:
        return np.zeros(X.shape[1], bool)
    m = X.max(axis=(0, 2))
    s = np.sqrt((X * X).sum(axis=(0, 2)))
    return (m != 0) & (np.abs(m) <= KAPPA_C * U * s)


def keep_decidable(voices, d, b, spec_banks):
    """True if no voice of clip ``b`` has a frame of ambiguous activity: its keep flags are then determined."""
    if not d.max_voices:
        return True
    nv = int(d.n_voices[b]) if d.max_voices > 1 else 1
    return not any(activity_ambiguous(voices[int(i)], spec_banks).any() for i in d.voice_id[b][:nv])


def pair_scale(a, spec_banks):
    """Error scale of every (bin, frame, channel) from the term sums ``a`` ``[F, T, C]``: the L2 norm over the
    bins of the frame and both channels of its FFT pair (waveform banks), the cell itself (spectrogram banks)."""
    if spec_banks:
        return a.copy()
    F, T, C = a.shape
    s = np.empty_like(a)
    for c0 in range(0, C, 2):
        c1 = min(c0 + 2, C)
        s[:, :, c0:c1] = np.sqrt((a[:, :, c0:c1] ** 2).sum(axis=(0, 2)))[None, :, None]
    return s


def remap(x, kind, factor=None, n_out=0):
    """The channel remaps on ``[..., 2C]`` re | im columns (data_utils.py:73-117), in float64.  Every coefficient
    is >= 0, so applied to column error scales this is their |coefficient|-weighted sum."""
    if kind is None:
        return x
    if kind == 'stereo_mono':
        return np.concatenate([x[..., :2], x[..., :1] + x[..., 1:2], x[..., 2:4], x[..., 2:3] + x[..., 3:4]], -1)
    if kind == 'mono_chan':                     # [re0 + re1, re0 + im0, re0 + im1]
        return x[..., :1] + x[..., 1:]
    if kind == 'merge_aug':
        f = np.asarray(factor, np.float32).astype(np.float64)
        assert f.shape == (n_out - 2,)
        re, im = x[..., :2], x[..., 2:]
        aug_re = f * re[..., :1] + np.sqrt(1.0 - f) * re[..., 1:]
        aug_im = np.repeat(im[..., :1] + im[..., 1:], n_out - 2, -1)
        return np.concatenate([re, aug_re, im, aug_im], -1)
    raise ValueError(kind)


def dlog(e, v):
    """Bound of |log(v') - log(v)| for |v' - v| <= e, v > 0 (inf where e >= v)."""
    e = np.asarray(e, np.float64)
    v = np.asarray(v, np.float64)
    r = np.divide(e, v, out=np.full(np.broadcast(e, v).shape, np.inf), where=v > 0)
    out = np.full(r.shape, np.inf)
    ok = r < 1
    out[ok] = -np.log1p(-r[ok])
    return out


def log_budget(y, gpu):
    """``__logf`` budget of an output y = log(...) (0 for the float32 oracle's correctly rounded np.log)."""
    if not gpu:
        return 0.0
    return A_LOG_ABS + A_LOG_ULP * np.spacing(np.abs(y).astype(np.float32)).astype(np.float64)


def _minmax_log(mel, emel, gpu):
    """data_utils.minmax + log_on_mel of one clip with its bound; cells above UNCONSTRAINED get inf."""
    lo_i = np.argmin(mel)
    hi_i = np.argmax(mel)
    mn, mx = mel.flat[lo_i], mel.flat[hi_i]
    # the computed minimum lies in [min(x - e), x_argmin + e_argmin]; the maximum likewise
    dmn = max(mn - (mel - emel).min(), emel.flat[lo_i])
    dmx = max((mel + emel).max() - mx, emel.flat[hi_i])
    R = mx - mn
    dR = dmn + dmx
    den = max(R, EPSILON)
    y = (mel - mn) / den
    if R - dR > EPSILON:
        ey = (emel + dmn + y * dR) / (R - dR) + R_OUT * U * y
    else:
        ey = np.full(mel.shape, np.inf)
    z = np.log(y + EPSILON)
    ez = dlog(ey, y + EPSILON) + log_budget(z, gpu) + R_OUT * U * np.abs(z)
    ez[~(ez <= UNCONSTRAINED)] = np.inf
    return z, ez


MODES = ('complex', 'magphase', 'log_magphase', 'mel', 'logmel', 'logmel_minmax', 'se')


def clip_features(banks, vlabels, d, b, mode, spec_banks, remap_kind=None, n_out=0, stft_filter=0, mel_w=None,
                  keep=None, gpu=True, kappa_c=KAPPA_C, kappa_m=KAPPA_M, cache=None):
    """One clip of ``mode`` -> ``(value, bound)`` in the layout of the features (``[F or n_mel, T, cols]``); for
    'se' a list of three such pairs (x, only_voice, only_noise).  ``banks`` = float64 (bg, voices, noises)
    from :func:`bank_f64`; ``gpu`` adds the approximation terms of the CUDA kernels; ``cache``: a dict that keeps
    the synthesis of the clip for further modes on the same draws."""
    bg, voices, noises = banks
    if cache is not None and b in cache:
        det = cache[b]
    else:
        det = synth_index_level(bg, voices, vlabels, noises, d, b, K=len(vlabels[0]) if vlabels is not None else 3,
                                keep=keep, detail=True)
        if cache is not None:
            cache[b] = det
    x = det['x']
    F, T, W = x.shape
    C = W // 2
    m = np.ones((F, T, 1))
    if d.time_masks is not None:
        for size, off in d.time_masks[b]:
            m[:, int(off):int(off) + int(size)] = 0
    if d.freq_masks is not None:
        for size, off in d.freq_masks[b]:
            m[int(off):int(off) + int(size)] = 0
    if stft_filter:
        m[1:1 + stft_filter] = 0
    if mode == 'se':
        sv = kappa_c * U * pair_scale(det['av'], spec_banks)[..., :C]
        sn = kappa_c * U * pair_scale(det['an'], spec_banks)[..., :C]
        xv = x * m
        out = [(xv[1:, :, :C], ((sv + sn) * m)[1:]), (det['voice'][1:, :, :C // 2], sv[1:, :, :C // 2]),
               (det['noise'][1:, :, :C // 2], sn[1:, :, :C // 2])]
        return [(v, e + R_OUT * U * np.abs(v)) for v, e in out]
    e = kappa_c * U * pair_scale(det['ax'], spec_banks)
    e = np.concatenate([e, e], -1)
    factor = d.merge_factor[b] if remap_kind == 'merge_aug' else None
    x = remap(x * m, remap_kind, factor, n_out)
    e = remap(e * m, remap_kind, factor, n_out)
    if mode == 'complex':
        return x, e + R_OUT * U * np.abs(x)
    n = x.shape[-1] // 2
    re, im, ere, eim = x[..., :n], x[..., n:], e[..., :n], e[..., n:]
    mag = np.hypot(re, im)
    emag = np.hypot(ere, eim) + R_OUT * U * mag
    if mode in ('magphase', 'log_magphase'):
        ph = np.arctan2(im, re)
        eph = np.divide(np.hypot(ere, eim), mag, out=np.full(mag.shape, np.inf), where=mag > 0)
        eph = eph + (A_ATAN if gpu else 0.0) + R_OUT * U * np.abs(ph)
        if mode == 'log_magphase':
            lm = np.log(mag + EPSILON)
            elm = dlog(emag, mag + EPSILON) + log_budget(lm, gpu) + R_OUT * U * np.abs(lm)
            return np.concatenate([lm, ph], -1), np.concatenate([elm, eph], -1)
        return np.concatenate([mag, ph], -1), np.concatenate([emag, eph], -1)
    w = np.asarray(mel_w, np.float32).astype(np.float64)          # the product's float32 matrix, promoted
    mel = np.einsum('ftc,fm->mtc', mag, w)
    emel = np.einsum('ftc,fm->mtc', emag, w) + kappa_m * U * mel
    if mode == 'mel':
        return mel, emel
    if mode == 'logmel':
        lg = np.log(mel + EPSILON)
        return lg, dlog(emel, mel + EPSILON) + log_budget(lg, gpu) + R_OUT * U * np.abs(lg)
    assert mode == 'logmel_minmax', mode
    return _minmax_log(mel, emel, gpu)


def features(banks, vlabels, d, mode, spec_banks, clips=None, keep=None, **kw):
    """:func:`clip_features` of every clip, stacked -> ``(value [B, ...], bound [B, ...])`` or, for 'se', three
    such pairs.  ``keep``: per-clip keep flags ``[B, V]`` (e.g. the GPU's) or None."""
    clips = range(d.batch) if clips is None else clips
    per = [clip_features(banks, vlabels, d, b, mode, spec_banks, keep=None if keep is None else keep[b], **kw)
           for b in clips]
    if mode == 'se':
        return [(np.stack([p[i][0] for p in per]), np.stack([p[i][1] for p in per])) for i in range(3)]
    return np.stack([p[0] for p in per]), np.stack([p[1] for p in per])


def phase_columns(mode, width):
    """Boolean mask of the phase columns of a feature of ``width`` columns (magphase / log_magphase)."""
    cols = np.zeros(width, bool)
    if mode in ('magphase', 'log_magphase'):
        cols[width // 2:] = True
    return cols


def ratio(got, ref, bound, mode):
    """|got - ref| / bound per cell (circular difference in the phase columns); 0 where both are equal, inf
    where a bound of 0 is exceeded.  Unconstrained cells (bound inf) give 0 for a finite value; a NaN or an
    infinity where the reference is finite gives inf, whatever the bound."""
    got = np.asarray(got, np.float64)
    with np.errstate(invalid='ignore', over='ignore'):
        diff = np.abs(got - ref)
        ph = phase_columns(mode, got.shape[-1])
        if ph.any():
            diff[..., ph] = np.abs(np.angle(np.exp(1j * (got[..., ph] - ref[..., ph]))))
    with np.errstate(divide='ignore', invalid='ignore'):
        r = np.where(got == ref, 0.0, diff / bound)
    r[np.isnan(r) | (~np.isfinite(got) & np.isfinite(ref))] = np.inf
    return r


def worst(r):
    """(largest ratio, its index)."""
    i = np.unravel_index(np.argmax(r), r.shape)
    return float(r[i]), tuple(int(v) for v in i)
