"""Every stand-alone drop-in operation (include/iris.h, second half: k_ops.cu, k_resample.cu, iris_stft) against the
float64 values and per-cell bounds of oracle/f64_ops.py, or bit for bit against the float32 form in the kernel's
order, at the shapes where kernels go wrong: the launchers' splits and grid-stride loops, the size limits of
iris_ops_abi.cu at the limit and one past it, T = 1, the shortest clip load_wav takes, odd channel counts, long
files, and signals with quiet tails, quiet channels, exact zeros and DC / Nyquist tones.  The evaluation feature
chain of ``metrics.evaluate`` is checked stage by stage, each stage fed the GPU output of the one before, so that
every bound is an exact-input bound.  Per configuration one line: the largest ratio error / bound, where it
occurs, and the normalised max error beside it (profiles/r11_ops_f64.txt).  Of the evaluation-side operations
(k_eval.cu, checked against the oracle in tests/test_eval_chain.py) only get_er's row limits are tested here."""
import ctypes as C

import numpy as np
import pytest

from conftest import nmax_err
from oracle import f64, f64_ops as F

pytestmark = pytest.mark.gpu

_lines = []


def _np(t):
    return t.detach().float().cpu().numpy()


@pytest.fixture(scope='module')
def mods(engine):
    import challenge_b200
    from challenge_b200 import data_utils, engine as E, metrics, trainer, transforms
    E._engines[0] = engine          # share the session engine
    challenge_b200.set_seed(0)
    yield transforms, data_utils, metrics, trainer
    engine.set_mel(80)


def _line(tag, r, at, nm):
    line = '%-64s ratio %9.3g at %-22s nmax %.2e' % (tag, r, str(at), nm)
    _lines.append(line)
    print(line)
    return r


def check(tag, got, val, bnd, fails=None):
    """One configuration against its bound; appends (tag, ratio) to ``fails`` when the ratio exceeds 1."""
    got = np.asarray(got)
    assert got.shape == val.shape, (tag, got.shape, val.shape)
    if got.size == 0:
        return _line(tag + ' (empty)', 0.0, (), 0.0)
    r, at = f64.worst(F.ratio(got, val, bnd))
    with np.errstate(invalid='ignore', over='ignore'):
        nm = nmax_err(np.where(np.isfinite(val), got, 0), np.where(np.isfinite(val), val, 0))
    _line(tag, r, at, nm)
    if fails is not None and not r <= 1:
        fails.append((tag, r, at))
    return r


def check_exact(tag, got, ref, fails):
    got = np.asarray(got, np.float32)
    r, at = f64.worst(F.bitexact_ratio(got, ref))
    _line(tag + ' (bit exact)', r, at, nmax_err(got, ref) if got.size else 0.0)
    if r != 0:
        fails.append((tag, r, at))


def _sig(kind, C, n, seed):
    return F.signal(np.random.default_rng(seed), kind, C, n)


# ---- load_wav / Engine.stft ----
LOAD_N = (257, 300, 511, 512, 513, 767, 768, 769, 48000, 48001, 48255)


def test_load_wav(engine, mods):
    """Every n x C in 1..5 on a structured signal each (normalize on / off and device / host input alternating);
    the imaginary parts of bins 0 and 256 are exactly +0."""
    import torch
    _, D, _, _ = mods
    fails = []
    k = 0
    for n in LOAD_N:
        for C in (1, 2, 3, 4, 5):
            kind = F.SIGNALS[k % len(F.SIGNALS)]
            norm, dev = k % 3 != 2, k % 2 == 1
            w = _sig(kind, C, n, k)
            src = torch.from_numpy(w).cuda() if dev else w
            got = _np(D.load_wav(src) if norm and k % 4 == 0 else engine.stft(src, normalize=norm))
            val, bnd = F.stft_value_bound(w, normalize=norm)
            check('load_wav n=%d C=%d %s norm=%d %s' % (n, C, kind, norm, 'device' if dev else 'host'), got, val, bnd,
                  fails=fails)
            im = got[[0, 256], :, C:]
            if im.any() or np.signbit(im).any():
                fails.append(('bins 0 / 256 imaginary not +0', n, C))
            k += 1
    assert not fails, fails


def test_load_wav_30_minute_stereo(engine, mods):
    """One 30-minute stereo file (T = 112501), checked in blocks of frames."""
    w = _sig('pink', 2, 30 * 60 * 16000, 1)
    got = _np(engine.stft(w))
    assert got.shape == (257, 112501, 4)
    wn = f64.normalize_f64(w)
    fails, worst = [], (0.0, None)
    for t0 in range(0, 112501, 8192):
        t1 = min(t0 + 8192, 112501)
        val, bnd = F.stft_value_bound(wn, normalize=False, frames=(t0, t1))
        r, at = f64.worst(F.ratio(got[:, t0:t1], val, bnd))
        if r > worst[0]:
            worst = (r, (at[0], at[1] + t0, at[2]))
    _line('load_wav 30 min stereo T=112501 pink', worst[0], worst[1], float('nan'))
    assert worst[0] <= 1, worst


def test_stft_pair_stride_limit_refused(engine):
    """A 3-channel source of 1073741312 samples would need a pair-plane stride above 2^31 - 1 floats: refused by
    iris_stft and by the bank registration before anything is copied (a real device tensor of that size)."""
    import torch
    from challenge_b200 import _lib as L
    n = 1073741312
    if torch.cuda.mem_get_info()[0] < 64 << 30:
        pytest.skip('needs 64 GB of free device memory')
    w = torch.empty((3, n), dtype=torch.float32, device='cuda')
    with pytest.raises(NotImplementedError, match='pair stride'):
        engine.stft(w)
    off = np.array([0, n], np.int64)
    rc = engine.lib.iris_bank_register(engine._ctx, L.BANK_BG, 1, 3, C.c_void_p(w.data_ptr()), off.ctypes.data, None,
                                       0, 1, engine._stream())
    assert rc == L.IRIS_ERR_UNSUPPORTED
    assert 'pair stride' in L.load().iris_last_error().decode()
    del w
    torch.cuda.empty_cache()


# ---- resample ----
def test_resample(engine):
    """Down from 22050 / 32000 / 44100 / 48000 / 96000, up from 8000 / 11025 / 12000, and 44101 -> 16000 (a table of
    2.2 MB: the global-table path); n_in in {1, 2, W - 1, W, 30001}; every output within its local bound."""
    import torch
    fails = []
    for orig in (22050, 32000, 44100, 48000, 96000, 8000, 11025, 12000, 44101):
        table = F.kaldi_table(orig, 16000)
        W = table[1].shape[1]
        for j, n in enumerate((1, 2, W - 1, W, 30001)):
            kind = ('burst_tail', 'pair100', 'dc_nyquist', 'white', 'burst_tail')[j]
            w = _sig(kind, 2, n, orig + n) if n > 2 else np.float32([[0.5, -0.25][:n], [1e-6, 3e-7][:n]])
            src = torch.from_numpy(w).cuda() if j % 2 else w
            got = _np(engine.resample(src, orig, 16000))
            val, bnd = F.resample_value_bound(w, orig, 16000, table)
            check('resample %d -> 16000 n_in=%d W=%d %s' % (orig, n, W, kind), got, val, bnd, fails=fails)
    # 5 minutes at 48 kHz: 4.8 M outputs, chunks of 4096
    w = _sig('burst_tail', 2, 48000 * 300, 3)
    got = _np(engine.resample(w, 48000, 16000))
    check('resample 48000 -> 16000 5 min (chunk 4096)', got, *F.resample_value_bound(w, 48000, 16000), fails=fails)
    assert not fails, fails


def test_bank_of_mixed_rates_item_by_item(engine):
    """iris_bank_register_audio on a bank of items at 44101 / 22050 / 8000 / 16000 Hz: the complex features of each
    item (one clip per item, background only) against the float64 STFT of the float64 resampled item; the bound is
    the fused 'complex' cell plus the resampler's bound carried through the window."""
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    rates = (44101, 22050, 8000, 16000)
    items = [(_sig(kind, 2, int(1.3 * r), r), r) for kind, r in zip(('burst_tail', 'tones', 'pair80', 'chirp'), rates)]
    frames = engine.register_bank(L.BANK_BG, items)
    other = [_sig('white', 2, 4000, 1)]                   # 2-channel voice / noise banks the plan does not draw from
    engine.register_bank(L.BANK_VOICE, other, labels=np.eye(3, dtype=np.float32)[[0]])
    engine.register_bank(L.BANK_NOISE, other)
    T = int(frames.min())
    d = draw_batch(np.random.default_rng(0), len(items), T, frames)
    d.bg_id[:] = np.arange(len(items))
    d.bg_offset[:] = 0
    engine.upload_plan(d)
    got = _np(engine.features(L.FEAT_COMPLEX))
    hann = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(512) / 512)
    fails = []
    for b, (w, r) in enumerate(items):
        if r == 16000:
            x, ex = w.astype(np.float64), np.zeros(w.shape)
        else:
            x, ex = F.resample_value_bound(w, r, 16000)
        rms10 = 10 * np.sqrt(np.mean(x * x))
        rho = np.sqrt(np.mean(ex * ex)) * 10 / rms10      # |rms' / rms - 1| <= ||e|| / ||x||
        xn, ex = x / rms10, ex / rms10
        val, bnd = F.stft_value_bound(xn, normalize=False, frames=(0, T))
        bnd = bnd + rho * np.abs(val)
        N = xn.shape[1]
        idx = np.abs(256 * np.arange(T)[:, None] + np.arange(512)[None, :] - 256)
        idx = np.where(idx > N - 1, 2 * (N - 1) - idx, idx)
        # the resampler's bound and the rounding of each normalised sample (the division by the RMS), carried
        # through the analysis window of each frame: local to the frame, like every other term
        carry = ((ex[:, idx] + F.U * np.abs(xn[:, idx])) * hann).sum(-1) * (1 + 8 * F.U)     # [C, T]
        bnd = bnd + np.concatenate([carry.T, carry.T], -1)[None]
        check('bank item %d at %d Hz, T=%d' % (b, r, T), got[b], val, bnd, fails=fails)
    assert not fails, fails


# ---- pointwise ----
def test_pointwise(mods):
    """complex_to_magphase (incl. mono_chan's 3 columns), magphase_to_complex, log_magphase, log_on_mel and
    multiply_label on values spanning 1e-30 .. 1e18 with +-0, subnormals and squares that overflow; T = 1 too."""
    TR, D, _, _ = mods
    rng = np.random.default_rng(5)
    fails = []
    for shape in ((257, 70, 6), (257, 1, 2), (13000, 50, 4)):      # 2.6 M cells: the grid-stride loop iterates
        x = F.span_values(rng, shape)
        got = _np(TR.complex_to_magphase(x))
        val, bnd, exact = F.complex_to_magphase(x)
        c = shape[-1] // 2
        m32 = F.magnitude_f32(x)
        if not np.array_equal(got[..., :c][exact].view(np.uint32), m32[exact].view(np.uint32)):
            fails.append(('complex_to_magphase over / underflow cells not bit exact', shape))
        val[..., :c][exact] = m32[exact]
        check('complex_to_magphase %s (%d cells bit exact)' % (shape, exact.sum()), got, val, bnd, fails)
    x = F.span_values(rng, (257, 40, 3))
    got = _np(TR.complex_to_magphase(x))
    val, bnd, exact = F.complex_to_magphase(x)
    m32 = F.magnitude_f32(x)
    val[..., :2][exact] = m32[exact]
    check('complex_to_magphase mono_chan [re, im0, im1]', got, val, bnd, fails)
    for shape in ((257, 70, 6), (5, 257, 1, 2)):
        n = shape[-1] // 2
        mp = np.concatenate([F.span_values(rng, shape[:-1] + (n,), signed=False),
                             F.span_values(rng, shape[:-1] + (n,))], -1)
        check('magphase_to_complex %s' % (shape,), _np(TR.magphase_to_complex(mp)), *F.magphase_to_complex(mp),
              fails=fails)
        pos = F.span_values(rng, shape, signed=False)
        check('log_magphase %s' % (shape,), _np(TR.log_magphase(pos, n_chan=n)), *F.log_magphase(pos, n),
              fails=fails)
        check('log_on_mel %s' % (shape,), _np(D.log_on_mel(pos)), *F.log_eps(pos), fails=fails)
        xs = F.span_values(rng, shape)
        check('multiply_label 0.3 %s' % (shape,), _np(D.multiply_label(0.3)(None, xs)[1]), *F.multiply(xs, 0.3),
              fails=fails)
    assert not fails, fails


def test_normalize(mods):
    _, D, _, _ = mods
    fails = []
    for i, (kind, shape) in enumerate((('pair80', (2, 160000)), ('burst_tail', (4, 40001)), ('pair100', (2, 300)),
                                       ('white', (3, 7)), ('dc_nyquist', (1, 4096)), ('white', (2, 600000)))):
        w = _sig(kind, shape[0], shape[1], i) if shape[1] > 8 else _sig('white', *shape, i)
        check('normalize %s %s' % (kind, shape), _np(D.normalize(w)), *F.normalize_value_bound(w), fails=fails)
    assert not fails, fails


# ---- magphase_to_mel ----
def _mags(B, C, T, seed):
    from oracle import data_utils as OD, transforms as OT
    out = []
    for b in range(B):
        kind = ('brown', 'tones', 'chirp', 'dc_nyquist', 'burst_tail', 'zeros')[(b + seed) % 6]
        w = _sig(kind, C, max(256 * (T - 1), 257), seed + b)
        out.append(OT.complex_to_magphase(OD.load_wav_array(w))[:, :T])
    return np.stack(out).astype(np.float32)


def test_magphase_to_mel(engine, mods):
    """80 (default) / 40 bands, 128 bands to 8000 Hz (support reaches bin 256), lower edge 0 (bin 0 in the support);
    T = 1, C in {1, 3}, unbatched input; and one input of 1.28 M outputs: more than the 148 * 16 CTAs of the capped
    grid cover (1,212,416 at two outputs per thread), so the grid-stride loop iterates."""
    from challenge_b200.engine import default_mel_matrix
    TR, _, _, _ = mods
    fails = []
    try:
        for n_mel, kw in ((80, {}), (40, {}), (128, dict(upper_edge_hertz=8000.0)), (80, dict(lower_edge_hertz=0.0))):
            mw = default_mel_matrix(n_mel, 257, 16000, **kw)
            for B, C, T in ((2, 2, 40), (1, 1, 1), (3, 3, 17)):
                x = _mags(B, C, T, n_mel + C)
                check('mel %d %s B=%d C=%d T=%d' % (n_mel, kw, B, C, T), _np(TR.magphase_to_mel(n_mel, **kw)(x)),
                      *F.mel_value_bound(x, mw), fails=fails)
            x = _mags(1, 2, 30, 1)[0]
            check('mel %d %s unbatched' % (n_mel, kw), _np(TR.magphase_to_mel(n_mel, **kw)(x)),
                  *F.mel_value_bound(x, mw), fails=fails)
        x = _mags(4, 2, 2000, 3)
        check('mel 80 B=4 C=2 T=2000 (capped grid, grid-stride)', _np(TR.magphase_to_mel(80)(x)),
              *F.mel_value_bound(x, default_mel_matrix(80, 257, 16000)), fails=fails)
    finally:
        engine.set_mel(80)
    assert not fails, fails


# ---- minmax / minmax_norm_magphase ----
def test_minmax(mods):
    """40000 samples (the 32768 split of launch_minmax), 320 k cells per sample (64 CTAs per sample in the atomics),
    -0.0 as a minimum, a constant sample, an all-negative sample, and the unbatched per-row quirk."""
    TR, D, _, _ = mods
    rng = np.random.default_rng(9)
    fails = []
    x = rng.standard_normal((40000, 5, 2)).astype(np.float32)
    x[7] = 2.5
    x[32769] = -np.abs(x[32769]) - 1
    x[32767] = np.abs(x[32767])
    x[32767, 0, 0] = -0.0
    x[32767, 1, 1] = 0.0
    for name, y in (('minmax [40000, 5, 2]', x), ('minmax [3, 80, 2000, 2]',
                                                  (rng.standard_normal((3, 80, 2000, 2)) * 7).astype(np.float32)),
                    ('minmax unbatched [80, 63, 2] (per row)', _mags(1, 2, 63, 2)[0, :80, :, :2].copy())):
        check_exact(name, _np(D.minmax(y)), F.minmax_f32(y), fails)
    z = np.abs(rng.standard_normal((40000, 3, 4))).astype(np.float32)
    z[5] = -1.5
    z[32770, ..., :2] = -np.abs(z[32770, ..., :2]) - 0.5
    z[40, 0, 0] = -0.0
    for name, y in (('minmax_norm_magphase [40000, 3, 4]', z),
                    ('minmax_norm_magphase [2, 257, 700, 4]', _mags(2, 2, 700, 4)),
                    ('minmax_norm_magphase unbatched [257, 30, 4]', _mags(1, 2, 30, 5)[0])):
        check_exact(name, _np(TR.minmax_norm_magphase(y)), F.minmax_norm_magphase_f32(y), fails)
    assert not fails, fails


# ---- cos_sim ----
def test_cos_sim(mods):
    """K = 1 .. 8 at T = 200 and T = 1, with a sample of no class, an all-zero prediction and predictions below the
    1e-12 floor; K = 9 refused."""
    _, _, MT, _ = mods
    rng = np.random.default_rng(10)
    fails = []
    for K in range(1, 9):
        for T in (200, 1):
            yt = (rng.random((16, T, K)) < 0.3).astype(np.float32)
            yt[3] = 0
            yp = np.clip(yt + rng.normal(0, 0.35, yt.shape), 0, 1).astype(np.float32)
            yp[4] = 0
            yp[5] *= np.float32(1e-8)
            check('cos_sim K=%d T=%d' % (K, T), _np(MT.cos_sim(yt, yp)), *F.cos_sim_value_bound(yt, yp), fails=fails)
    with pytest.raises(NotImplementedError):
        MT.cos_sim(np.ones((2, 5, 9), np.float32), np.ones((2, 5, 9), np.float32))
    assert not fails, fails


# ---- phase_vocoder ----
def test_phase_vocoder_magnitudes(mods):
    """|output| against the float64 interpolation of the frame norms: rates {0.3, 0.7, 1.5, 3.0, 1.0001} x T in
    {1, 2, 5, 626} x F in {2, 257} x C in {1, 3}; T_out = 5461 accepted, 5462 refused."""
    from oracle import data_utils as OD
    TR, _, _, _ = mods
    fails = []
    for F_ in (2, 257):
        for C_ in (1, 3):
            for T in (1, 2, 5, 626):
                if F_ == 257:
                    x = OD.load_wav_array(_sig('tones', C_, max(256 * (T - 1), 257), T))[:, :T]
                else:
                    x = np.random.default_rng(T).standard_normal((2, T, 2 * C_)).astype(np.float32)
                for rate in (0.3, 0.7, 1.5, 3.0, 1.0001):
                    pv = _np(TR.phase_vocoder(x, rate))
                    mag = np.hypot(pv[..., :C_].astype(np.float64), pv[..., C_:])
                    check('phase_vocoder F=%d C=%d T=%d rate=%g' % (F_, C_, T, rate), mag,
                          *F.vocoder_magnitude(x, rate), fails=fails)
    x = np.random.default_rng(1).standard_normal((2, 5461, 2)).astype(np.float32)
    pv = _np(TR.phase_vocoder(x, 1.0001))
    assert pv.shape == (2, 5461, 2)
    check('phase_vocoder T_out=5461 (limit)', np.hypot(pv[..., :1].astype(np.float64), pv[..., 1:]),
          *F.vocoder_magnitude(x, 1.0001), fails=fails)
    with pytest.raises(NotImplementedError):
        TR.phase_vocoder(np.zeros((2, 5462, 2), np.float32), 1.0001)
    assert not fails, fails


# ---- bit-exact maps and label ops ----
def test_bit_exact_ops(engine, mods):
    """mask, stft_filter, random_shift, stereo_mono, mono_chan, random_merge_aug (number 2 .. 8 over several
    samples), to_frame_labels, label_downsample / er smoothing (r not dividing T, r > T, T = 1), preprocess_labels
    (odd and even T), to_density_labels (V = 1, V = 64; V = 65 refused)."""
    import torch
    from challenge_b200 import _lib as L, _ops as O
    from oracle import data_utils as OD, transforms as OT
    TR, D, _, TRN = mods
    rng = np.random.default_rng(11)
    fails = []
    spec = F.span_values(rng, (257, 33, 4))
    dr = np.array([[5, 3], [0, 7], [10, 20]], np.int32)
    check_exact('mask axis -2', _np(TR.mask(spec, axis=-2, max_mask_size=24, n_mask=3, draws=dr)),
                OT.mask(spec, axis=-2, max_mask_size=24, n_mask=3, draws=dr), fails)
    check_exact('stft_filter 16', _np(D.stft_filter(16)(spec)), OD.stft_filter(16)(spec), fails)
    check_exact('random_shift axis 0', _np(TR.random_shift(spec, axis=0, width=16, offset=5)),
                OT.random_shift(spec, axis=0, width=16, offset=5), fails)
    check_exact('stereo_mono', _np(D.stereo_mono(spec)), F.chan_map_f32(spec, 'stereo_mono'), fails)
    check_exact('mono_chan', _np(D.mono_chan(spec, 'y')[0]), F.chan_map_f32(spec, 'mono_chan'), fails)
    S, rows = 5, 257 * 33
    xs = F.span_values(rng, (S, 257, 33, 4))
    t = O.dev(xs)
    for number in range(2, 9):
        f = (np.float32(0.1) + rng.random((S, number - 2), dtype=np.float32) * np.float32(0.8))
        out = O.empty((S, 257, 33, 2 * number))
        fp = f.ctypes.data_as(C.c_void_p) if number > 2 else None
        O.call('iris_op_chan_map', L.MAP_MERGE_AUG, O.ptr(t), O.ptr(out), S * rows, 4, 2 * number, fp, S, rows)
        ref = np.stack([F.chan_map_f32(xs[s], 'merge_aug', f[s]) for s in range(S)])
        check_exact('random_merge_aug number=%d over %d samples' % (number, S), _np(out), ref, fails)
    y = rng.random((3, 7, 40, 3)).astype(np.float32)
    check_exact('to_frame_labels', _np(D.to_frame_labels(None, y)[1]), F.sum_voices_f32(y), fails)
    for T, r in ((100, 7), (31, 32), (1, 4), (626, 32), (5, 31)):
        yb = (rng.random((40, T, 3)) < 0.5).astype(np.float32)
        check_exact('label_downsample T=%d r=%d' % (T, r), _np(D.label_downsample(r)(None, yb)[1]),
                    F.avg_pool_time_f32(yb, r, True)[:r], fails)
        yf = rng.random((6, T, 3)).astype(np.float32)
        tf, out = O.dev(yf), O.empty((6, -(-T // r), 3))
        O.call('iris_op_avg_pool_time', O.ptr(tf), O.ptr(out), 6, T, 3, r, 0)
        check_exact('avg_pool_time (er smoothing) T=%d r=%d' % (T, r), _np(out), F.avg_pool_time_f32(yf, r, False),
                    fails)
    for T in (626, 627, 33, 1, 2):
        yp = (rng.random((4, T, 3)) * 3).astype(np.float32)
        check_exact('preprocess_labels T=%d' % T, _np(TRN.preprocess_labels(0.25)(None, yp)[1]),
                    F.preprocess_labels_f32(yp, 0.25), fails)
    for V in (1, 7, 64):
        yv = (rng.random((3, V, 50, 3)) < 0.1).astype(np.float32)
        yv[0, 0] = 0
        check_exact('to_density_labels V=%d' % V, _np(TRN.to_density_labels(None, yv)[1]), F.density_labels_f32(yv),
                    fails)
    with pytest.raises(NotImplementedError):
        TRN.to_density_labels(None, np.zeros((2, 65, 10, 3), np.float32))
    # the host 0 / 1 vector of mask / stft_filter fills 64000 of the 64 KB parameter slice at 16000 cells
    x = F.span_values(rng, (16000, 3))
    dr = np.array([[700, 15000], [0, 15999], [1, 0]], np.int32)
    check_exact('mask axis 0 of 16000 (limit)', _np(TR.mask(x, axis=0, n_mask=3, draws=dr)),
                OT.mask(x, axis=0, n_mask=3, draws=dr), fails)
    check_exact('stft_filter of 16000 bins (limit)', _np(D.stft_filter(15998)(x)), OD.stft_filter(15998)(x), fails)
    x1 = np.zeros((16001, 3), np.float32)
    with pytest.raises(NotImplementedError):
        TR.mask(x1, axis=0, n_mask=1, draws=[[1, 0]])
    with pytest.raises(NotImplementedError):
        D.stft_filter(3)(x1)
    torch.cuda.synchronize()
    assert not fails, fails


def test_get_er_event_limits(mods):
    """iris_op_get_er takes up to 2^20 predicted rows and 2^20 ground-truth rows.  At 2^20 rows of the events
    kernel's layout ([n, 4], the count on the device) the matching gives the oracle's answer; 2^20 + 1 predicted or
    ground-truth rows are refused.  (2^20 ground-truth rows are not run: the single-CTA rank sort is O(m^2).)"""
    import torch
    from oracle import evaluate as OE
    _, _, MT, _ = mods
    gt = np.array([[0, 10, 20], [1, 5, 9], [0, 30, 40]], np.int32)
    rows = torch.zeros((1 << 20, 4), dtype=torch.int32, device='cuda')
    ev = torch.tensor([[0, 12, 18, 15], [1, 6, 8, 7], [2, 30, 40, 35]], dtype=torch.int32)
    rows[:3] = ev.cuda()
    n_rows = torch.tensor([3], dtype=torch.int32, device='cuda')
    N, answer, m = (int(v) for v in MT.er_counts_events(gt, (rows, n_rows)).cpu().numpy())
    er, N_ref, answer_ref = OE.get_er(gt, ev.numpy()[:, [0, 3]])
    assert (N, answer, m) == (N_ref, answer_ref, 3) and (N - answer) / m == er
    _line('get_er 2^20 predicted rows (limit), 3 counted', 0.0, (), 0.0)
    with pytest.raises(NotImplementedError):
        MT.er_counts_events(gt, (torch.zeros(((1 << 20) + 1, 4), dtype=torch.int32, device='cuda'), n_rows))
    with pytest.raises(NotImplementedError):
        MT.get_er(np.zeros(((1 << 20) + 1, 3), np.int32), [[0, 1]])
    torch.cuda.synchronize()


# ---- the evaluation feature chain, stage by stage ----
def _chain(tag, D, TR, w, fails):
    """load_wav -> stft_filter(16) -> complex_to_magphase -> magphase_to_mel(80) -> minmax -> log_on_mel, each stage
    checked on the GPU output of the one before."""
    from challenge_b200.engine import default_mel_matrix
    from oracle import data_utils as OD
    spec = D.load_wav(w)
    check(tag + ' load_wav', _np(spec), *F.stft_value_bound(w), fails=fails)
    x = D.stft_filter(16)(spec)
    check_exact(tag + ' stft_filter', _np(x), OD.stft_filter(16)(_np(spec)), fails)
    xin = _np(x)
    mp = TR.complex_to_magphase(x)
    val, bnd, exact = F.complex_to_magphase(xin)
    val[..., :xin.shape[-1] // 2][exact] = F.magnitude_f32(xin)[exact]
    check(tag + ' complex_to_magphase', _np(mp), val, bnd, fails)
    mel = TR.magphase_to_mel(80)(mp)
    check(tag + ' magphase_to_mel', _np(mel), *F.mel_value_bound(_np(mp), default_mel_matrix(80, 257, 16000)),
          fails=fails)
    mm = D.minmax(mel)
    check_exact(tag + ' minmax (per mel row)', _np(mm), F.minmax_f32(_np(mel)), fails)
    check(tag + ' log_on_mel', _np(D.log_on_mel(mm)), *F.log_eps(_np(mm)), fails=fails)


def test_evaluation_chain(engine, mods):
    TR, D, _, _ = mods
    fails = []
    for i, kind in enumerate(F.SIGNALS):
        _chain('chain %s 3 s' % kind, D, TR, _sig(kind, 2, 48000, 100 + i), fails)
    _chain('chain brown 5 min', D, TR, _sig('brown', 2, 5 * 60 * 16000, 7), fails)
    engine.set_mel(80)
    assert not fails, fails

