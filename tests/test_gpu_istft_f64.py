"""The inverse STFT (k_istft: iris_istft, Engine.istft, data_utils.to_waveform) against the float64 value and
per-sample bound of oracle/f64_ops.py istft_value_bound: KAPPA_ISTFT u times the covering frames' weights times
their channel pair's norm over sqrt(512), so that a quiet item, pair or channel is held to its own frames rather
than to the loudest thing in the call.  Spectra: the float64 STFT of every F.SIGNALS kind, an item 80 dB down in a
loud batch, a quiet pair beside a loud one, a quiet channel inside a loud pair, all-zero frames inside a clip and
bins around 1e-40.  Shapes: every channel count path (kC = 2, 1 and the scalar loads, odd C), T at the 7-hop tile
edges, lengths one sample either side of 256 (T - 1) and 256 T, B up to its limit of 65535 and a length of
2^31 - 1 samples.  Also the load_wav round trips, bfloat16 / float16 input and non-finite bins.  Where no frame
covers a sample (s >= 256 T) the output must be exactly +0.  Per configuration one line: the largest ratio
error / bound, where it occurs, and the normalised max error beside it (profiles/r12_istft_f64.txt)."""
import numpy as np
import pytest

from conftest import nmax_err
from oracle import f64, f64_ops as F

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().float().cpu().numpy()


@pytest.fixture(scope='module')
def D(engine):
    from challenge_b200 import data_utils, engine as E
    E._engines[0] = engine          # share the session engine
    import torch
    print('\n# %s' % torch.cuda.get_device_name(0))
    try:
        import subprocess
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            '0'], capture_output=True, text=True, timeout=30)
        print('# nvidia-smi: %s' % q.stdout.strip())
    except (OSError, subprocess.SubprocessError) as e:
        print('# nvidia-smi not available: %s' % e)
    return data_utils


def _line(tag, r, at, nm):
    print('%-72s ratio %9.3g at %-20s nmax %.2e' % (tag, r, str(at), nm))


def check(tag, got, val, bnd, T, fails):
    """One configuration: every sample within its bound, samples from 256 T on exactly +0."""
    got = np.asarray(got)
    assert got.shape == val.shape, (tag, got.shape, val.shape)
    r, at = f64.worst(F.ratio(got, val, bnd))
    z = got[..., 256 * T:]
    if z.size and (np.any(z != 0) or np.signbit(z).any()):
        fails.append((tag, 'not +0 from 256 T on'))
    nm = nmax_err(got, val) if got.size and np.abs(val).max() > 0 else 0.0
    _line(tag, r, at, nm)
    if not r <= 1:
        fails.append((tag, r, at))
    return r


def run(engine, tag, spec, lengths, fails):
    """Engine.istft of ``spec`` at every length, checked against one reference at the longest (the samples of a
    shorter length are a prefix of a longer one's)."""
    T = spec.shape[-2]
    Lmax = max(256 * (T - 1) if n is None else n for n in lengths)
    val, bnd = F.istft_value_bound(spec, Lmax)
    for n in lengths:
        L = 256 * (T - 1) if n is None else n
        got = _np(engine.istft(spec, n))
        check('%s L=%s' % (tag, n if n is not None else 'default %d' % L), got, val[..., :L], bnd[..., :L], T, fails)


def _sig(kind, C, n, seed):
    return F.signal(np.random.default_rng(seed), kind, C, n)


def test_signals(engine, D):
    """The float64 STFT (rounded to float32) of every F.SIGNALS kind at C = 1 .. 5, two items a batch with the
    second one 40 dB down, the default length and n."""
    fails = []
    for i, kind in enumerate(F.SIGNALS):
        C = 1 + i % 5
        n = 256 * 60 + 3 * i
        spec = np.stack([f64.spec_f64(_sig(kind, C, n, i)), 1e-2 * f64.spec_f64(_sig(kind, C, n, 50 + i))])
        run(engine, 'signal %s C=%d n=%d' % (kind, C, n), spec.astype(np.float32), [None, n], fails)
    assert not fails, fails


def test_quiet_structures(engine, D):
    """An item 80 dB down in a loud batch; a quiet pair beside a loud one (C = 4); a quiet channel inside a loud pair;
    all-zero frames inside a clip (both channels of a pair, and of one channel only); bins around 1e-40 (subnormal
    samples)."""
    fails = []
    n = 256 * 50 + 100
    loud = [f64.spec_f64(_sig(k, 4, n, 7 + j)) for j, k in enumerate(('pink', 'tones', 'chirp'))]
    b = np.stack(loud + [1e-4 * f64.spec_f64(_sig('white', 4, n, 3))]).astype(np.float32)
    run(engine, 'item 3 at -80 dB in a loud batch B=4 C=4', b, [None, n], fails)
    p = loud[0].copy()
    p[..., [2, 3, 6, 7]] *= 1e-4
    run(engine, 'pair 1 at -80 dB beside a loud pair C=4', p.astype(np.float32)[None], [n], fails)
    q = f64.spec_f64(_sig('pink', 2, n, 4)).astype(np.float32)
    q[..., [1, 3]] *= np.float32(1e-4)
    run(engine, 'channel 1 at -80 dB inside a loud pair C=2', q, [n], fails)
    zf = f64.spec_f64(_sig('brown', 3, n, 5)).astype(np.float32)
    zf[:, 13:21] = 0                             # all channels, frames 13 .. 20 (across a tile edge)
    zf[:, 30:32, [2, 5]] = 0                     # channel 2 (alone in pair 1), frames 30, 31
    zf[:, 40, [0, 3]] = 0                        # channel 0 of pair 0 only: pair 0's norm stays > 0
    run(engine, 'all-zero frames inside a clip C=3', zf, [None, n], fails)
    x = np.random.default_rng(6).standard_normal((3, 257, 20, 6))
    x *= 1e-40
    x[1] *= 1e-3
    x[2, :, :, [0, 3]] *= 1e38                   # a normal channel beside a subnormal one
    run(engine, 'bins around 1e-40 and 1e-43 B=3 C=3', x.astype(np.float32), [None, 256 * 20 + 30], fails)
    assert not fails, fails


CS = (1, 2, 3, 4, 5, 7, 31, 32)
TS = (1, 2, 6, 7, 8, 9, 14, 15, 626)
BS = (1, 3, 17)


def _lengths(T):
    c = [1, 255, 256, 257, 256 * (T - 1) - 1, 256 * (T - 1), 256 * (T - 1) + 1, 256 * T - 1, 256 * T, 256 * T + 1,
         256 * T + 700]
    return sorted({n for n in c if n >= 1}) + ([None] if T > 1 else [])


def test_shapes(engine, D):
    """Every C x T, with B cycling through 1, 3, 17 (B = 1 where T = 626 and C > 4), random spectra whose items and
    channel pairs span 0 .. -100 dB, at every length of _lengths(T)."""
    fails = []
    k = 0
    for C in CS:
        for T in TS:
            B = 1 if T == 626 and C > 4 else BS[k % 3]
            k += 1
            rng = np.random.default_rng(1000 * C + T)
            x = rng.standard_normal((B, 257, T, 2 * C))
            x *= 10.0 ** (-rng.integers(0, 6, size=(B, 1, 1, 1)))                 # per item
            pair_db = 10.0 ** (-rng.integers(0, 6, size=(B, 1, 1, (C + 1) // 2)))
            x *= np.concatenate([np.repeat(pair_db, 2, -1)[..., :C]] * 2, -1)     # per pair
            run(engine, 'C=%d T=%d B=%d' % (C, T, B), x.astype(np.float32), _lengths(T), fails)
    assert not fails, fails


def test_batch_limit(engine, D):
    """B = 65535 (the grid's z limit), T = 2, C = 3, L = 256 T + 1; checked in blocks of items."""
    import torch
    B, T, C, L = 65535, 2, 3, 513
    x = np.random.default_rng(8).standard_normal((B, 257, T, 2 * C)).astype(np.float32)
    x *= (10.0 ** -(np.arange(B) % 7)).astype(np.float32)[:, None, None, None]
    got = engine.istft(x, L)
    fails, worst = [], (0.0, None)
    for b0 in range(0, B, 8192):
        b1 = min(b0 + 8192, B)
        val, bnd = F.istft_value_bound(x[b0:b1], L)
        g = _np(got[b0:b1])
        r, at = f64.worst(F.ratio(g, val, bnd))
        if r > worst[0]:
            worst = (r, (at[0] + b0,) + at[1:])
        if np.any(g[..., 256 * T:] != 0) or np.signbit(g[..., 256 * T:]).any():
            fails.append(('not +0 from 256 T on', b0))
    _line('B=65535 T=2 C=3 L=513 (limit)', worst[0], worst[1], float('nan'))
    del got
    torch.cuda.empty_cache()
    assert worst[0] <= 1 and not fails, (worst, fails)


def test_length_limit(engine, D):
    """L = 2^31 - 1 with B = 2, C = 2, T = 5: output offsets past 2^32 floats (34 GB).  The covered samples against
    the bound; everything from 256 T on +0, checked on the device in chunks."""
    import torch
    B, T, C, L = 2, 5, 2, 2 ** 31 - 1
    if torch.cuda.mem_get_info()[0] < (B * C * L * 4 + (2 << 30)):
        pytest.skip('needs 36 GB of free device memory')
    x = np.random.default_rng(9).standard_normal((B, 257, T, 2 * C)).astype(np.float32)
    x[1] *= np.float32(1e-5)
    got = engine.istft(x, L)
    head = 256 * T + 1000
    val, bnd = F.istft_value_bound(x, head)
    fails = []
    check('B=2 C=2 T=5 L=2^31-1 (limit), first %d samples' % head, _np(got[..., :head]), val, bnd, T, fails)
    bad = 0
    step = 1 << 28
    for b in range(B):
        for c in range(C):
            row = got[b, c]
            for s0 in range(256 * T, L, step):
                bad += int(torch.count_nonzero(row[s0:min(s0 + step, L)].view(torch.int32)))
    print('L=2^31-1: %d samples from 256 T on that are not +0 (bits)' % bad)
    del got, row
    torch.cuda.empty_cache()
    assert bad == 0 and not fails, (bad, fails)


def round_trip_value_bound(w, spec):
    """to_waveform(load_wav(w), length=n) of ``w [C, n]``, given the float32 spectrum load_wav made -> (normalize(w)
    in float64, bound): the inverse's bound on ``spec``, istft_carry of load_wav's bound, and the normalisation's
    rounding, 4 u |value|."""
    n = w.shape[1]
    ref = f64.normalize_f64(w)
    _, bnd = F.istft_value_bound(spec, n)
    _, sb = F.stft_value_bound(w)
    return ref, bnd + F.istft_carry(sb, spec.shape[1], n) + 4 * F.U * np.abs(ref)


@pytest.mark.parametrize('C', [1, 2, 3])
def test_round_trips(engine, D, C):
    """to_waveform(load_wav(w)) against normalize(w) in float64, for every F.SIGNALS kind and n around the frame
    edges.  Bound: the inverse's own bound on the spectrum it was given, plus istft_carry of load_wav's bound (what
    the forward STFT's error moves the exact inverse), plus the normalisation's rounding (4 u |value|)."""
    fails = []
    ns = (257, 511, 512, 513, 256 * 40 - 1, 256 * 40, 256 * 40 + 1, 48001)
    for i, kind in enumerate(F.SIGNALS):
        for n in (ns[i % len(ns)], ns[(i + 3 + C) % len(ns)]):
            w = _sig(kind, C, n, 31 * i + n + C)
            spec = D.load_wav(w)
            T = int(spec.shape[1])
            length = None if n % 256 == 0 else n
            got = _np(D.to_waveform(spec, length=length))
            ref, bnd = round_trip_value_bound(w, _np(spec))
            check('round trip %s C=%d n=%d' % (kind, C, n), got, ref, bnd, T, fails)
    assert not fails, fails


def test_half_precision_input(engine, D):
    """to_waveform of bfloat16 / float16 COMPLEX features is to_waveform of the same features after .float(), bit for
    bit (the promotion is exact)."""
    import torch
    x = torch.as_tensor(np.random.default_rng(12).standard_normal((3, 257, 30, 4)).astype(np.float32)).cuda()
    for dt in (torch.bfloat16, torch.float16):
        h = x.to(dt)
        a, b = _np(D.to_waveform(h)), _np(D.to_waveform(h.float()))
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), dt
        val, bnd = F.istft_value_bound(_np(h.float()))
        fails = []
        check('%s input B=3 C=2 T=30' % str(dt).split('.')[-1], a, val, bnd, 30, fails)
        assert not fails, fails


@pytest.mark.parametrize('value', [np.nan, np.inf])
def test_non_finite_bin(engine, D, value):
    """A NaN or inf in one bin of channel 0 at frame 7 (the halo of tile 0, the first frame of tile 1) of item 1:
    torch.istft makes that channel's two covering hops (6 and 7) non-finite.  The kernel inverts channels 0 and 1 in
    one complex FFT, so channel 1 may turn non-finite there too; nothing else may: not other hops, pairs or items,
    and every other sample stays within its bound."""
    C, T, t = 3, 20, 7
    x = np.random.default_rng(13).standard_normal((2, 257, T, 2 * C)).astype(np.float32)
    x[1, 40, t, 0] = value
    L = 256 * T + 100
    got = _np(engine.istft(x, L))
    hops = slice(256 * (t - 1), 256 * (t + 1))
    ref = F.istft_f64(x, L)
    assert not np.isfinite(ref[1, 0, hops]).any() and np.isfinite(np.delete(ref[1], 0, 0)).all()
    fin = np.isfinite(got)
    assert not fin[1, 0, hops].any(), 'channel 0 of the bad frame must be non-finite'
    allowed = np.zeros(got.shape, bool)
    allowed[1, 0:2, hops] = True
    assert fin[~allowed].all(), 'non-finite samples outside the two hops of the pair'
    clean = x.copy()
    clean[1, 40, t, 0] = 0
    val, bnd = F.istft_value_bound(clean, L)
    ok = np.where(allowed, val, got)
    fails = []
    check('non-finite %s in item 1 ch 0 frame 7: %d of ch 1\'s 512 samples there non-finite'
          % (value, (~fin[1, 1, hops]).sum()), ok, val, bnd, T, fails)
    assert not fails, fails
