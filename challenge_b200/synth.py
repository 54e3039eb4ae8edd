"""Synthetic waveform banks of the benchmark workloads (SURVEY.md 8d / BASELINE.md 3)."""
import numpy as np


def synthetic_banks(seed, n_chan, n_bg=64, n_voice=256, n_noise=64, sr=16000, bg_seconds=10.0,
                    lo_s=0.5, hi_s=4.0, n_classes=3):
    """The synthetic banks of SURVEY.md 8(d): N(0,1)*0.1 waveforms; voices get a trailing
    0-25 % of exact zeros (exercises the ``> 0`` activity mask like pipeline_test.py:21-24)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    f32 = np.float32
    bgs = [(rng.standard_normal((n_chan, int(bg_seconds * sr)), dtype=f32) * f32(0.1))
           for _ in range(n_bg)]
    voices, labels = [], []
    for _ in range(n_voice):
        n = int(rng.integers(int(lo_s * sr), int(hi_s * sr) + 1))
        w = rng.standard_normal((n_chan, n), dtype=f32) * f32(0.1)
        z = int(n * rng.uniform(0, 0.25))
        if z:
            w[:, n - z:] = 0
        voices.append(w)
        labels.append(int(rng.integers(n_classes)))
    labels = np.eye(n_classes, dtype=f32)[labels]
    noises = []
    for _ in range(n_noise):
        n = int(rng.integers(int(lo_s * sr), int(hi_s * sr) + 1))
        noises.append(rng.standard_normal((n_chan, n), dtype=f32) * f32(0.1))
    return bgs, voices, labels, noises


STRUCTURED_KINDS = ('white', 'pink', 'brown', 'tones', 'chirp', 'clicks', 'quiet', 'zeros', 'pair80')


def structured_source(rng, kind, n_chan, n, sr=16000):
    """One float32 source ``[n_chan, n]`` of a signal with dynamic range inside it, at RMS 0.1 over all
    its channels.  Kinds (STRUCTURED_KINDS):

    white   N(0, 1) noise, the flat-spectrum baseline
    pink    1/f noise, brown 1/f^2 noise: more than 60 dB from bin 1 to Nyquist
    tones   a DC offset, bins 1 and 255, tones at bin centres and half-bin offsets and an alternating-sign
            Nyquist tone, at levels 0 .. -60 dB
    chirp   linear sweep 0 Hz -> sr / 2 over the source: every bin and every mel band dominates once
    clicks  a few unit impulses on silence-level noise (-80 dB)
    quiet   brown noise with a section at -60 dB
    zeros   pink noise with exact-zero sections away from the tail
    pair80  brown noise on the even channels, the odd channels 80 dB below (a packed FFT pair
            whose quiet member shares the loud member's transform)
    """
    t = np.arange(n, dtype=np.float64)

    def colored(alpha):
        spec = np.fft.rfft(rng.standard_normal((n_chan, n)), axis=-1)
        f = np.arange(spec.shape[-1], dtype=np.float64)
        f[0] = np.inf                                   # no DC
        return np.fft.irfft(spec * f ** (-alpha / 2), n, axis=-1)

    if kind == 'white':
        x = rng.standard_normal((n_chan, n))
    elif kind == 'pink':
        x = colored(1.0)
    elif kind in ('brown', 'quiet', 'pair80'):
        x = colored(2.0)
        if kind == 'quiet':
            lo = int(rng.integers(n // 5, n // 2))
            x[:, lo:lo + max(n // 4, 1)] *= 1e-3
        elif kind == 'pair80':
            x[1::2] *= 1e-4
    elif kind == 'zeros':
        x = colored(1.0)
        for lo in (int(rng.integers(0, n // 3)), int(rng.integers(n // 3, 2 * n // 3))):
            x[:, lo:lo + max(n // 8, 1)] = 0.0
    elif kind == 'tones':
        bin_hz = sr / 512.0
        x = np.full((n_chan, n), 0.05)                  # DC offset
        x += np.cos(2 * np.pi * bin_hz * t / sr)        # bin 1
        x += 1e-3 * np.cos(2 * np.pi * 255 * bin_hz * t / sr + 0.3)
        x += 1e-2 * (-1.0) ** t                         # Nyquist, alternating sign
        for k, level in ((17, 0.3), (40.5, 0.1), (96, 1e-2), (128.5, 1e-3), (200, 3e-2)):
            x += level * np.sin(2 * np.pi * k * bin_hz * t / sr + rng.uniform(0, 2 * np.pi, (n_chan, 1)))
    elif kind == 'chirp':
        x = np.cos(np.pi * (sr / 2) / n * t * t / sr + rng.uniform(0, 2 * np.pi, (n_chan, 1)))
    elif kind == 'clicks':
        x = 1e-4 * rng.standard_normal((n_chan, n))
        for pos in rng.integers(0, n, size=(n_chan, 6)).T:
            x[np.arange(n_chan), pos] = 1.0
    else:
        raise ValueError('unknown kind %r' % kind)
    x *= 0.1 / np.sqrt(np.mean(x * x))
    return x.astype(np.float32)


def structured_banks(seed, n_chan, n_bg=4, n_voice=12, n_noise=4, sr=16000, bg_seconds=2.0, lo_s=0.3,
                     hi_s=1.5, n_classes=3):
    """Banks of :func:`structured_source` signals, laid out like :func:`synthetic_banks`' return:
    ``(bgs, voices, labels, noises)``.  The kinds are cycled in a seeded order over the backgrounds, then the
    voices, then the noises, so a bank of at least len(STRUCTURED_KINDS) items (the voices by default) holds every
    kind and a smaller one as many different kinds as it has items."""
    rng = np.random.Generator(np.random.PCG64(seed))
    order = list(rng.permutation(len(STRUCTURED_KINDS)))

    def kinds():
        i = 0
        while True:
            yield STRUCTURED_KINDS[order[i % len(order)]]
            i += 1
    k = kinds()
    bgs = [structured_source(rng, next(k), n_chan, int(bg_seconds * sr), sr) for _ in range(n_bg)]
    voices = [structured_source(rng, next(k), n_chan, int(rng.integers(int(lo_s * sr), int(hi_s * sr) + 1)), sr)
              for _ in range(n_voice)]
    labels = np.eye(n_classes, dtype=np.float32)[rng.integers(n_classes, size=n_voice)]
    noises = [structured_source(rng, next(k), n_chan, int(rng.integers(int(lo_s * sr), int(hi_s * sr) + 1)), sr)
              for _ in range(n_noise)]
    return bgs, voices, labels, noises
