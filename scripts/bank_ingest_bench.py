#!/usr/bin/env python
"""Waveform banks from 44.1 / 48 kHz audio: one iris_bank_register_audio call per bank against the per-item
route it replaces (Engine.resample of every item, .cpu(), then a 16 kHz register_bank), on one GPU.

  python scripts/bank_ingest_bench.py [--reps N]      # registration wall time, the two routes alternated
  python scripts/bank_ingest_bench.py --profile       # k_resample device time (torch.profiler, own process)

Workload: the synthetic_banks sizes of bench.py (64 backgrounds of 10 s, 256 voices and 64 noises of 0.5-4 s,
2 channels, seed 20202) generated at 44.1 and 48 kHz.  Registration wall time is a host clock around the
registration of the three banks, ending in a device synchronise, median of N per route.  Kernel time is the
sum of the k_resample launches of the three banks in one registration.  Its algorithmic bytes are the float32
samples read (at the item rates) and written (at 16 kHz); its FMAs are one per tap, output sample and channel.
The share of peak is the larger of bytes / 7.7 TB/s and FMAs / (75 TFLOP/s / 2) (HGX B200 data sheet, one
GPU: HBM3e bandwidth and dense FP32) over the kernel time, with the bound named.  The GPU's name and power
limit are printed beside the numbers."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HBM_BPS = 7.7e12
FP32_FMA_PS = 75e12 / 2


def gpu_line():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            os.environ.get('CUDA_VISIBLE_DEVICES', '0').split(',')[0]],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pass
    import torch
    return torch.cuda.get_device_name(0) + ', power limit unknown'


def kaldi_taps(orig, new=16000):
    """W of iris_resample's filter bank (taps per output sample), in its float32 arithmetic."""
    g = np.gcd(orig, new)
    f32 = np.float32
    cutoff = 0.99 * 0.5 * min(orig, new)
    width = f32(6.0 / (2.0 * cutoff))
    t = np.arange(new // g, dtype=np.float32) / f32(new)
    lo = np.ceil((t - width) * f32(orig))
    hi = np.floor((t + width) * f32(orig))
    return int((hi - lo + f32(1)).max())


def banks_at(rate):
    from bench import CFG
    from challenge_b200.synth import synthetic_banks
    return synthetic_banks(CFG['seed'], CFG['n_chan'], CFG['n_bg'], CFG['n_voice'], CFG['n_noise'], sr=rate)


def register_audio(eng, banks, rate):
    from challenge_b200 import _lib as L
    bgs, voices, labels, noises = banks
    return [eng.register_bank(L.BANK_BG, [(w, rate) for w in bgs]),
            eng.register_bank(L.BANK_VOICE, [(w, rate) for w in voices], labels=labels),
            eng.register_bank(L.BANK_NOISE, [(w, rate) for w in noises])]


def register_per_item(eng, banks, rate):
    from challenge_b200 import _lib as L
    bgs, voices, labels, noises = banks

    def res(xs):
        return [eng.resample(w, rate).cpu().numpy() for w in xs]
    return [eng.register_bank(L.BANK_BG, res(bgs)),
            eng.register_bank(L.BANK_VOICE, res(voices), labels=labels),
            eng.register_bank(L.BANK_NOISE, res(noises))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5, help='registrations per route (alternated)')
    ap.add_argument('--profile', action='store_true', help='only the k_resample device time (torch.profiler)')
    args = ap.parse_args()

    import torch
    from challenge_b200.engine import Engine

    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: nothing to measure')
    print('# GPU: %s' % gpu_line(), flush=True)
    eng = Engine(0)
    for rate in (44100, 48000):
        banks = banks_at(rate)
        items = banks[0] + banks[1] + banks[3]
        n_in = sum(w.shape[1] for w in items)
        n_out = sum(int(eng.lib.iris_resample_len(w.shape[1], rate, 16000)) for w in items)
        C = items[0].shape[0]
        W = kaldi_taps(rate)
        b_in, b_out, fma = 4 * C * n_in, 4 * C * n_out, C * n_out * W
        print('# %d Hz: %d items, %.1f s of audio, %d channels; %.1f MB in, %.1f MB out, %d taps (%.3g G FMA)'
              % (rate, len(items), n_in / rate, C, b_in / 1e6, b_out / 1e6, W, fma / 1e9), flush=True)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            for route, fn in (('audio call', register_audio), ('per item', register_per_item)):
                fn(eng, banks, rate)
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    fn(eng, banks, rate)
                    torch.cuda.synchronize()
                ks = [e for e in prof.events() if e.device_type.name == 'CUDA' and 'k_resample' in e.name]
                us = sum(e.time_range.elapsed_us() for e in ks)
                t_bytes, t_fma = (b_in + b_out) / HBM_BPS * 1e6, fma / FP32_FMA_PS * 1e6
                bound = 'HBM bytes' if t_bytes >= t_fma else 'FP32 FMA'
                print('%-10s k_resample: %4d launches, %9.1f us  (%.2f TB/s, %.1f TFLOP/s; %.1f %% of the %s bound, '
                      '%.1f us)' % (route, len(ks), us, (b_in + b_out) / us / 1e6, 2 * fma / us / 1e6,
                                    100 * max(t_bytes, t_fma) / us, bound, max(t_bytes, t_fma)), flush=True)
            continue
        t = {'audio call': [], 'per item': []}
        ref = register_audio(eng, banks, rate)             # warm-up of both routes
        got = register_per_item(eng, banks, rate)
        assert all(a.tolist() == b.tolist() for a, b in zip(ref, got)), 'frame counts differ'
        for _ in range(args.reps):
            for route, fn in (('audio call', register_audio), ('per item', register_per_item)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(eng, banks, rate)
                torch.cuda.synchronize()
                t[route].append(time.perf_counter() - t0)
        for route, v in t.items():
            print('%-10s registration of the 3 banks: median %8.1f ms (min %8.1f, max %8.1f) over %d'
                  % (route, 1e3 * np.median(v), 1e3 * min(v), 1e3 * max(v), len(v)), flush=True)
        print('# per item / audio call: x%.1f' % (np.median(t['per item']) / np.median(t['audio call'])), flush=True)
    eng.close()


if __name__ == '__main__':
    main()
