#!/usr/bin/env python
"""sj_train's n_chan = 1 chain (mono_chan -> stft_filter -> complex_to_magphase -> magphase_to_mel -> minmax ->
log_on_mel): the fused step against the un-fused composition, on one GPU, alternated within one process.

  python scripts/mono_chain_bench.py [--launches N]
Two sizes: B = 256, T = 626 (bench.py's configs[1] clips) and sj_train's B = 12, T = 512; V = 7, M = 2, 6 time
masks + 1 frequency mask, stft_filter(3), the default 80-bin mel matrix, min-max log-mel features.  Per size,
variants on the same draws (each launch after a 256 MiB write that flushes L2; median of N launches, CUDA events):
  (a) iris_step with mono_chan (metric leg on), and the same features on one uploaded plan (iris_features);
  (b) on that plan, the un-fused composition the drop-in runs when mono_chan is not absorbed: COMPLEX features,
      then per clip mono_chan and stft_filter (stand-alone ops), a stack, complex_to_magphase of the 3-column
      spectrogram, magphase_to_mel, minmax, log_on_mel;
  (c) the configs[1] step (no remap) and (d) the stereo_mono step as reference points.
k_fused time is the summed device time of the feature kernel launches (iris_profile_*).  (a) and (b) are compared
on the plan they were timed on.  The GPU's name and power limit are printed beside the numbers."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--launches', type=int, default=30, help='timed launches per variant (alternated)')
    args = ap.parse_args()

    import torch
    from bench import CFG
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.engine import Engine
    from challenge_b200.plan import draw_config, uniforms_per_clip
    from challenge_b200.synth import synthetic_banks

    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: nothing to measure')
    dev = torch.device('cuda', 0)
    print('# GPU: %s' % gpu_line(), flush=True)
    K = 3
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    eng = Engine(0)
    eng.set_mel(80)
    bgs, voices, labels, noises = synthetic_banks(CFG['seed'], 2, CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
    eng.register_bank(L.BANK_BG, bgs)
    eng.register_bank(L.BANK_VOICE, voices, labels=labels)
    eng.register_bank(L.BANK_NOISE, noises)
    mode = L.FEAT_LOGMEL_MINMAX
    mel_stages = (TR.magphase_to_mel(80), D.minmax, D.log_on_mel)

    for B, T in ((256, 626), (12, 512)):
        rng = np.random.default_rng(CFG['seed'])
        y_pred = torch.rand((B, T, K), device=dev, generator=torch.Generator(dev).manual_seed(CFG['seed']))
        cfg = draw_config(B, T, 7, 2, -20, 1.0, 0.5, 6, 24, 1, 16)
        us = [rng.random((B, uniforms_per_clip(cfg))) for _ in range(4)]   # the same draws for every step variant

        def step_variant(remap, n_out):
            scfg = eng.step_config(cfg, mode, stft_filter=3, chan_remap=remap, n_out_chan=n_out)
            st = dict(scfg=scfg, i=0, out=torch.empty((B, 80, T, n_out or 2), device=dev),
                      frame=torch.empty((B, T, K), device=dev), triples=torch.zeros((B, 3), dtype=torch.int32, device=dev),
                      counts=torch.zeros(6, dtype=torch.int64, device=dev))

            def run():
                st['i'] += 1
                eng.step(st['scfg'], us[st['i'] % 4], out=st['out'], frame=st['frame'], y_pred=y_pred,
                         triples=st['triples'], counts=st['counts'])
                eng.counts_wait(0)
            st['run'] = run
            return st

        steps = {'(a) step mono_chan': step_variant(L.REMAP_MONO_CHAN, 2),
                 '(c) step configs[1] no remap': step_variant(L.REMAP_NONE, 0),
                 '(d) step stereo_mono': step_variant(L.REMAP_STEREO_MONO, 3)}
        sa = steps['(a) step mono_chan']
        sa['run']()
        d = eng.step_draws(sa['scfg'])
        fused_kw = dict(stft_filter=3, chan_remap=L.REMAP_MONO_CHAN, n_out_chan=2)
        feat_out = torch.empty((B, 80, T, 2), device=dev)

        def fused():
            return eng.features(mode, out=feat_out)

        def unfused():
            x = eng.features(L.FEAT_COMPLEX)          # the plan's masks, no remap, no filter
            xs = [D.stft_filter(3)(*D.mono_chan(x[b], 0))[0] for b in range(B)]
            x = TR.complex_to_magphase(torch.stack(xs))
            for fn in mel_stages:
                x = fn(x)
            return x

        plans = {'(a) features on the plan': (fused, fused_kw), '(b) un-fused composition': (unfused, {})}

        def on_plan(k):
            fn, kw = plans[k]
            eng.upload_plan(d, **kw)
            eng.labels()
            return fn

        new = on_plan('(a) features on the plan')().cpu().numpy().astype(np.float64)
        old = on_plan('(b) un-fused composition')().cpu().numpy().astype(np.float64)

        timed = [k for k in steps] + list(plans)
        for k in timed:                              # warm-up of every shape
            for _ in range(3):
                (steps[k]['run'] if k in steps else on_plan(k))()
        torch.cuda.synchronize()
        eng.profile(True)
        ts = {k: [] for k in timed}
        kf = {k: [] for k in timed}
        for _ in range(args.launches):
            for k in timed:
                fn = steps[k]['run'] if k in steps else on_plan(k)   # plan upload + labels outside the window
                flush.fill_(1)
                torch.cuda.synchronize()
                eng.profile_read(reset=True)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize()
                ts[k].append(a.elapsed_time(b) * 1e3)
                ms, n = eng.profile_read(reset=True)
                kf[k].append(ms * 1e3)
        eng.profile(False)

        print('# B=%d T=%d V=7 M=2, masks + stft_filter(3), 80 mel bins, min-max log-mel fp32; L2 flushed before '
              'every launch; median of %d launches per variant, variants alternated' % (B, T, args.launches))
        print('# step = iris_step incl. draws, plan upload, labels, metric leg; "on the plan" = features only')
        for k in timed:
            print('%-32s median %9.1f us (min %9.1f, max %9.1f)   k_fused %8.1f us'
                  % (k, np.median(ts[k]), min(ts[k]), max(ts[k]), np.median(kf[k])), flush=True)
        nx, ny = np.exp(new), np.exp(old)
        print('# (a) vs (b) on the plan: max|diff| %.3g, normalised max error of exp(features) %.3g'
              % (float(np.abs(new - old).max()), float(np.abs(nx - ny).max() / np.abs(ny).max())))
        print('# speed-up of the features on the plan, (b) / (a): x%.1f; mono step / configs[1] step: %.3f'
              % (np.median(ts['(b) un-fused composition']) / np.median(ts['(a) features on the plan']),
                 np.median(ts['(a) step mono_chan']) / np.median(ts['(c) step configs[1] no remap'])), flush=True)


if __name__ == '__main__':
    main()
