#!/usr/bin/env python
"""Min-max log-mel features behind a channel remap: the fused step against the composition that ran before
the remap was fused, on one GPU, alternated within one process.

  python scripts/remap_mel_bench.py [--launches N]
B = 256, T = 626, V = 7, M = 2, 6 time masks + 1 frequency mask, stft_filter(3), the default 80-bin mel
matrix.  Variants (each launch after a 256 MiB write that flushes L2; median of N launches, CUDA events):
  (a) iris_step with stereo_mono + LOGMEL_MINMAX (metric leg on), float32 and bfloat16 features, and the
      same features on one uploaded plan (iris_features);
  (b) on that plan, the old composition: iris_features(MAGPHASE) with the remap -> iris_op_mel ->
      stand-alone min-max -> log (-> .to(bfloat16));
  (c) iris_step with random_merge_aug(4) + LOGMEL_MINMAX;
  (d) the configs[1] step (no remap) as the anchor.
k_fused time is the summed device time of the feature kernel launches (iris_profile_*), bytes are
iris_plan_bytes (sources read once + features written once).  The largest normalised difference between
(a) and (b) is taken on the same plan.  The GPU's name and power limit are printed beside the numbers."""
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
    ap.add_argument('--launches', type=int, default=50, help='timed launches per variant (alternated)')
    args = ap.parse_args()

    import torch
    from bench import CFG
    from challenge_b200 import _lib as L
    from challenge_b200 import _ops as O
    from challenge_b200 import data_utils as D
    from challenge_b200.engine import Engine, out_flag
    from challenge_b200.plan import draw_config, uniforms_per_clip
    from challenge_b200.synth import synthetic_banks

    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: nothing to measure')
    dev = torch.device('cuda', 0)
    print('# GPU: %s' % gpu_line(), flush=True)
    B, T, K = 256, 626, 3
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    eng = Engine(0)
    eng.set_mel(80)
    bgs, voices, labels, noises = synthetic_banks(CFG['seed'], 2, CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
    eng.register_bank(L.BANK_BG, bgs)
    eng.register_bank(L.BANK_VOICE, voices, labels=labels)
    eng.register_bank(L.BANK_NOISE, noises)
    y_pred = torch.rand((B, T, K), device=dev, generator=torch.Generator(dev).manual_seed(CFG['seed']))
    rng = np.random.default_rng(CFG['seed'])

    def step_variant(remap, n_out, dtype):
        cfg = draw_config(B, T, 7, 2, -20, 1.0, 0.5, 6, 24, 1, 16,
                          merge_extra=n_out - 2 if remap == L.REMAP_MERGE_AUG else 0)
        scfg = eng.step_config(cfg, L.FEAT_LOGMEL_MINMAX, stft_filter=3, chan_remap=remap, n_out_chan=n_out,
                               out_dtype=dtype)
        c = n_out if remap else 2
        st = dict(scfg=scfg, us=[rng.random((B, uniforms_per_clip(cfg))) for _ in range(4)], i=0,
                  out=torch.empty((B, 80, T, c), dtype=dtype, device=dev), frame=torch.empty((B, T, K), device=dev),
                  triples=torch.zeros((B, 3), dtype=torch.int32, device=dev),
                  counts=torch.zeros(6, dtype=torch.int64, device=dev), remap=remap, n_out=n_out, dtype=dtype)

        def run():
            st['i'] += 1
            eng.step(st['scfg'], st['us'][st['i'] % 4], out=st['out'], frame=st['frame'], y_pred=y_pred,
                     triples=st['triples'], counts=st['counts'])
            eng.counts_wait(0)
        st['run'] = run
        return st

    variants = {
        '(a) step stereo_mono fp32': step_variant(L.REMAP_STEREO_MONO, 3, torch.float32),
        '(a) step stereo_mono bf16': step_variant(L.REMAP_STEREO_MONO, 3, torch.bfloat16),
        '(c) step merge_aug(4) fp32': step_variant(L.REMAP_MERGE_AUG, 4, torch.float32),
        '(d) step configs[1] no remap fp32': step_variant(L.REMAP_NONE, 0, torch.float32),
    }

    # ---- one stereo_mono plan (the draws of a step) for the feature-only comparison (a) vs (b) ----
    sa = variants['(a) step stereo_mono fp32']
    sa['run']()
    d = eng.step_draws(sa['scfg'])
    plan_kw = dict(stft_filter=3, chan_remap=L.REMAP_STEREO_MONO, n_out_chan=3)
    mode = L.FEAT_LOGMEL_MINMAX

    def on_plan(fn):
        def run():
            eng.upload_plan(d, **plan_kw)
            eng.labels()
            fn()
        return run

    feat_out = {dt: torch.empty((B, 80, T, 3), dtype=dt, device=dev) for dt in (torch.float32, torch.bfloat16)}

    def old_chain(dtype):
        mp = eng.features(L.FEAT_MAGPHASE)
        mel = torch.empty((B, 80, T, 3), device=dev)
        L.check(eng.lib.iris_op_mel(eng._ctx, O.ptr(mp), O.ptr(mel), B, T, 3, eng._stream()))
        x = D.log_on_mel(D.minmax(mel))
        return x if dtype == torch.float32 else x.to(dtype)

    plan_variants = {
        '(a) features on the plan fp32': lambda: eng.features(mode, out=feat_out[torch.float32]),
        '(a) features on the plan bf16': lambda: eng.features(mode, out=feat_out[torch.bfloat16]),
        '(b) old composition fp32': lambda: old_chain(torch.float32),
        '(b) old composition bf16': lambda: old_chain(torch.bfloat16),
    }
    eng.upload_plan(d, **plan_kw)
    eng.labels()
    new = eng.features(mode).cpu().numpy().astype(np.float64)
    old = old_chain(torch.float32).cpu().numpy().astype(np.float64)
    new_b = eng.features(mode, dtype=torch.bfloat16).float().cpu().numpy()
    old_b = old_chain(torch.bfloat16).float().cpu().numpy()
    _, _, keep = eng.labels()
    keep = keep.cpu().numpy()
    bi, bo = eng.plan_bytes(mode, keep)
    bi_b, bo_b = eng.plan_bytes(mode | out_flag(torch.bfloat16), keep)
    bi_m, bo_m = eng.plan_bytes(L.FEAT_MAGPHASE, keep)

    timed = dict((k, v['run']) for k, v in variants.items())
    timed.update((k, on_plan(fn)) for k, fn in plan_variants.items())
    for fn in timed.values():                           # warm-up of every shape
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    eng.profile(True)
    ts = {k: [] for k in timed}
    kf = {k: [] for k in timed}
    for _ in range(args.launches):
        for k, fn in timed.items():
            if k.startswith('(a) features') or k.startswith('(b)'):
                eng.upload_plan(d, **plan_kw)           # outside the timed window
                eng.labels()
            flush.fill_(1)
            torch.cuda.synchronize()
            eng.profile_read(reset=True)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            (plan_variants[k] if k in plan_variants else fn)()
            b.record()
            torch.cuda.synchronize()
            ts[k].append(a.elapsed_time(b) * 1e3)
            ms, n = eng.profile_read(reset=True)
            kf[k].append(ms * 1e3)
    eng.profile(False)

    print('# B=%d T=%d V=7 M=2, masks + stft_filter(3), 80 mel bins; L2 flushed before every launch; '
          'median of %d launches per variant, variants alternated' % (B, T, args.launches))
    print('# step = iris_step incl. draws, plan upload, labels, metric leg; "on the plan" = features only')
    for k in timed:
        print('%-36s median %8.1f us (min %8.1f, max %8.1f)   k_fused %8.1f us'
              % (k, np.median(ts[k]), min(ts[k]), max(ts[k]), np.median(kf[k])), flush=True)
    print('# algorithmic bytes (iris_plan_bytes, this plan): LOGMEL_MINMAX in %.1f MB + out %.1f MB (fp32) / %.1f MB '
          '(bf16); the old chain also writes and reads the MAGPHASE intermediate of %.1f MB'
          % (bi / 1e6, bo / 1e6, bo_b / 1e6, bo_m / 1e6))
    for dt, (x, y) in (('fp32', (new, old)), ('bf16', (new_b, old_b))):
        nx, ny = np.exp(x), np.exp(y)
        print('# (a) vs (b) %s: max|diff| %.3g, normalised max error of exp(features) %.3g'
              % (dt, float(np.abs(x - y).max()), float(np.abs(nx - ny).max() / np.abs(ny).max())))
    print('# speed-up of the features on the plan, (b) / (a): fp32 x%.2f, bf16 x%.2f'
          % (np.median(ts['(b) old composition fp32']) / np.median(ts['(a) features on the plan fp32']),
             np.median(ts['(b) old composition bf16']) / np.median(ts['(a) features on the plan bf16'])))


if __name__ == '__main__':
    main()
