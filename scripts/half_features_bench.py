#!/usr/bin/env python
"""float32 vs bfloat16 vs float16 features on one GPU, alternated within one process.

  python scripts/half_features_bench.py [--reps R] [--steps N] [--e2e-steps N]
      1. device time (CUDA events, L2 flushed by a 256 MiB write before every timed launch) and algorithmic
         bytes (iris_plan_bytes(mode | flag)) of
           - the configs[1] step: iris_step, min-max log-mel, B = 256, T = 626, 2 channels, with the metric leg;
           - 2-channel COMPLEX and 4-channel (cfg3 shape) COMPLEX / MAGPHASE features, B = 256, T = 626;
      2. end-to-end clips/s of bench.py's e2e loop (IrisDataset chain, features + labels + counts to pinned
         host memory, two buffers and a copy stream) with and without cast_features(torch.bfloat16), and
         the device -> pinned host ceiling of each feature width (the staging is torch's pin_memory, typed
         like the features, instead of bench.py's NUMA-local float32 iris_host_alloc buffers);
  python scripts/half_features_bench.py --profile
      3. the kernel list of one bf16 configs[1] step from torch.profiler (run it as its own process: tracing
         slows the host).
The GPU's name and power limit are printed beside the numbers."""
import argparse
import os
import subprocess
import sys
import time

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
    ap.add_argument('--reps', type=int, default=5, help='alternation rounds of the device timings')
    ap.add_argument('--steps', type=int, default=10, help='timed launches per dtype and round')
    ap.add_argument('--e2e-steps', type=int, default=30, help='e2e batches per arm and round')
    ap.add_argument('--e2e-rounds', type=int, default=3)
    ap.add_argument('--profile', action='store_true', help='only the torch.profiler kernel list of a bf16 step')
    args = ap.parse_args()

    import torch
    from bench import CFG, drop_in_dataset
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D
    from challenge_b200 import _ops as O
    from challenge_b200.engine import Engine, out_flag
    from challenge_b200.plan import draw_batch, draw_config, uniforms_per_clip
    from challenge_b200.synth import synthetic_banks

    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: nothing to measure')
    dev = torch.device('cuda', 0)
    print('# GPU: %s' % gpu_line(), flush=True)
    dtypes = [torch.float32, torch.bfloat16, torch.float16]
    B, T, K = CFG['batch'], CFG['n_frame'], 3
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rng = np.random.default_rng(CFG['seed'])

    # ---- the configs[1] step (iris_step with its metric leg), as bench.py times it ----
    banks2 = synthetic_banks(CFG['seed'], 2, CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
    O.set_seed(CFG['seed'] + 100)
    ds = drop_in_dataset(banks2, B)
    eng = ds.engine
    ds._prepare()                                         # sets the mel matrix of the chain
    cfg = draw_config(B, T, CFG['max_voices'], CFG['max_noises'], CFG['snr'], CFG['min_ratio'], 0.5,
                      CFG['n_time_masks'], 24, CFG['n_freq_masks'], 16)
    n_u = uniforms_per_clip(cfg)
    y_pred = torch.rand((B, T, K), device=dev, generator=torch.Generator(dev).manual_seed(CFG['seed']))
    steps = {}
    for dt in dtypes:
        steps[dt] = dict(scfg=eng.step_config(cfg, L.FEAT_LOGMEL_MINMAX, out_dtype=dt),
                         out=torch.empty((B, CFG['n_mels'], T, 2), dtype=dt, device=dev),
                         frame=torch.empty((B, T, K), device=dev), triples=torch.zeros((B, 3), dtype=torch.int32, device=dev),
                         counts=torch.zeros(6, dtype=torch.int64, device=dev))

    def run_step(dt, u):
        s = steps[dt]
        eng.step(s['scfg'], u, out=s['out'], frame=s['frame'], y_pred=y_pred, triples=s['triples'], counts=s['counts'])
        eng.counts_wait(0)

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        u = rng.random((B, n_u))
        for _ in range(3):
            run_step(torch.bfloat16, u)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_step(torch.bfloat16, u)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type.name == 'CUDA']
        kernels = [n for n in names if n.startswith(('iris::', 'void iris::')) or 'k_' in n]
        print('# kernels of one bf16 configs[1] step (torch.profiler, CUDA activity, launch order):')
        for n in kernels:
            print('  ' + n)
        print('# k_tiles launched: %s' % any('k_tiles' in n for n in kernels))
        return

    def timed(fn, dt):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(dt)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3

    def alternate(label, fn, alg_bytes):
        for dt in dtypes:                                 # warm-up of every shape
            for _ in range(3):
                fn(dt)
        torch.cuda.synchronize()
        ts = {dt: [] for dt in dtypes}
        for _ in range(args.reps):
            for dt in dtypes:
                ts[dt] += [timed(fn, dt) for _ in range(args.steps)]
        base = np.median(ts[torch.float32])
        for dt in dtypes:
            med = float(np.median(ts[dt]))
            print('%-44s %-8s median %8.1f us  (min %8.1f, max %8.1f, n %d)  alg %7.1f MB  %5.2f TB/s  x%.3f of fp32'
                  % (label, str(dt).replace('torch.', ''), med, min(ts[dt]), max(ts[dt]), len(ts[dt]),
                     alg_bytes[dt] / 1e6, alg_bytes[dt] / med / 1e6, base / med), flush=True)

    us = [rng.random((B, n_u)) for _ in range(8)]
    k = {'i': 0}

    def step_fn(dt):
        k['i'] += 1
        run_step(dt, us[k['i'] % len(us)])

    alg = {}
    for dt in dtypes:                                      # bytes of the last plan with its keep flags
        run_step(dt, us[0])
        _, _, keep = eng.labels()
        bi, bo = eng.plan_bytes(L.FEAT_LOGMEL_MINMAX | out_flag(dt), keep.cpu().numpy())
        alg[dt] = bi + bo
    print('# 1. device time, alternated fp32 / bf16 / fp16, %d rounds x %d launches each' % (args.reps, args.steps))
    alternate('configs[1] step (min-max log-mel, B=256, 2-ch)', step_fn, alg)

    # ---- spectrogram modes: features() on one uploaded plan (mix + masks, B = 256, T = 626) ----
    for n_chan, modes in ((2, (L.FEAT_COMPLEX,)), (4, (L.FEAT_COMPLEX, L.FEAT_MAGPHASE))):
        e = eng if n_chan == 2 else Engine(0)
        if n_chan == 4:
            bgs, voices, labels, noises = synthetic_banks(CFG['seed'], 4, CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
            bf = e.register_bank(L.BANK_BG, bgs)
            vf = e.register_bank(L.BANK_VOICE, voices, labels=labels)
            nf = e.register_bank(L.BANK_NOISE, noises)
        else:
            bf, vf, nf = (e.bank_frames[k_] for k_ in (L.BANK_BG, L.BANK_VOICE, L.BANK_NOISE))
        d = draw_batch(np.random.default_rng(1), B, T, bf, vf, nf, max_voices=7, max_noises=2, snr=-20, min_ratio=1,
                       n_time_masks=6, n_freq_masks=1)
        e.upload_plan(d)
        _, _, keep = e.labels()
        keep = keep.cpu().numpy()
        for mode in modes:
            outs = {dt: torch.empty((B, 257, T, 2 * n_chan), dtype=dt, device=dev) for dt in dtypes}
            alg = {}
            for dt in dtypes:
                bi, bo = e.plan_bytes(mode | out_flag(dt), keep)
                alg[dt] = bi + bo
            name = {L.FEAT_COMPLEX: 'COMPLEX', L.FEAT_MAGPHASE: 'MAGPHASE'}[mode]
            alternate('%d-ch %s features (B=256, mix + masks)' % (n_chan, name),
                      lambda dt, e=e, mode=mode, outs=outs: e.features(mode, out=outs[dt]), alg)
        if n_chan == 4:
            e.close()
            del e
            torch.cuda.empty_cache()

    # ---- 2. end to end: bench.py's e2e loop, with and without cast_features(torch.bfloat16) ----
    dss = {torch.float32: ds, torch.bfloat16: drop_in_dataset(banks2, B).map(D.cast_features(torch.bfloat16))}
    assert dss[torch.bfloat16]._lower()[0]['out_flag'] == L.OUT_BF16
    its = {dt: iter(d_) for dt, d_ in dss.items()}
    copy_stream = torch.cuda.Stream(device=dev)
    e_counts = torch.zeros(6, dtype=torch.int64, device=dev)
    host = {dt: dict(feat=[torch.empty((B, CFG['n_mels'], T, 2), dtype=dt, pin_memory=True) for _ in range(2)],
                     lbl=[torch.empty((B, T, K), pin_memory=True) for _ in range(2)],
                     cnt=[torch.empty(6, dtype=torch.int64, pin_memory=True) for _ in range(2)],
                     copied=[torch.cuda.Event() for _ in range(2)]) for dt in dss}

    def e2e_step(dt, i):
        h = host[dt]
        j = i & 1
        x, y = next(its[dt])
        assert x.dtype == dt
        dss[dt].engine.metric_counts(y, y_pred, counts=e_counts, want_er=False)
        done = torch.cuda.Event()
        done.record()
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done)
            h['feat'][j].copy_(x, non_blocking=True)
            h['lbl'][j].copy_(y, non_blocking=True)
            h['cnt'][j].copy_(e_counts, non_blocking=True)
            h['copied'][j].record()
            x.record_stream(copy_stream)
            y.record_stream(copy_stream)
        h['copied'][j ^ 1].synchronize()
        return x

    def e2e_run(dt, n):
        for i in range(3):
            e2e_step(dt, i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(n):
            x = e2e_step(dt, 3 + i)
        torch.cuda.synchronize()
        return B * n / (time.perf_counter() - t0), x

    rates = {dt: [] for dt in dss}
    last = {}
    for _ in range(args.e2e_rounds):
        for dt in dss:
            r, last[dt] = e2e_run(dt, args.e2e_steps)
            rates[dt].append(r)
    print('# 2. end to end (bench.py e2e loop: IrisDataset chain, features + labels + counts to pinned host memory, '
          'two buffers + copy stream), %d rounds x %d batches per arm, alternated' % (args.e2e_rounds, args.e2e_steps))
    for dt in dss:
        h = host[dt]
        d2h = h['feat'][0].numel() * h['feat'][0].element_size() + h['lbl'][0].numel() * 4 + 6 * 8
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(8):
            h['feat'][i & 1].copy_(last[dt], non_blocking=True)
        torch.cuda.synchronize()
        ceil = 8 * h['feat'][0].numel() * h['feat'][0].element_size() / (time.perf_counter() - t0) / 1e9
        med = float(np.median(rates[dt]))
        print('e2e %-8s median %9.0f clips/s (rounds: %s)  d2h %.1f MB/batch = %.1f GB/s; feature D2H ceiling %.1f GB/s'
              % (str(dt).replace('torch.', ''), med, ', '.join('%.0f' % r for r in rates[dt]), d2h / 1e6,
                 d2h * med / B / 1e9, ceil), flush=True)
    print('e2e bf16 / fp32: x%.3f' % (np.median(rates[torch.bfloat16]) / np.median(rates[torch.float32])))


if __name__ == '__main__':
    main()
