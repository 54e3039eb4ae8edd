#!/usr/bin/env python
"""2-channel mel from the banks' STFT bin planes against the FFT path, two libiris builds alternated on one GPU.

  python scripts/mel_plane_bench.py --old path/to/parent/libiris.so [--new path] [--reps 3] [--launches 20]
Each repetition runs one worker process per build (IRIS_LIB), old then new.  A worker registers bench.py's
synthetic 2-channel banks (CUDA events around each registration: with the plane build it includes the k_fused
pass that writes the plane), then on configs[1]'s shape (B = 256, T = 626, V = 7, M = 2, 6 time masks + 1
frequency mask, stft_filter(3), 80 mel bins, min-max log-mel fp32) times, each launch after a 256 MiB write that
flushes L2, median of --launches:
  step      iris_step incl. draws, plan upload, labels and the metric leg (bench.py's timed step);
  features  iris_features on one uploaded plan (labels done), k_fused + k_logmel_post;
  k_fused   the feature kernel alone, from the profile hook (iris_profile_*), in both windows;
and reports the algorithmic bytes of the features launch (kept sources + features, Engine.plan_bytes) over the
k_fused time and over a copy-measured HBM peak (2 GiB device-to-device copy, read + write bytes).  The GPU's
name, power limit and clocks are read in the same call."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_line():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem',
                            '--format=csv,noheader', '-i', os.environ.get('CUDA_VISIBLE_DEVICES', '0').split(',')[0]],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pass
    import torch
    return torch.cuda.get_device_name(0) + ', power limit unknown'


def worker(launches):
    import torch
    from bench import CFG
    from challenge_b200 import _lib as L
    from challenge_b200.engine import Engine
    from challenge_b200.plan import draw_config, uniforms_per_clip
    from challenge_b200.synth import synthetic_banks

    dev = torch.device('cuda', 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    eng = Engine(0)
    eng.set_mel(80)
    bgs, voices, labels, noises = synthetic_banks(CFG['seed'], 2, CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
    reg_ms, plane_bytes = {}, 0
    for name, kind, items, kw in (('bg', L.BANK_BG, bgs, {}), ('voice', L.BANK_VOICE, voices, dict(labels=labels)),
                                  ('noise', L.BANK_NOISE, noises, {})):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        frames = eng.register_bank(kind, items, **kw)
        b.record()
        torch.cuda.synchronize()
        reg_ms[name] = a.elapsed_time(b)
        plane_bytes += sum(2048 * (int(t) + 1) for t in frames)   # one 2 KB row per frame + the last row
    B, T, K = 256, 626, 3
    rng = np.random.default_rng(CFG['seed'])
    y_pred = torch.rand((B, T, K), device=dev, generator=torch.Generator(dev).manual_seed(CFG['seed']))
    cfg = draw_config(B, T, 7, 2, -20, 1.0, 0.5, 6, 24, 1, 16)
    us = [rng.random((B, uniforms_per_clip(cfg))) for _ in range(4)]
    mode = L.FEAT_LOGMEL_MINMAX
    scfg = eng.step_config(cfg, mode, stft_filter=3)
    out = torch.empty((B, 80, T, 2), device=dev)
    st = dict(i=0, frame=torch.empty((B, T, K), device=dev), triples=torch.zeros((B, 3), dtype=torch.int32, device=dev),
              counts=torch.zeros(6, dtype=torch.int64, device=dev))

    def step():
        st['i'] += 1
        eng.step(scfg, us[st['i'] % 4], out=out, frame=st['frame'], y_pred=y_pred, triples=st['triples'],
                 counts=st['counts'])
        eng.counts_wait(0)
    step()
    d = eng.step_draws(scfg)
    eng.upload_plan(d, stft_filter=3)
    _, _, keep = eng.labels()
    bi, bo = eng.plan_bytes(mode, keep.cpu().numpy())
    feat = torch.empty((B, 80, T, 2), device=dev)

    def features():
        eng.features(mode, out=feat)
    for _ in range(3):
        step()
        features()
    # HBM peak by a device-to-device copy (read + write)
    src = torch.empty(1 << 31, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    for _ in range(2):
        dst.copy_(src)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        dst.copy_(src)
    b.record()
    torch.cuda.synchronize()
    peak = 5 * 2 * src.numel() / (a.elapsed_time(b) / 1e3)
    del src, dst
    res = {}
    eng.profile(True)
    for name, fn in (('step', step), ('features', features)):
        ts, kf = [], []
        for _ in range(launches):
            flush.fill_(1)
            torch.cuda.synchronize()
            eng.profile_read(reset=True)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
            ms, n = eng.profile_read(reset=True)
            kf.append(ms * 1e3 / max(n, 1))
        res[name] = float(np.median(ts))
        res[name + '_kfused'] = float(np.median(kf))
    eng.profile(False)
    res.update(reg_ms=reg_ms, plane_bytes=plane_bytes, alg_bytes=float(bi + bo), peak=peak)
    np.save(os.path.join(os.environ['MPB_OUT'], 'features.npy'), feat.cpu().numpy())
    print('RESULT ' + json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--old', required=True, help='libiris.so of the parent revision')
    ap.add_argument('--new', default=os.path.join(ROOT, 'challenge_b200', 'libiris.so'))
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--launches', type=int, default=20)
    ap.add_argument('--worker', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--out', default=None,
                    help='directory for the features of the two builds (default: a temporary directory)')
    args = ap.parse_args()
    if args.worker:
        return worker(args.launches)
    if args.out is None:
        args.out = tempfile.mkdtemp(prefix='mel_plane_bench_')
    print('# GPU: %s' % gpu_line(), flush=True)
    runs = {'old': [], 'new': []}
    for rep in range(args.reps):
        for name, lib in (('old', args.old), ('new', args.new)):
            out = os.path.join(args.out, name)
            os.makedirs(out, exist_ok=True)
            env = dict(os.environ, IRIS_LIB=os.path.abspath(lib), MPB_OUT=out)
            r = subprocess.run([sys.executable, os.path.abspath(__file__), '--worker', '--old', args.old,
                                '--launches', str(args.launches)], env=env, capture_output=True, text=True, cwd=ROOT)
            line = [x for x in r.stdout.splitlines() if x.startswith('RESULT ')]
            if r.returncode or not line:
                sys.stderr.write(r.stdout + r.stderr)
                raise SystemExit('worker %s failed' % name)
            res = json.loads(line[0][7:])
            runs[name].append(res)
            print('rep %d %-3s step %7.1f us (k_fused %6.1f)  features %7.1f us (k_fused %6.1f)  registration '
                  'bg %.1f voice %.1f noise %.1f ms' % (rep, name, res['step'], res['step_kfused'], res['features'],
                                                       res['features_kfused'], res['reg_ms']['bg'],
                                                       res['reg_ms']['voice'], res['reg_ms']['noise']), flush=True)
    print('# B=256 T=626 V=7 M=2, masks + stft_filter(3), 80 mel bins, min-max log-mel fp32; L2 flushed before every '
          'launch; per worker the median of %d launches; workers alternated old / new, %d each'
          % (args.launches, args.reps))
    for name in ('old', 'new'):
        rs = runs[name]
        k = np.median([r['features_kfused'] for r in rs])
        alg, peak = rs[0]['alg_bytes'], np.median([r['peak'] for r in rs])
        print('%-3s step %7.1f us  features %7.1f us  k_fused %6.1f us  algorithmic %.1f MB -> %.2f TB/s = %.2f of '
              'the copy-measured peak %.2f TB/s; registration %.1f ms'
              % (name, np.median([r['step'] for r in rs]), np.median([r['features'] for r in rs]), k, alg / 1e6,
                 alg / (k * 1e-6) / 1e12, alg / (k * 1e-6) / peak, peak / 1e12,
                 np.median([sum(r['reg_ms'].values()) for r in rs])))
    print('# bin planes of the three banks: %.1f MB (new build only)' % (runs['new'][0]['plane_bytes'] / 1e6))
    a = np.load(os.path.join(args.out, 'old', 'features.npy')).astype(np.float64)
    b = np.load(os.path.join(args.out, 'new', 'features.npy')).astype(np.float64)
    ea, eb = np.exp(a), np.exp(b)
    print('# features old vs new on one plan: max|diff| %.3g, normalised max error of exp(features) %.3g'
          % (float(np.abs(a - b).max()), float(np.abs(ea - eb).max() / np.abs(ea).max())))


if __name__ == '__main__':
    main()
