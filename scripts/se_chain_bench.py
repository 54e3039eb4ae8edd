#!/usr/bin/env python
"""The batch of the 'se' model (make_pipeline(seperate_noise_voice=True) -> speech_enhancement_preprocess ->
batch, sj_train.py:99-106): the fused IRIS_FEAT_SE step against the composition IrisDataset ran before it,
on one GPU, alternated within one process.

  python scripts/se_chain_bench.py [--launches N]
Workloads: B = 12 (sj_train's default batch) and 256, T = 512 and 626, waveform and spectrogram banks (the
spectrogram banks are load_wav of the same waveforms), V = 7, M = 2, min_ratio 1, no masks.  Variants, on the
same uniforms (hence the same draws):
  (a) iris_step in IRIS_FEAT_SE: x, only_voice, only_noise and the frame labels;
  (b) what IrisDataset did before: iris_step in IRIS_FEAT_COMPLEX with the [B,V,T,K] labels, the two
      iris_features_select launches (only_voice, only_noise), speech_enhancement_preprocess per clip, and the
      three stacks.
Each batch follows a 256 MiB write that flushes L2.  Host time: perf_counter around the batch and a device
synchronise; device time: CUDA events around the same.  Medians of N batches.  (a) is checked against (b):
array_equal for spectrogram banks, the tolerances of tests/test_gpu_se_chain.py for waveform banks.  The GPU's
name and power limit are printed beside the numbers."""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402

from remap_mel_bench import gpu_line  # noqa: E402


def nmax(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--launches', type=int, default=20, help='timed batches per variant (alternated)')
    args = ap.parse_args()

    import torch
    from bench import CFG
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D
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
    bgs, voices, labels, noises = synthetic_banks(CFG['seed'], 2, CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
    specs = {k: [eng.stft(w).cpu().numpy() for w in ws] for k, ws in (('bg', bgs), ('voice', voices), ('noise', noises))}

    def register(fmt):
        if fmt == 'wave':
            eng.register_bank(L.BANK_BG, bgs)
            eng.register_bank(L.BANK_VOICE, voices, labels=labels)
            eng.register_bank(L.BANK_NOISE, noises)
        else:
            eng.register_bank(L.BANK_BG, specs['bg'])
            eng.register_bank(L.BANK_VOICE, specs['voice'], labels=labels)
            eng.register_bank(L.BANK_NOISE, specs['noise'])

    rng = np.random.default_rng(CFG['seed'])
    print('# V=7 M=2 min_ratio=1, no masks; L2 flushed before every batch; median of %d batches per variant, '
          'variants alternated' % args.launches)
    print('# host = wall time of the batch up to a device synchronise; device = CUDA events around it')
    for fmt in ('wave', 'spec'):
        register(fmt)
        for B in (12, 256):
            for T in (512, 626):
                cfg = draw_config(B, T, 7, 2, -20, 1.0, 0.5, 0, 24, 0, 16)
                s_se = eng.step_config(cfg, L.FEAT_SE)
                s_cx = eng.step_config(cfg, L.FEAT_COMPLEX)
                us = [rng.random((B, uniforms_per_clip(cfg))) for _ in range(2)]
                frame = torch.empty((B, T, K), device=dev)
                vtk = torch.empty((B, 7, T, K), device=dev)
                i = [0]

                def fused():
                    (x, v, n), f = eng.step(s_se, us[i[0] % 2], frame=frame)
                    return x, (f, v, n)

                def composed():
                    x, _ = eng.step(s_cx, us[i[0] % 2], vtk=vtk, want_frame=False)
                    y = (vtk, eng.features(L.FEAT_COMPLEX, select=L.SELECT_VOICES),
                         eng.features(L.FEAT_COMPLEX, select=L.SELECT_BG_NOISE))
                    xs, ys = [], []
                    for b in range(B):
                        xb, yb = D.speech_enhancement_preprocess(x[b], tuple(t[b] for t in y))
                        xs.append(xb)
                        ys.append(yb)
                    return torch.stack(xs), tuple(torch.stack([yb[k] for yb in ys]) for k in range(3))

                variants = {'(a) fused': fused, '(b) composed': composed}
                # (a) against (b) on the same draws
                xa, ya = fused()
                xb, yb = composed()
                torch.cuda.synchronize()
                xa, xb = xa.cpu().numpy(), xb.cpu().numpy()
                va, vb, na, nb = ya[1].cpu().numpy(), yb[1].cpu().numpy(), ya[2].cpu().numpy(), yb[2].cpu().numpy()
                labels_equal = torch.equal(ya[0], yb[0])
                if fmt == 'spec':
                    same = bool(np.array_equal(xa, xb) and np.array_equal(va, vb) and np.array_equal(na, nb))
                    check = 'x / only_voice / only_noise array_equal: %s' % same
                else:
                    ex, ev, en = nmax(xa, xb), float(np.abs(va - vb).max() / np.abs(xb).max()), nmax(na, nb)
                    same = ex <= 1e-5 and ev <= 1e-5 and en <= 1e-5
                    check = 'nmax x %.2e, only_voice %.2e (of max|x|), only_noise %.2e: %s' % (
                        ex, ev, en, 'within 1e-5' if same else 'OUTSIDE 1e-5')
                for fn in variants.values():   # warm-up
                    for _ in range(2):
                        fn()
                torch.cuda.synchronize()
                host = {k: [] for k in variants}
                devt = {k: [] for k in variants}
                for r in range(args.launches):
                    i[0] = r
                    for k, fn in variants.items():
                        flush.fill_(1)
                        torch.cuda.synchronize()
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        t0 = time.perf_counter()
                        a.record()
                        fn()
                        b.record()
                        torch.cuda.synchronize()
                        host[k].append((time.perf_counter() - t0) * 1e6)
                        devt[k].append(a.elapsed_time(b) * 1e3)
                ha, hb = np.median(host['(a) fused']), np.median(host['(b) composed'])
                da, db = np.median(devt['(a) fused']), np.median(devt['(b) composed'])
                print('%-5s B=%3d T=%d  (a) fused    host %9.1f us  device %9.1f us' % (fmt, B, T, ha, da))
                print('%-5s B=%3d T=%d  (b) composed host %9.1f us  device %9.1f us   (b)/(a): host x%.2f, '
                      'device x%.2f' % (fmt, B, T, hb, db, hb / ha, db / da))
                print('#   check: %s; frame labels equal: %s' % (check, labels_equal), flush=True)


if __name__ == '__main__':
    main()
