#!/usr/bin/env python
"""Device time of iris_istft (k_istft) on a pipeline-sized COMPLEX batch.

  python scripts/istft_bench.py [--batch 256] [--frames 626] [--chan 2] [--launches 20] [--out FILE]
Times Engine.istft's kernel on a random [B, 257, T, 2C] float32 batch (default 256 x 626, 2 channels: the batch of
bench.py's shape) into [B, C, 256 (T - 1)], CUDA events around each launch, each launch after a 256 MiB write that
flushes L2, median of --launches.  Reports the algorithmic bytes (read B * 257 * T * 2C * 4, write B * C * L * 4)
over that time and as a fraction of a copy-measured HBM peak (2 GiB device-to-device copy, read + write bytes).
The GPU's name, power limit and clocks are read in the same call.  Writes only to stdout and --out."""
import argparse
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_line():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem',
                        '--format=csv,noheader', '-i', os.environ.get('CUDA_VISIBLE_DEVICES', '0').split(',')[0]],
                       capture_output=True, text=True, timeout=30)
    if r.returncode or not r.stdout.strip():
        raise SystemExit('nvidia-smi could not name the GPU: ' + r.stderr)
    return r.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--frames', type=int, default=626)
    ap.add_argument('--chan', type=int, default=2)
    ap.add_argument('--launches', type=int, default=20)
    ap.add_argument('--out')
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('istft_bench needs a CUDA device')
    from challenge_b200 import _lib as L
    from challenge_b200.engine import Engine

    B, T, Cn = a.batch, a.frames, a.chan
    n = 256 * (T - 1)
    eng = Engine(0)
    dev = eng.device
    x = torch.randn((B, 257, T, 2 * Cn), device=dev)
    out = torch.empty((B, Cn, n), device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = eng._stream()

    def launch():
        L.check(eng.lib.iris_istft(eng._ctx, C.c_void_p(x.data_ptr()), B, T, Cn, 0, C.c_void_p(out.data_ptr()), st))

    for _ in range(3):
        launch()
    ms = []
    for _ in range(a.launches):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    src = torch.empty(1 << 31, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    peak = 5 * 2 * src.numel() / (e0.elapsed_time(e1) / 1e3)

    t = float(np.median(ms)) * 1e-3
    rd, wr = B * 257 * T * 2 * Cn * 4, B * Cn * n * 4
    lines = [
        '# GPU: %s' % gpu_line(),
        '# iris_istft [%d, 257, %d, %d] -> [%d, %d, %d] float32, L2 flushed before every launch, median of %d'
        % (B, T, 2 * Cn, B, Cn, n, a.launches),
        'k_istft %.1f us (min %.1f, max %.1f); algorithmic bytes %.1f MB read + %.1f MB written = %.2f TB/s, '
        '%.2f of the copy-measured peak %.2f TB/s'
        % (t * 1e6, min(ms) * 1e3, max(ms) * 1e3, rd / 1e6, wr / 1e6, (rd + wr) / t / 1e12, (rd + wr) / t / peak,
           peak / 1e12),
    ]
    text = '\n'.join(lines)
    print(text, flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(text + '\n')
    eng.close()


if __name__ == '__main__':
    main()
