#!/usr/bin/env python
"""Times iris_features(MEL / LOGMEL_MINMAX) for cfg1 / cfg2 at C=2, B=256 (other builds via IRIS_LIB)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from challenge_b200 import _lib as L
from challenge_b200.engine import Engine
from challenge_b200.plan import draw_batch
from challenge_b200.synth import synthetic_banks
B = 256
eng = Engine(0); eng.set_mel(80)
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
def timeit(fn, n=15):
    for _ in range(3): fn()
    ts = []
    for i in range(n):
        flush.fill_(i & 255)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ts)), float(np.min(ts))
bgs, voices, labels, noises = synthetic_banks(20202, 2, 64, 256, 64)
bf = eng.register_bank(L.BANK_BG, bgs); vf = eng.register_bank(L.BANK_VOICE, voices, labels=labels)
nf = eng.register_bank(L.BANK_NOISE, noises)
rng = np.random.default_rng(1)
plans = {'cfg1': draw_batch(rng, B, 626, bf),
         'cfg2': draw_batch(rng, B, 626, bf, vf, nf, max_voices=7, max_noises=2, snr=-20, min_ratio=1, n_time_masks=6, n_freq_masks=1)}
out = []
for name, d in plans.items():
    eng.upload_plan(d)
    if d.max_voices: eng.labels()
    for mname, mode in (('MEL', L.FEAT_MEL), ('LMM', L.FEAT_LOGMEL_MINMAX)):
        o = torch.empty(eng.feature_shape(mode), device='cuda')
        med, mn = timeit(lambda: eng.features(mode, out=o))
        out.append('%s %s %.1f/%.1f' % (name, mname, med, mn))
print('%-28s %s' % (os.path.basename(os.path.dirname(os.environ.get('IRIS_LIB') or 'x/default/l')), ' | '.join(out)))
