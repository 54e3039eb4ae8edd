#!/usr/bin/env python
"""Benchmark of the hot path: augmented spectrogram clips/sec (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # the CUDA path (libiris)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm
  python bench.py ... --dump-outputs DIR                   # + the outputs of the last timed step

--dump-outputs writes what the caller of the timed step holds after the last timed step as
DIR/<name>.npy (float32 / float64, under 64 MB): `features` and `frame_labels` [n, ...] and
`triples` [n, 3] of the clips listed in `clips` (all of them, or a fixed seeded sample when they do
not fit), `counts` [6] (TP, FP, FN, sum n_true, sum n_pred, sum correct over warm-up + timed steps),
and at N > 1 `counts_reduced` / `triples_global` of the all-reduce.  The banks, the uniforms of
every step and the stand-in predictions are seeded, so the same arguments give the same inputs.

Workload (`config.workload`).  N = 1: BASELINE.json configs[1] -- synthetic 2-ch 16 kHz 10 s
clips, background + voices + noise mixed at sampled gains, 6 time + 1 frequency mask, batch 256,
n_fft 512 / hop 256 / 80 mel, min-max + log, frame labels, then the integer F1 / error-rate
counting of the frame labels against a synthetic prediction.  The same line carries
`configs3_one_gpu`: configs[3]'s 8192-clip batch on this one GPU.  N > 1: BASELINE.json
configs[3] -- that 8192-clip batch sharded 8192 / N per GPU, the counts (int64[6] + the
[8192,3] per-sample triples) all-reduced over NCCL inside libiris (the path's only exchange).

One step = one batch = ONE C call (iris_step).  `value` is timed with CUDA events on the
launching stream with the banks resident and the host uniforms drawn beforehand (L2 flushed
between steps); `e2e` iterates the public drop-in chain (make_pipeline(...).map(...).batch(B)...)
with host draws in and pinned host features + labels + counts out.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The CPU arm runs one process per core: BLAS / OpenMP pools inside each worker would
# oversubscribe the box (round 1: 82 clips/s on 16 cores, ~500 with one thread per worker).
# numpy reads these when it is first imported, so they are set before that; the GPU arm only
# uses numpy for the host draws.
_THREAD_ENV = ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS', 'NUMEXPR_NUM_THREADS',
               'VECLIB_MAXIMUM_THREADS')
for _k in _THREAD_ENV:
    os.environ[_k] = '1'

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(n_chan=2, batch=256, n_frame=626, max_voices=7, max_noises=2, snr=-20, min_ratio=1,
           n_mels=80, n_time_masks=6, n_freq_masks=1, n_bg=64, n_voice=256, n_noise=64,
           seed=20202, global_batch_cfg3=8192)
METRIC = 'augmented spectrogram clips/sec'
UNIT = 'clips/s'
DUMP_BYTES = 64_000_000 - 4096     # --dump-outputs: array bytes of all files, .npy headers kept below 4 KB


def dump_outputs(dirname, arrays):
    """--dump-outputs: one DIR/<name>.npy per array (float32 / float64), so that two builds can be
    compared output for output on the same seeded inputs."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(dirname, name + '.npy'), a)
    sys.stderr.write('bench.py: %d arrays, %.1f MB written to %s\n'
                     % (len(arrays), sum(a.nbytes for a in arrays.values()) / 1e6, dirname))


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_fused<FM_MEL> launch of the configs[1]
    workload, read from the newest committed `ncu --set full` capture under profiles/ (below the
    algorithmic bytes: the 175 MB of banks are shared by the clips and partly stay in the 126 MB
    L2; measured with ncu's own cache flush in front of the launch, in place it is 559-575 MB read)."""
    import glob
    import re
    unit = {'byte': 1, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    files = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*_fused_ncu_raw.txt')),
                   key=lambda p: [int(x) for x in re.findall(r'\d+', os.path.basename(p))])
    for path in reversed(files):
        tot = {}
        for line in open(path):
            m = re.match(r'(dram__bytes_(?:read|write)\.sum)\s+([0-9.,]+)\s+(\w+)', line)
            if m and m.group(3) in unit:
                tot[m.group(1)] = float(m.group(2).replace(',', '')) * unit[m.group(3)]
        if len(tot) == 2:
            return int(sum(tot.values())), os.path.relpath(path, ROOT)
    return None, 'no ncu capture under profiles/'


def workload_config(n_gpus, per_gpu=None):
    """N = 1: BASELINE configs[1] (the configuration the metric is quoted on; it fits one GPU).
    N > 1: BASELINE configs[3]: the 8192-clip batch of the same workload sharded 8192 / N per GPU
    (strong scaling) with the NCCL all-reduce of the F1 / ER counts."""
    what = ('2-ch 16 kHz 10 s clips + noise mixing at random SNR + time/freq masking -> min-max '
            'log-mel [B,80,626,2] + frame labels [B,626,3] + F1/ER counts')
    if n_gpus == 1:
        per_gpu = per_gpu or CFG['batch']
        name = 'BASELINE configs[1] (batch %d on 1 B200): ' % per_gpu
        glob_b = per_gpu
    else:
        glob_b = CFG['global_batch_cfg3']
        per_gpu = per_gpu or glob_b // n_gpus
        name = ('BASELINE configs[3] (batch %d sharded over %d B200 = %d clips per GPU, NCCL all-reduce of '
                'the F1/ER counts + the [%d,3] per-sample triples): ' % (glob_b, n_gpus, per_gpu, glob_b))
    return {
        'workload': name + what,
        'batch_per_gpu': per_gpu, 'global_batch': glob_b,
        'n_fft': 512, 'hop': 256, 'n_mels': CFG['n_mels'], 'n_frame': CFG['n_frame'],
        'max_voices': CFG['max_voices'], 'max_noises': CFG['max_noises'],
        'banks': '%d bg x 10 s, %d voices / %d noises 0.5-4 s (seed %d), replicated per GPU' % (
            CFG['n_bg'], CFG['n_voice'], CFG['n_noise'], CFG['seed']),
        'parallelism': 'dp%d (batch sharded by clip; the only exchange is the count all-reduce)' % n_gpus,
        'l2': 'flushed between timed steps (256 MiB write); banks + outputs exceed L2',
    }


# --------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(',')]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': float(np.max(mx)) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def measured_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback 6.65 TB/s (B200_PROFILING.md)'


# --------------------------------------------------------------------------------------
# CPU arm: the oracle restatement of the reference pipeline, timed on host cores
_CPU = {}


def _cpu_prepare(seed):
    """Once, in the parent, before the worker processes are forked: the synthetic banks and
    load_wav (STFT) of every source -- the reference does this offline and keeps the result as
    its pickled banks (utils.load_data), so it is outside the timed region; the workers inherit
    the arrays copy-on-write."""
    if _CPU.get('seed') == seed:
        return
    import torch
    torch.set_num_threads(1)
    from challenge_b200.synth import synthetic_banks
    from oracle.data_utils import load_wav_array
    raw = synthetic_banks(seed, CFG['n_chan'], CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
    _CPU['raw'] = raw
    _CPU['spec'] = tuple([load_wav_array(w) for w in raw[k]] for k in (0, 1, 3))
    _CPU['seed'] = seed


def _cpu_worker_init():
    import torch
    torch.set_num_threads(1)


def _cpu_clips(args):
    """The reference chain for clips [lo, hi) of draws d."""
    d, lo, hi = args
    from oracle import chain
    from oracle import metrics as M
    banks = _CPU['spec']
    x, y, _, _ = chain.dataset_batch(banks[0], banks[1], _CPU['raw'][2], banks[2], d,
                                     mode='logmel_minmax', n_mels=CFG['n_mels'],
                                     clips=range(lo, hi))
    yp = np.clip(y + 0.25, 0, 1).astype(np.float32)
    M.er_parts(y, yp)
    M.f1_counts(y, yp)
    return hi - lo


def cpu_draws(n_clips, seed):
    from challenge_b200.plan import draw_batch
    raw = _CPU['raw']
    frames = [np.array([1 + w.shape[1] // 256 for w in raw[k]], np.int32) for k in (0, 1, 3)]
    rng = np.random.default_rng(seed)
    return draw_batch(rng, n_clips, CFG['n_frame'], frames[0], frames[1], frames[2],
                      max_voices=CFG['max_voices'], max_noises=CFG['max_noises'], snr=CFG['snr'],
                      min_ratio=CFG['min_ratio'], n_time_masks=CFG['n_time_masks'],
                      n_freq_masks=CFG['n_freq_masks'])


class CpuPool:
    """All host cores: one single-threaded worker process per core (fork; banks shared
    copy-on-write), clips handed out two at a time as workers become free."""

    def __init__(self, cores):
        import multiprocessing as mp
        self.cores = cores
        _cpu_prepare(CFG['seed'])
        self.pool = mp.get_context('fork').Pool(cores, initializer=_cpu_worker_init) if cores > 1 else None

    def run(self, d, n_clips):
        """Wall seconds for n_clips clips of d spread over the cores."""
        chunks = [(d, lo, min(lo + 2, n_clips)) for lo in range(0, n_clips, 2)]
        t0 = time.perf_counter()
        if self.pool is None:
            for c in chunks:
                _cpu_clips(c)
        else:
            for _ in self.pool.imap_unordered(_cpu_clips, chunks):
                pass
        return time.perf_counter() - t0

    def close(self):
        if self.pool is not None:
            self.pool.terminate()


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def thread_settings():
    return ', '.join('%s=%s' % (k, os.environ.get(k)) for k in _THREAD_ENV[:3])


def run_reference_arm(args):
    """--impl reference: the reference's CPU algorithm (oracle port) on all host cores; each step
    is a bounded sample of the same workload (clips are independent, so clips/s does not depend on
    the batch they are drawn into)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = host_cores()
    per_step = max(16 * cores, 64)   # as in cpu_baseline(): 4 clips per core left the workers ragged (303 vs 496 clips/s on 16 cores)
    pool = CpuPool(cores)
    try:
        d = cpu_draws(per_step * (args.steps + args.warmup), CFG['seed'] + 1)
        times = []
        for s in range(args.warmup + args.steps):
            ds = d.slice(s * per_step, (s + 1) * per_step)
            dt = pool.run(ds, per_step)
            if s >= args.warmup:
                times.append(dt)
    finally:
        pool.close()
    total = float(np.sum(times))
    value = per_step * args.steps / total
    sample = ('%d clips per step on %d worker processes, one thread each (%s); per-source load_wav '
              '(STFT) precomputed offline as in the reference' % (per_step, cores, thread_settings()))
    cfg = workload_config(args.gpus)
    cfg['clips_per_step'] = per_step
    cfg['note'] = ('CPU arm: every step is a bounded sample of %d clips of the workload above (not the '
                   'whole batch); compare clips/s, not ms_per_step' % per_step)
    out = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT,
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * total / args.steps, 'higher_is_better': True,
        'scaling': 'weak' if args.gpus == 1 else 'strong',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': cfg,
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------------------
def drop_in_dataset(banks, B):
    """The public drop-in call chain of sj_train.make_dataset (sj_train.py:92-130) on the GPU
    pipeline: make_pipeline -> to_frame_labels -> augment -> batch -> complex_to_magphase ->
    magphase_to_mel(80) -> minmax -> log_on_mel (lowered to one iris_step per batch)."""
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import make_pipeline
    bgs, voices, labels, noises = banks
    ds = make_pipeline(bgs, voices, labels, noises, n_frame=CFG['n_frame'], max_voices=CFG['max_voices'],
                       max_noises=CFG['max_noises'], snr=CFG['snr'], min_ratio=CFG['min_ratio'])
    return (ds.map(D.to_frame_labels).map(D.augment).batch(B).map(TR.complex_to_magphase)
            .map(TR.magphase_to_mel(CFG['n_mels'])).map(D.minmax).map(D.log_on_mel))


def run_gpu_arm(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from challenge_b200 import _lib as L
    from challenge_b200 import _ops as O
    from challenge_b200.plan import draw_config, uniforms_per_clip
    from challenge_b200.synth import synthetic_banks

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    from challenge_b200.dist import bind_to_gpu_numa, shard_range
    numa_cores = bind_to_gpu_numa(local) if world > 1 else None   # before any pinned allocation
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    banks = synthetic_banks(CFG['seed'], CFG['n_chan'], CFG['n_bg'], CFG['n_voice'], CFG['n_noise'])
    T, K = CFG['n_frame'], 3
    if world == 1:
        B = Bg = args.batch or CFG['batch']   # --batch: experiments only (config.workload names it)
        lo = 0
    else:
        Bg = CFG['global_batch_cfg3']
        lo, hi = shard_range(Bg, world, rank)
        B = hi - lo
    O.set_seed(CFG['seed'] + 100 + rank)
    ds = drop_in_dataset(banks, B)          # registers the banks on this pipeline's engine
    eng = ds.engine
    fused, _, _ = ds._prepare()             # sets the mel matrix; the step configuration below is the lowered chain
    assert fused['mode'] == L.FEAT_LOGMEL_MINMAX
    rng = np.random.default_rng(CFG['seed'] + 100 + rank)

    comm = None
    if world > 1:      # the communicator of the count all-reduce lives inside libiris
        ids = [eng.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = eng.nccl_comm(ids[0], rank, world)

    def step_setup(b, b_global, b_lo):
        cfg = draw_config(b, T, CFG['max_voices'], CFG['max_noises'], CFG['snr'], CFG['min_ratio'], 0.5,
                          CFG['n_time_masks'], 24, CFG['n_freq_masks'], 16)
        st = dict(scfg=eng.step_config(cfg, L.FEAT_LOGMEL_MINMAX), n_u=uniforms_per_clip(cfg), b=b,
                  feat=[torch.empty((b, CFG['n_mels'], T, CFG['n_chan']), device=dev) for _ in range(2)],
                  frame=[torch.empty((b, T, K), device=dev) for _ in range(2)],
                  # stand-in for the model output the metric kernels score (fixed, seeded, generated once)
                  y_pred=torch.rand((b, T, K), device=dev,
                                    generator=torch.Generator(dev).manual_seed(CFG['seed'] + rank)),
                  counts=torch.zeros(6, dtype=torch.int64, device=dev),
                  reduced=torch.zeros(6, dtype=torch.int64, device=dev),
                  send=torch.zeros((b_global, 3), dtype=torch.int32, device=dev),
                  glob=torch.zeros((b_global, 3), dtype=torch.int32, device=dev), b_global=b_global, lo=b_lo)
        return st

    def one_step(st, u, i):
        """ONE C call (iris_step): draws -> plan upload -> labels -> {features || metric counts
        (+ count all-reduce on the side stream)}."""
        j = i & 1
        eng.step(st['scfg'], u, out=st['feat'][j], frame=st['frame'][j], y_pred=st['y_pred'],
                 triples=st['send'][st['lo']:st['lo'] + st['b']], counts=st['counts'], comm=comm,
                 counts_reduced=st['reduced'] if comm is not None else None,
                 triples_send=st['send'] if comm is not None else None,
                 triples_global=st['glob'] if comm is not None else None, global_batch=st['b_global'])
        return j

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    LAG = 2          # the reduced counts are a logged metric: consumed two steps late (N > 1)

    def last_outputs(st, j):
        """What the caller of the timed step holds after its last step: the features, frame labels and
        per-sample triples of every clip (of a fixed, seeded sample of the clips when they exceed
        DUMP_BYTES), the counts accumulated over all steps (+ the all-reduced ones at N > 1)."""
        b, lo = st['b'], st['lo']
        fixed = 6 * 8 + ((6 + st['b_global'] * 3) * 8 if comm is not None else 0)
        per_clip = (st['feat'][j][0].numel() + st['frame'][j][0].numel()) * 4 + 3 * 8 + 8
        n = min(b, (DUMP_BYTES - fixed) // per_clip)
        clips = np.arange(b) if n == b else np.sort(np.random.default_rng(CFG['seed']).choice(b, n, replace=False))
        idx = torch.from_numpy(clips).to(dev)
        out = {'clips': clips.astype(np.float64),
               'features': st['feat'][j].index_select(0, idx).cpu().numpy(),
               'frame_labels': st['frame'][j].index_select(0, idx).cpu().numpy(),
               'triples': st['send'][lo:lo + b].index_select(0, idx).cpu().numpy().astype(np.float64),
               'counts': st['counts'].cpu().numpy().astype(np.float64)}
        if comm is not None:
            out['counts_reduced'] = st['reduced'].cpu().numpy().astype(np.float64)
            out['triples_global'] = st['glob'].cpu().numpy().astype(np.float64)
        return out

    def timed_loop(st, n_warm, n_steps, sampler=None, keep_last=False):
        us = [rng.random((st['b'], st['n_u'])) for _ in range(n_warm + n_steps)]
        eng.profile(False)
        for s in range(n_warm):
            one_step(st, us[s], s)
            eng.counts_wait(0)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if sampler is not None:
            sampler.start()
        eng.profile(True)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(n_steps)]
        for s in range(n_steps):
            flush.fill_(s & 0xff)                               # evict L2 (untimed)
            ev[s][0].record()
            one_step(st, us[n_warm + s], s)
            # one GPU: the step ends when its counts are there.  Several ranks: the collective is also a
            # rendezvous of the ranks, so a step only waits for the counts issued LAG steps earlier
            # and the last ones are drained inside the timed region.
            eng.counts_wait(0 if (world == 1 or s == n_steps - 1) else LAG)
            ev[s][1].record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        last = last_outputs(st, (n_steps - 1) & 1) if keep_last else None   # before the replay below overwrites them
        total_ms = float(np.sum([a.elapsed_time(b) for a, b in ev]))
        fused_ms, n_fused = eng.profile_read()
        eng.profile(False)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # algorithmic bytes (SURVEY.md 8d: kept sources only) of EVERY timed step: the steps are replayed
        # untimed with the same uniforms, the keep flags of each plan read back (they differ by ~2 % from
        # draw to draw, which a figure taken from the last plan alone would carry into `frac`)
        k_clips = eng.profile_clips() or st['b']   # the launch the roofline hook timed: the batch, or the first part of a split batch
        alg = ker = 0
        for s in range(n_steps):
            one_step(st, us[n_warm + s], s)
            eng.counts_wait(0)
            _, _, keep = eng.labels()
            keep = keep.cpu().numpy()
            bi, bo = eng.plan_bytes(L.FEAT_LOGMEL_MINMAX, keep)
            ki, ko = eng.plan_bytes(L.FEAT_LOGMEL_MINMAX, keep, clips=(0, k_clips))
            alg += bi + bo
            ker += ki + ko
        return dict(total_ms=total_ms, total_ms_max=float(t.item()), fused_ms=fused_ms, n_fused=n_fused,
                    alg_bytes=alg / n_steps, kernel_bytes=ker / n_steps, kernel_clips=k_clips, last=last)

    # ---- device-timed: inputs (banks) resident, the uniforms of every step drawn beforehand ----
    st = step_setup(B, Bg, lo)
    sampler = ClockSampler(local)
    r = timed_loop(st, args.warmup, args.steps, sampler, keep_last=args.dump_outputs is not None and rank == 0)
    value = Bg * args.steps / (r['total_ms_max'] / 1e3)

    # ---- end to end through the public drop-in call chain: host uniforms in (numpy) -> one iris_step
    # per batch inside IrisDataset -> features + labels + counts copied to pinned host memory; the
    # device->host copies of batch i overlap the kernels of batch i+1 (two buffers, two streams) ----
    n_e2e = 0 if args.no_e2e else args.steps
    n_e2e_warm = 0 if args.no_e2e else max(args.warmup, 3)
    feat_shape = (B, CFG['n_mels'], T, CFG['n_chan'])
    h2d = d2h = 0
    e2e_value = e2e_dev_value = None
    numa_node = None
    if not args.no_e2e:
        h_feat = []
        for _ in range(2):      # pinned staging on the NUMA node of this rank's GPU
            a, numa_node = eng.host_alloc(feat_shape, np.float32)
            h_feat.append(torch.from_numpy(a))
        h_lbl = [torch.empty((B, T, K), dtype=torch.float32, pin_memory=True) for _ in range(2)]
        h_cnt = [torch.empty(6, dtype=torch.int64, pin_memory=True) for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        copied = [torch.cuda.Event() for _ in range(2)]
        e_counts = torch.zeros(6, dtype=torch.int64, device=dev)
        e_reduced = torch.zeros(6, dtype=torch.int64, device=dev)
        it = iter(ds)

        def e2e_step(i, features_to_host=True):
            nonlocal h2d, d2h
            j = i & 1
            x, y = next(it)                                     # host uniforms -> iris_step (public drop-in)
            eng.metric_counts(y, st['y_pred'], counts=e_counts, want_er=False)
            src_counts = e_counts
            if comm is not None:
                eng.allreduce_counts(comm, e_counts, e_reduced)
                src_counts = e_reduced
            done = torch.cuda.Event()
            done.record()
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done)
                if features_to_host:
                    h_feat[j].copy_(x, non_blocking=True)
                h_lbl[j].copy_(y, non_blocking=True)
                h_cnt[j].copy_(src_counts, non_blocking=True)
                copied[j].record()
                x.record_stream(copy_stream)
                y.record_stream(copy_stream)
            copied[j ^ 1].synchronize()                         # the consumer has batch i-1 on the host
            if features_to_host:
                h2d = eng.plan_upload_bytes()   # the packed plan blob (segments, ids, masks) of this batch
                d2h = h_feat[j].numel() * 4 + h_lbl[j].numel() * 4 + h_cnt[j].numel() * 8

        def e2e_loop(n_warm, n, to_host):
            for i in range(n_warm):
                e2e_step(i, to_host)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for i in range(n):
                e2e_step(n_warm + i, to_host)
            torch.cuda.synchronize()
            t = torch.tensor([max(time.perf_counter() - t0, 1e-9)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return Bg * n / float(t.item()), float(t.item())

        e2e_value, e2e_s = e2e_loop(n_e2e_warm, n_e2e, True)
        # the same loop with the features left on the device (what a Keras / torch model fed through
        # DLPack sees: INTEGRATION.md section 3); labels and counts still go to the host
        e2e_dev_value, _ = e2e_loop(2, n_e2e, False)
        # the ceiling of the read-back: every rank copies a feature batch device -> pinned host,
        # nothing else running, all ranks at once
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(8):
            h_feat[i & 1].copy_(st['feat'][i & 1], non_blocking=True)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        d2h_ceiling = 8 * h_feat[0].numel() * 4 / float(t.item()) / 1e9
    clocks = sampler.stop()

    # ---- N = 1: the multi-GPU configuration (configs[3], 8192 clips) on this one GPU, for the
    # strong-scaling base of the N > 1 lines ----
    cfg3 = None
    if world == 1 and not args.no_cfg3:
        st3 = step_setup(CFG['global_batch_cfg3'], CFG['global_batch_cfg3'], 0)
        r3 = timed_loop(st3, 5, 4)     # 5 warm-up steps: every slot of the plan ring is allocated
        cfg3 = {'workload': 'BASELINE configs[3] on ONE GPU: batch 8192 in one step (same per-clip workload)',
                'value': 8192 * 4 / (r3['total_ms'] / 1e3), 'unit': UNIT, 'ms_per_step': r3['total_ms'] / 4,
                'steps': 4, 'algorithmic_bytes_per_step': int(r3['alg_bytes']),
                'step_frac': r3['alg_bytes'] * 4 / (r3['total_ms'] / 1e3) / 1e9 / measured_peak()[0]}
        del st3
        torch.cuda.empty_cache()

    # ---- N = 1: BASELINE configs[4], the input-bound check.  sj_train.py's Keras step cannot run
    # (TensorFlow is absent), so a SUBSTITUTE consumer of the pipeline's tensors is timed beside it ----
    consumer = None
    if world == 1 and not args.no_consumer_check:
        consumer = consumer_check(dev, B, T, K, r['total_ms'] / args.steps)

    peak, peak_src = measured_peak()
    fused_avg_ms = r['fused_ms'] / max(r['n_fused'], 1)
    achieved = r['kernel_bytes'] / (fused_avg_ms / 1e3) / 1e9 if fused_avg_ms > 0 else 0.0
    traffic, traffic_src = ncu_traffic()
    # k_labels also builds the per-tile stage lists of the feature kernel behind it (no k_tiles launch
    # on the step path); the metric leg forks behind k_fused and runs beside k_logmel_post
    KERNELS = ['k_labels', 'k_fused<FM_MEL>', 'k_logmel_post', 'k_metric_counts']
    out = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': r['total_ms_max'] / args.steps,
        'higher_is_better': True, 'scaling': 'weak' if world == 1 else 'strong', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(world, B),
        'clocks': clocks,
        'kernels_per_step': KERNELS,
        'roofline': {'bound': 'hbm', 'kernel': 'k_fused<FM_MEL>', 'achieved': achieved,
                     'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak if peak else None,
                     'traffic': traffic, 'traffic_source': traffic_src,
                     'peak_source': peak_src,
                     'algorithmic_bytes_per_launch': int(r['kernel_bytes']),
                     'clips_per_launch': int(r['kernel_clips']),
                     'launch_note': ('one k_fused launch over the whole batch (CUDA events around it on the '
                                     'launching stream; its tile lists were built by k_labels)' if r['kernel_clips'] == B else
                                     'the batch is split into parts of %d clips whose second pass (k_logmel_post) '
                                     'overlaps the next part; the hook times k_tiles + k_fused of the first part'
                                     % r['kernel_clips']),
                     'algorithmic_bytes_per_step': int(r['alg_bytes']),
                     'kernel_ms': fused_avg_ms,
                     'kernel_share_of_step': (r['fused_ms'] * B / max(r['kernel_clips'], 1)) / r['total_ms'],
                     'step_frac': r['alg_bytes'] * args.steps / (r['total_ms'] / 1e3) / 1e9 / peak},
        'step_call': 'one iris_step C call per batch (host planner + plan upload + 4 kernel launches'
                     + (' + 1 NCCL group' if world > 1 else '') + ')',
    }
    if e2e_value is not None:
        out['e2e'] = {
            'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
            'd2h_gb_per_s_per_rank': d2h * n_e2e / e2e_s / 1e9,
            'd2h_ceiling_gb_per_s_per_rank': d2h_ceiling,
            'd2h_ceiling_note': 'plain cudaMemcpyAsync of the feature batch to the same pinned buffers, all ranks at '
                                'once, nothing else running: what the host fabric of this box gives',
            'pinned_numa_node': numa_node,
            'note': 'public drop-in chain (make_pipeline(...).map(to_frame_labels).map(augment).batch(B)'
                    '.map(complex_to_magphase).map(magphase_to_mel(80)).map(minmax).map(log_on_mel)) iterated '
                    'on the host: numpy uniforms -> one iris_step per batch -> metric counts -> features + '
                    'labels + counts copied to pinned host memory (NUMA-local to the GPU); wall clock; the D2H '
                    'of batch i overlaps the kernels of batch i+1; PCIe-bound (features are 400 KB per clip)',
            'features_on_device_value': e2e_dev_value,
            'features_on_device_note': 'same loop, features handed over on the device (DLPack) instead of '
                                       'copied to the host; labels + counts still read back'}
    if cfg3 is not None:
        out['configs3_one_gpu'] = cfg3
    if consumer is not None:
        out['input_bound_check'] = consumer
    if world > 1:
        out['config']['host_binding'] = ('each rank pinned to the %d cores NVML lists for its GPU' % len(numa_cores)
                                         if numa_cores else 'none (NVML affinity not available)')
        out['config']['count_allreduce'] = ('iris_allreduce_counts (NCCL inside libiris, one group of int64[6] + '
                                            'int32[%d,3] per step) on the context side stream; a step waits for the '
                                            'collective issued %d steps earlier, the last ones are drained inside the '
                                            'timed region' % (Bg, LAG))
        out['config']['efficiency_base'] = ('strong scaling of configs[3]: compare with configs3_one_gpu.value of the '
                                            'N = 1 line (8192 clips on one GPU), not with its configs[1] value')
    out['gpu_launches'] = int(args.steps * (len(KERNELS) + (1 if world > 1 else 0)))
    if comm is not None:
        torch.cuda.synchronize()
        dist.barrier()
        eng.nccl_comm_destroy(comm)
    if rank == 0:
        if not args.no_cpu_baseline:      # the CPU leg, on rank 0's host cores, at every N
            out['cpu_baseline'] = cpu_baseline()
        if args.dump_outputs is not None:
            dump_outputs(args.dump_outputs, r['last'])
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def consumer_check(dev, B, T, K, pipeline_ms):
    """BASELINE configs[4] ("pipeline feeding a train step: is the model input-bound?").  The
    reference's consumer is a Keras EfficientNet step (sj_train.py:158-188, 454-513) and cannot run
    here; the stand-in is a small bf16 conv net over the pipeline's own tensors ([B,80,T,2] features,
    [B,T,3] frame labels): 4 stride-2 conv stages + a frame-wise head, forward + backward + SGD in
    torch (library kernels; NOT part of the measured path, reported beside it)."""
    import torch

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            ch = [CFG['n_chan'], 32, 64, 128, 256]
            self.convs = torch.nn.ModuleList([torch.nn.Conv2d(ch[i], ch[i + 1], 3, stride=(2, 1), padding=1)
                                              for i in range(4)])
            self.head = torch.nn.Conv1d(256 * (CFG['n_mels'] // 16), K, 1)

        def forward(self, x):                      # [B, mel, T, C]
            x = x.permute(0, 3, 1, 2)
            for c in self.convs:
                x = torch.relu(c(x))
            return self.head(x.flatten(1, 2)).transpose(1, 2)

    try:
        net = Net().to(dev).to(memory_format=torch.channels_last)
        opt = torch.optim.SGD(net.parameters(), lr=1e-3)
        x = torch.randn(B, CFG['n_mels'], T, CFG['n_chan'], device=dev)
        y = (torch.rand(B, T, K, device=dev) < 0.3).float()

        def train_step():
            with torch.autocast('cuda', dtype=torch.bfloat16):
                loss = torch.nn.functional.binary_cross_entropy_with_logits(net(x).float(), y)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

        for _ in range(3):
            train_step()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(5):
            train_step()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 5
        del net, opt, x, y
        torch.cuda.empty_cache()
    except Exception as ex:   # the check is a side report: never fail the bench line over it
        return {'workload': 'BASELINE configs[4] input-bound check', 'unavailable': repr(ex)[:200]}
    return {'workload': 'BASELINE configs[4] input-bound check with a SUBSTITUTE consumer (TensorFlow / sj_train.py '
                        'cannot run here): 4-stage bf16 conv net + frame-wise head on [B,80,626,2] -> [B,626,3], '
                        'forward + backward + SGD in torch, batch %d' % B,
            'consumer_ms_per_step': ms, 'pipeline_ms_per_step': pipeline_ms,
            'pipeline_share_of_consumer_step': pipeline_ms / ms,
            'input_bound': bool(pipeline_ms > ms)}


def cpu_baseline():
    """The oracle port of the reference pipeline timed on this box's host cores on a bounded
    sample of the same workload (reported beside the GPU number; not the target)."""
    cores = host_cores()
    n = max(16 * cores, 64)         # ~10-15 s of CPU work
    pool = CpuPool(cores)
    try:
        d = cpu_draws(n, CFG['seed'] + 2)
        pool.run(d.slice(0, 2 * cores), 2 * cores)          # warm the workers (imports, first touches)
        wall = pool.run(d, n)
        one = CpuPool(1)
        n1 = 16
        one.run(d.slice(0, 2), 2)
        t1 = one.run(d.slice(0, n1), n1)
    finally:
        pool.close()
    return {'value': n / wall, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'single_thread_value': n1 / t1,
            'sample': '%d clips of the same workload on %d worker processes, one thread each (%s), '
                      'per-source load_wav (STFT) precomputed offline as in the reference; '
                      'single_thread_value: %d clips on 1 thread' % (n, cores, thread_settings(), n1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true', help='profiling runs only')
    ap.add_argument('--batch', type=int, default=0, help='N = 1 only: another batch size (experiments)')
    ap.add_argument('--no-cfg3', action='store_true', help='skip the 8192-clip single-GPU leg (profiling runs)')
    ap.add_argument('--no-consumer-check', action='store_true', help='skip the configs[4] substitute-consumer leg')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step (rank 0) to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs is not None and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200 (the reference arm keeps no outputs)')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == '__main__':
    main()
