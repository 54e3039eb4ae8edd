"""GPU tests of the one-call batch step (iris_step), the DLPack hand-over, per-pipeline bank
sets and the tf.data surface of IrisDataset -- all through the C ABI, checked against the CPU
oracle on the draws the step itself made (iris_step_draws)."""
import os

import numpy as np
import pytest

from conftest import nmax_err

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _oracle(w, d, **kw):
    from oracle import chain
    return chain.dataset_batch(w.o_bg, w.o_voice, w.labels, w.o_noise, d, **kw)


def _step_cfg(engine, B, T, mode, V=7, M=2, masks=True, min_ratio=1.0):
    from challenge_b200.plan import draw_config
    cfg = draw_config(B, T, V, M, -20, min_ratio, 0.5, 6 if masks else 0, 24, 1 if masks else 0, 16)
    return engine.step_config(cfg, mode)


@pytest.mark.parametrize('T,B', [(626, 6), (300, 9)])
def test_step_equals_the_multi_call_path_and_the_oracle(engine, workload_factory, T, B):
    """iris_step(uniforms) == iris_draw_batch -> iris_plan_upload -> iris_labels -> iris_features
    bit for bit, and both match the oracle on the same draws."""
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draws_from_uniforms, uniforms_per_clip
    w = workload_factory(2)
    scfg = _step_cfg(engine, B, T, L.FEAT_LOGMEL_MINMAX)
    u = np.random.default_rng(T).random((B, uniforms_per_clip(scfg.draw)))
    keep = torch.zeros((B, 7), dtype=torch.uint8, device='cuda')
    x, frame = engine.step(scfg, u, keep=keep)
    x, frame = x.clone(), frame.clone()
    d_step = engine.step_draws(scfg)
    d = draws_from_uniforms(scfg.draw, u, w.bg_frames, w.voice_frames, w.noise_frames)
    for k, v in vars(d).items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(getattr(d_step, k), v), k
    engine.upload_plan(d)
    frame2, _, keep2 = engine.labels()
    x2 = engine.features(L.FEAT_LOGMEL_MINMAX)
    assert torch.equal(x, x2) and torch.equal(frame, frame2) and torch.equal(keep, keep2)
    ref, ref_y, _, ref_keep = _oracle(w, d_step, mode='logmel_minmax')
    assert nmax_err(x.cpu().numpy(), ref) < TOL
    assert np.array_equal(frame.cpu().numpy(), ref_y)
    assert np.array_equal(keep.cpu().numpy(), np.stack(ref_keep))


def test_step_metric_leg_counts_bit_exact(engine, workload_factory):
    """The metric leg of iris_step (k_metric_counts on the side stream) against metrics.py:217-298
    restated: per-sample (n_true, n_pred, correct), accumulated TP / FP / FN and triple sums."""
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200.plan import uniforms_per_clip
    from oracle import metrics as M
    w = workload_factory(2)
    B, T = 12, 626
    scfg = _step_cfg(engine, B, T, L.FEAT_MEL)
    rng = np.random.default_rng(5)
    counts = torch.zeros(6, dtype=torch.int64, device='cuda')
    tot = np.zeros(6, np.int64)
    for it in range(3):
        y_pred = torch.rand((B, T, 3), device='cuda')
        triples = torch.zeros((B, 3), dtype=torch.int32, device='cuda')
        x, frame = engine.step(scfg, rng.random((B, uniforms_per_clip(scfg.draw))), y_pred=y_pred,
                               triples=triples, counts=counts)
        engine.counts_wait(0)
        torch.cuda.synchronize()
        yt, yp = frame.cpu().numpy(), y_pred.cpu().numpy()
        nt, npd, co = M.er_parts(yt, yp)
        assert np.array_equal(triples.cpu().numpy(), np.stack([nt, npd, co], 1))
        tot[:3] += np.array(M.f1_counts(yt, yp), np.int64)
        tot[3:] += np.array([nt.sum(), npd.sum(), co.sum()], np.int64)
        assert np.array_equal(counts.cpu().numpy(), tot), it
    er = engine.er_from_triples(triples)
    assert np.array_equal(er.cpu().numpy(), M.er_from_parts(nt, npd, co))


def test_step_runs_ahead_of_the_device(engine, workload_factory):
    """Many steps queued without a host sync (ring of pinned plan buffers): the last result is the
    same as when every step is synchronised."""
    import torch
    from challenge_b200 import _lib as L
    from challenge_b200.plan import uniforms_per_clip
    w = workload_factory(2)
    scfg = _step_cfg(engine, 16, 626, L.FEAT_LOGMEL_MINMAX)
    us = [np.random.default_rng(i).random((16, uniforms_per_clip(scfg.draw))) for i in range(12)]
    outs = [engine.step(scfg, u) for u in us]          # no synchronisation in between
    torch.cuda.synchronize()
    for u, (x, y) in list(zip(us, outs))[-3:]:
        x2, y2 = engine.step(scfg, u)
        torch.cuda.synchronize()
        assert torch.equal(x, x2) and torch.equal(y, y2)


def test_dlpack_round_trip_writes_in_place(engine, workload_factory):
    """north_star: tensors are exchanged via DLPack.  A tensor exported with to_dlpack is filled by
    iris_features_dlpack / iris_step_dlpack through data + byte_offset (no copy, same data_ptr) and a
    second call overwrites it in place; shape / dtype / device mismatches are refused."""
    import torch
    from torch.utils.dlpack import from_dlpack, to_dlpack
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch, uniforms_per_clip
    w = workload_factory(2)
    rng = np.random.default_rng(11)
    d = draw_batch(rng, 4, 626, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=7, max_noises=2,
                   min_ratio=1, n_time_masks=6, n_freq_masks=1)
    engine.upload_plan(d)
    direct = engine.features(L.FEAT_LOGMEL_MINMAX)
    # the tensor sits at a byte offset inside a larger allocation
    big = torch.zeros(8 + direct.numel(), device='cuda')
    t = big[8:].view(direct.shape)
    cap = to_dlpack(t)
    engine.features_dlpack(L.FEAT_LOGMEL_MINMAX, cap)
    back = from_dlpack(cap)                       # consumes the capsule; shares the memory
    assert back.data_ptr() == t.data_ptr()
    assert torch.equal(back, direct) and not big[:8].any()
    # second call through a fresh capsule of the same tensor: written in place
    d2 = draw_batch(rng, 4, 626, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=7, max_noises=2,
                    min_ratio=1, n_time_masks=6, n_freq_masks=1)
    engine.upload_plan(d2)
    engine.features_dlpack(L.FEAT_LOGMEL_MINMAX, to_dlpack(t))
    assert torch.equal(back, engine.features(L.FEAT_LOGMEL_MINMAX)) and not torch.equal(back, direct)
    # refusals: alignment (the kernels store 16-byte vectors), shape, dtype, host memory, non-contiguous
    with pytest.raises(ValueError, match='aligned'):
        engine.features_dlpack(L.FEAT_LOGMEL_MINMAX, to_dlpack(big[7:7 + direct.numel()].view(direct.shape)))
    with pytest.raises(ValueError):
        engine.features_dlpack(L.FEAT_LOGMEL_MINMAX, to_dlpack(torch.zeros((4, 80, 626, 3), device='cuda')))
    with pytest.raises(ValueError):
        engine.features_dlpack(L.FEAT_LOGMEL_MINMAX, to_dlpack(torch.zeros(direct.shape, device='cuda', dtype=torch.float64)))
    with pytest.raises(ValueError):
        engine.features_dlpack(L.FEAT_LOGMEL_MINMAX, to_dlpack(torch.zeros(direct.shape)))
    with pytest.raises(ValueError):
        engine.features_dlpack(L.FEAT_LOGMEL_MINMAX,
                               to_dlpack(torch.zeros((4, 80, 2, 626), device='cuda').permute(0, 1, 3, 2)))
    # the whole step through DLPack
    scfg = _step_cfg(engine, 4, 626, L.FEAT_LOGMEL_MINMAX)
    u = rng.random((4, uniforms_per_clip(scfg.draw)))
    x, y = engine.step(scfg, u)
    fx, fy = torch.empty_like(x), torch.empty_like(y)
    engine.step_dlpack(scfg, u, to_dlpack(fx), to_dlpack(fy))
    assert torch.equal(fx, x) and torch.equal(fy, y)


def _banks(seed, n_chan=2):
    from challenge_b200.synth import synthetic_banks
    return synthetic_banks(seed, n_chan, n_bg=3, n_voice=12, n_noise=4, bg_seconds=4.0)


def _chain(ds, n_frame_batch=4, n_mels=80):
    from challenge_b200 import data_utils as D, transforms as TR
    return (ds.map(D.to_frame_labels).map(D.augment).batch(n_frame_batch).map(TR.complex_to_magphase)
            .map(TR.magphase_to_mel(n_mels)).map(D.minmax).map(D.log_on_mel))


def test_two_live_pipelines_keep_their_own_banks():
    """The reference builds the train and the test dataset before training (sj_train.py:472-473) and
    iterates both.  Every pipeline owns its bank set: interleaved iteration gives what each pipeline
    gives alone with the same seed."""
    import torch
    from challenge_b200 import _ops as O
    from challenge_b200.pipeline import make_pipeline

    def build(seed):
        bgs, voices, labels, noises = _banks(seed)
        return _chain(make_pipeline(bgs, voices, labels, noises, n_frame=120, max_voices=4, max_noises=2,
                                    min_ratio=1))

    def alone(seed, n):
        O.set_seed(1000 + seed)
        return [(x.clone(), y.clone()) for x, y in build(seed).take(n)]

    a_ref, b_ref = alone(1, 3), alone(2, 3)
    # interleaved: both pipelines alive; each consumes its own seeded draw sequence
    O.set_seed(1001)
    pa = build(1)
    ia = iter(pa)
    got_a = [next(ia)]
    state_a = O.rng()
    O.set_seed(1002)
    pb = build(2)                   # registers the second bank set while the first is live
    ib = iter(pb)
    got_b = [next(ib)]
    state_b = O.rng()
    for _ in range(2):
        O._rng = state_a
        got_a.append(next(ia))
        O._rng = state_b
        got_b.append(next(ib))
    for (x, y), (rx, ry) in zip(got_a, a_ref):
        assert torch.equal(x, rx) and torch.equal(y, ry)
    for (x, y), (rx, ry) in zip(got_b, b_ref):
        assert torch.equal(x, rx) and torch.equal(y, ry)
    assert pa.engine is not pb.engine


def test_take_counts_elements_before_batch_and_batches_after():
    """tf.data: take(n) before batch() limits ELEMENTS (the last batch is partial unless
    drop_remainder), after batch() it limits batches."""
    from challenge_b200 import data_utils as D
    from challenge_b200.pipeline import make_pipeline
    bgs, voices, labels, noises = _banks(3)
    ds = make_pipeline(bgs, voices, labels, noises, n_frame=100, max_voices=3, max_noises=2, min_ratio=1)
    sizes = [x.shape[0] for x, _ in ds.map(D.to_frame_labels).take(5).batch(2)]
    assert sizes == [2, 2, 1]
    sizes = [x.shape[0] for x, _ in ds.map(D.to_frame_labels).take(5).batch(2, drop_remainder=True)]
    assert sizes == [2, 2]
    sizes = [x.shape[0] for x, _ in ds.map(D.to_frame_labels).batch(2).take(3)]
    assert sizes == [2, 2, 2]
    x, y = next(iter(ds.take(1)))
    assert x.shape == (257, 100, 4) and y.shape == (3, 100, 3)


def test_wide_mel_filters_fall_back_to_the_unfused_projection():
    """n_mels = 20: the longest filter of tf.signal.linear_to_mel_weight_matrix(20, 257, 16000) spans
    21 bins, more than the fused epilogue takes.  The chain still works: the fused kernel stops at
    magnitude + phase and magphase_to_mel runs as the stand-alone kernel (values vs the oracle)."""
    from challenge_b200 import _ops as O
    from challenge_b200.pipeline import make_pipeline
    from oracle import transforms as OT, data_utils as OD
    bgs, voices, labels, noises = _banks(4)
    ds = make_pipeline(bgs, voices, labels, noises, n_frame=100, max_voices=3, max_noises=2, min_ratio=1)
    O.set_seed(7)
    x, y = next(iter(_chain(ds, 3, n_mels=20)))
    assert x.shape == (3, 20, 100, 2) and not ds.engine.mel_fusable()
    # the same draws through the fused complex path, then the oracle's own mel / minmax / log
    from challenge_b200 import data_utils as D
    O.set_seed(7)    # a fresh pipeline: the shuffle streams of `ds` have advanced
    ds2 = make_pipeline(bgs, voices, labels, noises, n_frame=100, max_voices=3, max_noises=2, min_ratio=1)
    c, y2 = next(iter(ds2.map(D.to_frame_labels).map(D.augment).batch(3)))
    mp = OT.complex_to_magphase(c.cpu().numpy())
    ref = OD.log_on_mel(OD.minmax(OT.magphase_to_mel(20)(mp)))
    assert nmax_err(x.cpu().numpy(), ref) < TOL
    assert np.array_equal(y.cpu().numpy(), y2.cpu().numpy())


def test_too_many_mixing_segments_is_refused_at_make_pipeline():
    from challenge_b200.pipeline import make_pipeline
    from challenge_b200.synth import synthetic_banks
    bgs, voices, labels, noises = synthetic_banks(5, 2, n_bg=2, n_voice=30, n_noise=12, bg_seconds=0.5)
    with pytest.raises(ValueError, match='segments'):
        make_pipeline(bgs, voices, labels, noises, n_frame=626, max_voices=10, max_noises=10)
    # the legacy trainer defaults on full-length backgrounds are fine
    bgs, _, _, _ = synthetic_banks(5, 2, n_bg=2, n_voice=1, n_noise=1, bg_seconds=10.0)
    make_pipeline(bgs, voices, labels, noises, n_frame=300, max_voices=10, max_noises=10, min_ratio=1)


def test_numa_local_pinned_allocation(engine):
    import torch
    a, node = engine.host_alloc((1 << 20,), np.float32)
    assert a.shape == (1 << 20,) and node >= -1
    t = torch.from_numpy(a)
    src = torch.arange(1 << 20, dtype=torch.float32, device='cuda')
    t.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    assert a[12345] == 12345.0


def test_nccl_count_allreduce_two_ranks():
    """SURVEY.md 8e on real GPUs: two ranks, NCCL inside libiris (iris_allreduce_counts) --
    runs tests/nccl_worker.py under torch.distributed.run; skipped on a one-GPU box."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
                        '--master-addr', '127.0.0.1', '--master-port', '29533',
                        os.path.join(root, 'tests', 'nccl_worker.py')], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert 'NCCL_WORKER_OK' in r.stdout


def test_tile_lists_built_by_k_labels_match_k_tiles(engine, workload_factory, monkeypatch):
    """k_labels builds the per-tile stage lists of the feature launch it is told about (the mode of
    the previous feature launch, or iris_step's mode); a feature launch with another layout -- another
    mode family, only_voice / only_noise, another plan -- must notice and run k_tiles.  Every order
    of calls gives the bits of the plain labels -> k_tiles -> k_fused path."""
    from challenge_b200 import _lib as L
    from challenge_b200.plan import draw_batch
    engine.set_mel(80)
    w = workload_factory(2)
    plans = [draw_batch(np.random.default_rng(s), 5, 300, w.bg_frames, w.voice_frames, w.noise_frames, max_voices=5,
                        max_noises=2, snr=-20, min_ratio=2 / 3, n_time_masks=6, n_freq_masks=1) for s in (1, 2)]
    modes = [L.FEAT_LOGMEL_MINMAX, L.FEAT_COMPLEX, L.FEAT_MEL, L.FEAT_MAGPHASE, L.FEAT_LOGMEL]
    monkeypatch.setenv('IRIS_NO_LABEL_TILES', '1')
    ref = {}
    for i, d in enumerate(plans):
        engine.upload_plan(d)
        engine.labels()
        for m in modes:
            ref[i, m] = engine.features(m).clone()
        ref[i, 'voice'] = engine.features(L.FEAT_COMPLEX, select=L.SELECT_VOICES).clone()
    monkeypatch.delenv('IRIS_NO_LABEL_TILES')
    order = [(0, modes[0]), (0, modes[1]), (1, modes[1]), (1, modes[0]), (0, modes[3]), (0, modes[2]), (1, modes[4]),
             (1, modes[4]), (0, modes[0]), (0, modes[0])]
    for i, m in order:
        engine.upload_plan(plans[i])
        engine.labels()                       # hinted with the mode of the previous feature launch
        got = engine.features(m)
        assert torch_equal(got, ref[i, m]), (i, m)
        # another segment selection between two launches of one mode
        assert torch_equal(engine.features(L.FEAT_COMPLEX, select=L.SELECT_VOICES), ref[i, 'voice'])
        assert torch_equal(engine.features(m), ref[i, m]), (i, m, 'second launch on cached tile lists')


def torch_equal(a, b):
    import torch
    return bool(torch.equal(a, b))
