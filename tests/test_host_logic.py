"""CPU tests of the host side: draws, placement arithmetic, the C-ABI library (loads,
exports every symbol include/iris.h declares, fails loudly without a GPU), the FFT core's
math compiled for the host, and the product never importing the oracle."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_draw_ranges_follow_reference():
    from challenge_b200.plan import draw_batch, placement
    rng = np.random.default_rng(0)
    bf = np.array([626, 300, 40])
    vf = rng.integers(32, 251, 50)
    nf = rng.integers(32, 251, 20)
    T, V, M = 626, 7, 2
    d = draw_batch(rng, 500, T, bf, vf, nf, V, M, snr=-20, min_ratio=1, n_time_masks=6,
                   n_freq_masks=1, merge_extra=2)
    bgT = bf[d.bg_id]
    tiled = bgT * ((T + bgT - 1) // bgT)
    assert np.all((d.bg_offset >= 0) & (d.bg_offset <= tiled - T))          # pipeline.py:35
    assert np.all((d.n_voices >= 1) & (d.n_voices < V))                      # :43
    assert np.all((d.n_noises >= 0) & (d.n_noises < M))                      # :87
    assert np.all((d.voice_u >= 0) & (d.voice_u < 2)) and d.voice_u.dtype == np.float32
    # gain = pow(10., -u) (pipeline.py:50) from libm's powf; numpy's float32 power may differ in the last bit
    np.testing.assert_array_max_ulp(d.voice_gain, np.power(np.float32(10), -d.voice_u, dtype=np.float32), maxulp=1)
    for b in range(500):
        vP = vf[d.voice_id[b]].max()
        pad, length = placement(T, vP, 1)
        assert pad == T - vP and length == vP + 2 * pad
        assert np.all(d.voice_offset[b, :d.n_voices[b]] < length - T)         # :69
        nP = nf[d.noise_id[b]].max()
        _, nlen = placement(T, nP, 0.5)
        assert np.all(d.noise_offset[b, :d.n_noises[b]] <= nlen - T)          # :103
    size, off = d.time_masks[..., 0], d.time_masks[..., 1]
    assert np.all((size >= 0) & (size < 24) & (off >= 0) & (off < T - size))  # transforms.py:25-26
    size, off = d.freq_masks[..., 0], d.freq_masks[..., 1]
    assert np.all((size >= 0) & (size < 16) & (off >= 0) & (off < 257 - size))
    assert np.all((d.merge_factor >= 0.1) & (d.merge_factor < 0.9))           # data_utils.py:109
    s = d.slice(100, 164)
    assert s.batch == 64 and np.array_equal(s.voice_id, d.voice_id[100:164])


def test_placement_truncates_in_float32():
    from challenge_b200.plan import placement
    # 2/3 * 100 = 66.67 -> int32 66 ; pad = 34
    assert placement(100, 100, 2 / 3) == (34, 168)
    assert placement(626, 626, 1) == (0, 626)
    assert placement(10, 30, 0.5) == (0, 30)


def test_empty_offset_range_raises_in_planner():
    from challenge_b200.errors import InvalidArgumentError
    from challenge_b200.plan import draw_batch
    with pytest.raises(InvalidArgumentError):
        draw_batch(np.random.default_rng(0), 2, 100, np.array([100]), np.array([100, 50]),
                   None, max_voices=2, min_ratio=1)


def test_shuffle_stream_visits_everything():
    from challenge_b200.plan import ShuffleStream
    s = ShuffleStream(10, np.random.default_rng(0))
    ids = s.take(1000)
    assert set(ids.tolist()) == set(range(10))
    # repeat().shuffle(n): over a long run every id appears about equally often
    assert np.bincount(ids, minlength=10).min() > 60


def _planner_case(rng, V, M, ntm, nfm, me, B=64, T=626, with_streams=False, min_ratio=1.0):
    from challenge_b200.plan import ShuffleStream, draw_config, draws_from_uniforms, uniforms_per_clip
    from oracle import plan as OP
    bgf = rng.integers(30, 700, 9).astype(np.int32)
    vf = rng.integers(T // 2 + 1 if min_ratio < 1 else 8, 250, 23).astype(np.int32)
    nf = rng.integers(8, 250, 11).astype(np.int32)
    cfg = draw_config(B, T, V, M, -20, min_ratio, 0.5, ntm, 24, nfm, 16, 257, me)
    u = rng.random((B, uniforms_per_clip(cfg)))
    st_c = st_p = None
    if with_streams:
        st_c = {'bg': ShuffleStream(len(bgf), rng), 'voice': ShuffleStream(len(vf), rng),
                'noise': ShuffleStream(len(nf), rng, 5)}
        st_p = {'bg': OP.ShuffleStreamPy(len(bgf)), 'voice': OP.ShuffleStreamPy(len(vf)),
                'noise': OP.ShuffleStreamPy(len(nf), 5)}
    d = draws_from_uniforms(cfg, u, bgf, vf if V else None, nf if M else None, st_c)
    r = OP.draws_from_uniforms(u, T, bgf, vf, nf, V, M, -20, min_ratio, 0.5, ntm, 24, nfm, 16, 257, me, st_p)
    return d, r


@pytest.mark.parametrize('with_streams', [False, True])
@pytest.mark.parametrize('V,M,ntm,nfm,me', [(7, 2, 6, 1, 0), (1, 1, 0, 0, 2), (0, 0, 2, 0, 0),
                                             (4, 0, 0, 1, 3), (10, 6, 6, 1, 0), (2, 1, 1, 1, 1)])
def test_c_planner_is_bit_identical_to_the_numpy_restatement(V, M, ntm, nfm, me, with_streams):
    """iris_draw_batch (the planner iris_step runs) against oracle/plan.py on the same block of
    uniforms: every integer draw and every fp32 exponent draw identical; the gains
    pow(10., -u) (pipeline.py:50, 94) agree to the last bit or one ulp (libm vs numpy)."""
    d, r = _planner_case(np.random.default_rng(100 * V + M), V, M, ntm, nfm, me, with_streams=with_streams)
    assert set(r) <= {f for f in vars(d) if getattr(d, f) is not None}
    for k, v in r.items():
        a = getattr(d, k)
        assert a.dtype == v.dtype and a.shape == v.shape, k
        if k.endswith('_gain'):
            np.testing.assert_array_max_ulp(a, v, maxulp=1)
        else:
            assert np.array_equal(a, v), k


def test_planner_fuzz_edge_cases():
    """hypothesis fuzz of the planner's edge cases: V = 1 (n_voices fixed at 1, pipeline.py:41-46),
    M in {0, 1} (n_noises in [0, M) is always 0 for M = 1), backgrounds shorter than n_frame (tiled,
    pipeline.py:29-35), uniforms at the ends of [0, 1)."""
    from hypothesis import given, settings, strategies as st
    from challenge_b200.plan import draw_config, draws_from_uniforms, uniforms_per_clip
    from oracle import plan as OP

    @settings(max_examples=60, deadline=None)
    @given(st.integers(0, 3), st.integers(0, 2), st.integers(20, 400), st.integers(0, 2 ** 31 - 1),
           st.sampled_from([0.0, 0.5, 1.0 - 2.0 ** -53]))
    def run(V, M, T, seed, edge):
        rng = np.random.default_rng(seed)
        bgf = rng.integers(5, 2 * T, 4).astype(np.int32)       # some shorter than T: tiled
        vf = rng.integers(T + 1, 2 * T + 2, 6).astype(np.int32)  # min_ratio 1: len - T >= 1
        nf = rng.integers(3, 2 * T, 5).astype(np.int32)
        B = 5
        cfg = draw_config(B, T, V, M, -20, 1.0, 0.5, 2, 24 if T > 24 else T, 1, 16, 257, 1)
        u = rng.random((B, uniforms_per_clip(cfg)))
        u[0, :] = edge
        d = draws_from_uniforms(cfg, u, bgf, vf if V else None, nf if M else None)
        r = OP.draws_from_uniforms(u, T, bgf, vf, nf, V, M, -20, 1.0, 0.5, 2, cfg.time_mask_max, 1, 16, 257, 1)
        for k, v in r.items():
            a = getattr(d, k)
            if k.endswith('_gain'):
                np.testing.assert_array_max_ulp(a, v, maxulp=1)
            else:
                assert np.array_equal(a, v), k
        if V == 1:
            assert np.all(d.n_voices == 1)
        if M == 1:
            assert np.all(d.n_noises == 0)
        bgT = bgf[d.bg_id].astype(np.int64)
        assert np.all(d.bg_offset <= bgT * ((T + bgT - 1) // bgT) - T)
    run()


def test_planner_raises_where_the_reference_raises():
    """len == n_frame leaves the empty range [0, 0) for the voice offset: tf.random.uniform raises
    (pipeline.py:68-69) -> IRIS_ERR_EMPTY_RANGE -> InvalidArgumentError."""
    from challenge_b200.errors import InvalidArgumentError
    from challenge_b200.plan import draw_config, draws_from_uniforms, uniforms_per_clip
    cfg = draw_config(2, 100, 2, 0, -20, 1.0, 0.5)
    u = np.random.default_rng(0).random((2, uniforms_per_clip(cfg)))
    with pytest.raises(InvalidArgumentError):
        draws_from_uniforms(cfg, u, np.array([100]), np.array([100, 50]))
    draws_from_uniforms(cfg, u, np.array([100]), np.array([101, 50]))   # len - T = 1: fine


def _header_symbols():
    text = open(os.path.join(ROOT, 'include', 'iris.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(iris_[a-z0-9_]+)\s*\(', text)))


def test_library_loads_and_exports_every_declared_symbol():
    from challenge_b200 import _lib
    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 26
    assert sorted(_lib.SIGNATURES) == syms, 'include/iris.h and the ctypes binding differ'
    for name in syms:
        assert hasattr(lib, name), 'libiris.so does not export %s' % name
        assert name in _lib.SIGNATURES, 'no ctypes signature for %s' % name
    assert lib.iris_abi_version() == 2


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from challenge_b200 import _lib
    lib = _lib.load()
    ctx = ctypes.c_void_p()
    rc = lib.iris_ctx_create(0, ctypes.byref(ctx))
    assert rc == _lib.IRIS_ERR_CUDA and b'no CPU fallback' in lib.iris_last_error()
    from challenge_b200.engine import Engine
    with pytest.raises(Exception):
        Engine(0)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'challenge_b200')
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', src, flags=re.M), f


def test_native_environment_switches_are_the_documented_ones():
    """Every getenv of the native library is a switch INTEGRATION.md section 6 documents; the
    product path takes no other run-time option."""
    csrc = os.path.join(ROOT, 'challenge_b200', 'csrc')
    names = set()
    for f in os.listdir(csrc):
        names |= set(re.findall(r'getenv\(\s*"([^"]+)"\s*\)', open(os.path.join(csrc, f)).read()))
    assert names == {'IRIS_NCCL_LIB', 'IRIS_NO_FIXED_EPI', 'IRIS_NO_LABEL_TILES'}
    doc = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    section = re.search(r'^## 6\..*?(?=^## |\Z)', doc, flags=re.M | re.S).group(0)
    for n in names:
        assert '`%s' % n in section, n


def test_fftcore_math_on_host(tmp_path):
    """fftcore.cuh compiled with g++: the 16-lane x 32-point decomposition, the 4-round
    exchange geometry and the lane-local two-channel split reproduce a float64 DFT."""
    exe = str(tmp_path / 'fftcore_host')
    subprocess.check_call(['g++', '-std=c++17', '-O2', '-x', 'c++', '-I',
                           os.path.join(ROOT, 'challenge_b200', 'csrc'),
                           os.path.join(ROOT, 'tests', 'host', 'fftcore_host.cpp'), '-o', exe])
    r = json.loads(subprocess.check_output([exe]).decode())
    assert r['bad_seen'] == 0
    assert r['err_small'] < 2e-6
    assert r['err512'] / r['max_abs'] < 1e-6
    assert r['im_dc'] == 0.0 and r['im_nyq'] == 0.0


def test_fftwarp_math_on_host(tmp_path):
    """fftwarp.cuh (the warp-per-frame FFT of the fused kernel) compiled with g++: 32 emulated
    lanes, the exchange offsets, the DIF + partner/mirror maps and the two-channel split
    reproduce a float64 windowed DFT; bins < 128 need only half of pass 2's outputs."""
    exe = str(tmp_path / 'fftwarp_host')
    subprocess.check_call(['g++', '-std=c++17', '-O2', '-x', 'c++', '-I',
                           os.path.join(ROOT, 'challenge_b200', 'csrc'),
                           os.path.join(ROOT, 'tests', 'host', 'fftwarp_host.cpp'), '-o', exe])
    r = json.loads(subprocess.check_output([exe]).decode())
    assert r['bad_map'] == 0 and r['missing'] == 0 and r['bad_prune'] == 0
    assert r['err512'] / r['max_abs'] < 1e-6
    assert r['im_dc'] == 0.0 and r['im_nyq'] == 0.0


def test_default_mel_matrix_is_the_tf_restatement():
    from challenge_b200.engine import default_mel_matrix
    from oracle.transforms import linear_to_mel_weight_matrix
    assert np.array_equal(default_mel_matrix(80), linear_to_mel_weight_matrix(80, 257, 16000))
    # the product's matrix against the independent float64 golden (not only against the oracle's copy
    # of the same restatement): tests/golden/mel_matrix_80.json, scripts/make_mel_golden.py
    import json
    g = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'mel_matrix_80.json')))
    w = default_mel_matrix(80)
    assert (w != 0).sum() == g['nnz'] and (w != 0).sum(0).tolist() == g['taps_per_column']
    assert np.abs(w.sum(0) - np.array(g['column_sums'])).max() < 4e-5
    assert max(abs(float(w[f, j]) - v) for f, j, v in g["entries"]) < 2e-5
    assert np.array_equal(default_mel_matrix(40, lower_edge_hertz=80.0, upper_edge_hertz=7600.0),
                          linear_to_mel_weight_matrix(40, 257, 16000, 80.0, 7600.0))


def test_dropin_modules_mirror_the_reference_surface():
    """Every public function of the reference's hot-path modules exists under the same name
    (SURVEY.md 8b); importing the modules needs neither a GPU nor the oracle."""
    from challenge_b200 import data_utils, metrics, pipeline, transforms
    want = {
        pipeline: ['merge_complex_specs', 'make_pipeline'],
        transforms: ['mask', 'random_shift', 'magphase_to_mel', 'log_magphase',
                     'minmax_norm_magphase', 'complex_to_magphase', 'magphase_to_complex',
                     'phase_vocoder', 'EPSILON'],
        data_utils: ['load_wav', 'normalize', 'minmax', 'log_on_mel', 'augment', 'to_frame_labels',
                     'mono_chan', 'stereo_mono', 'label_downsample', 'random_merge_aug',
                     'multiply_label', 'stft_filter', 'speech_enhancement_preprocess'],
        metrics: ['er_score', 'f1_score', 'cos_sim'],
    }
    for mod, names in want.items():
        for n in names:
            assert hasattr(mod, n), '%s.%s missing' % (mod.__name__, n)


def test_dataset_lowering_recognises_the_sj_train_chain():
    """sj_train.make_dataset's stage order (sj_train.py:107-123) lowers to one fused launch."""
    from challenge_b200 import _lib as L
    from challenge_b200 import data_utils as D, transforms as TR
    from challenge_b200.pipeline import IrisDataset
    ds = IrisDataset({})
    ds = ds.map(D.to_frame_labels).map(D.augment).map(D.stft_filter(3)).batch(12)
    ds = ds.map(TR.complex_to_magphase).map(TR.magphase_to_mel(80)).map(D.minmax).map(D.log_on_mel)
    fused, rest = ds.prefetch(-1)._lower()
    assert rest == [] and fused['mode'] == L.FEAT_LOGMEL_MINMAX and fused['augment']
    assert fused['frame_labels'] and fused['filt'] == 3 and fused['n_mels'] == 80
    # 'nominmax' variant (sj_train.py:121) and a stage the fused kernel does not absorb
    ds = IrisDataset({}).map(D.to_frame_labels).batch(4).map(TR.complex_to_magphase)
    ds = ds.map(TR.magphase_to_mel(40)).map(D.log_on_mel).map(D.label_downsample(32))
    fused, rest = ds._lower()
    assert fused['mode'] == L.FEAT_LOGMEL and fused['n_mels'] == 40 and len(rest) == 1
    # out-of-order stages stay un-fused and keep their order
    ds = IrisDataset({}).map(D.augment).map(D.to_frame_labels).batch(2)
    fused, rest = ds._lower()
    assert fused['augment'] and not fused['frame_labels'] and len(rest) == 2


def test_resample_len_matches_the_kaldi_port_without_a_gpu():
    """iris_resample_len is host arithmetic (no device needed): it must agree with the oracle's
    restatement of kaldi.py::_get_num_LR_output_samples for every rate pair / length."""
    from challenge_b200 import _lib
    from oracle.data_utils import _lr_num_output_samples
    lib = _lib.load()
    rng = np.random.default_rng(3)
    for orig, new in ((44100, 16000), (48000, 16000), (8000, 16000), (22050, 16000), (11025, 16000),
                      (32000, 16000), (16000, 16000), (96000, 16000), (16000, 8000)):
        for n in [1, 2, 255, 256, 441, 16000, 44100, 160000] + [int(v) for v in rng.integers(1, 500000, 20)]:
            assert lib.iris_resample_len(n, orig, new) == _lr_num_output_samples(n, orig, new), (orig, new, n)
    assert lib.iris_resample_len(0, 44100, 16000) == 0


def test_numa_binding_is_a_no_op_without_nvml():
    """dist.bind_to_gpu_numa never raises: without a GPU / NVML it leaves the affinity alone."""
    from challenge_b200.dist import bind_to_gpu_numa
    before = os.sched_getaffinity(0)
    cores = bind_to_gpu_numa(0)
    assert cores is None or set(cores) <= before
    if cores is None:
        assert os.sched_getaffinity(0) == before
    else:
        os.sched_setaffinity(0, before)


def test_default_mel_matrix_has_the_shape_the_fixed_kernel_instances_assume():
    """k_fused<FM_MEL, 4, EPI_C2 | ...> unrolls the projection for filters of at most 2 / 4 / 6 bins
    in the three rounds of 32 and bins below 128 (fixed_mel_L in k_fused.cu; the launcher checks the
    same and falls back to the generic instance otherwise).  The reference's matrix
    (transforms.py:55, linear_to_mel_weight_matrix(80, 257, 16000)) has exactly that shape."""
    from oracle.transforms import linear_to_mel_weight_matrix
    W = linear_to_mel_weight_matrix(80, 257, 16000)
    lens, hi = [], 0
    for m in range(80):
        nz = np.nonzero(W[:, m])[0]
        assert np.all(np.diff(nz) == 1)                      # contiguous support
        lens.append(len(nz))
        hi = max(hi, int(nz[-1]))
    rounds = [max(lens[32 * r:32 * r + 32]) for r in range(3)]
    assert [n + (n & 1) for n in rounds] == [2, 4, 6] and hi < 128
    src = open(os.path.join(ROOT, 'challenge_b200', 'csrc', 'k_fused.cu')).read()
    assert 'return r == 0 ? 2 : (r == 1 ? 4 : (r == 2 ? 6 : 0));' in src


def test_work_claim_schedule_covers_every_tile_once():
    """k_fused hands its tiles out in claims that shrink towards the end of a launch (whole chunks, half
    chunks, single tiles; pairs of tiles for 4-channel clips whose two channel pairs share a store
    phase).  For any tile count / grid / chunk the claims 0, 1, 2, ... must tile [0, n_tiles) exactly
    once, in order, and -- with merged pairs -- start on even tiles with even lengths."""
    from challenge_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(5)
    cases = [(20224, 296, 6, 0), (2528, 296, 6, 0), (1, 296, 6, 0), (5, 1, 4, 0), (40448, 296, 6, 1),
             (2, 296, 6, 1), (647168, 296, 6, 0), (79, 296, 1, 0), (158, 64, 2, 1)]
    cases += [(int(rng.integers(1, 5000)) * 1, int(rng.integers(1, 400)), int(rng.integers(1, 17)), 0) for _ in range(40)]
    cases += [(int(rng.integers(1, 2500)) * 2, int(rng.integers(1, 400)), int(rng.integers(1, 17)), 1) for _ in range(40)]
    sched = (ctypes.c_int32 * 5)()
    first, ln = ctypes.c_int64(), ctypes.c_int32()
    for n_tiles, grid, chunk, merge in cases:
        nxt, q = 0, 0
        while True:
            assert lib.iris_debug_claims(n_tiles, grid, chunk, merge, q, sched, ctypes.byref(first), ctypes.byref(ln)) == 0
            if first.value >= n_tiles:
                break
            assert first.value == nxt, (n_tiles, grid, chunk, merge, q)
            assert ln.value >= 1
            if merge:
                assert first.value % 2 == 0 and ln.value % 2 == 0
            nxt = min(n_tiles, first.value + ln.value)
            q += 1
            assert q <= n_tiles + 1
        assert nxt == n_tiles, (n_tiles, grid, chunk, merge)
        ch, mid, tail, n_big, n_mid = list(sched)
        assert tail <= mid <= ch
        if n_tiles > grid * 8 and ch > (2 if merge else 1):    # a long launch ends on single tiles (tile pairs)
            assert tail == (2 if merge else 1) and n_big > 0
