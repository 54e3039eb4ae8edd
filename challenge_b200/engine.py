"""Per-device engine: owns an ``iris_ctx`` and exposes the C ABI with torch tensors for
device memory and streams (plumbing only -- every kernel is in libiris.so)."""
import ctypes as C

import numpy as np

from . import _lib as L
from .plan import BatchDraws


def _torch():
    import torch
    return torch


def out_flag(dtype):
    """IRIS_OUT_* flag of a feature dtype: 0 for torch.float32, OUT_BF16 / OUT_F16 for torch.bfloat16 /
    torch.float16 (or their names).  Any other dtype raises ValueError."""
    torch = _torch()
    if isinstance(dtype, str):
        dtype = getattr(torch, dtype, None) if dtype in ('float32', 'bfloat16', 'float16') else None
    flags = {torch.float32: 0, torch.bfloat16: L.OUT_BF16, torch.float16: L.OUT_F16}
    if dtype not in flags:
        raise ValueError('features are float32, bfloat16 or float16, not %r' % (dtype,))
    return flags[dtype]


def out_dtype(mode):
    """torch dtype of the features of a mode with or without an IRIS_OUT_* flag."""
    torch = _torch()
    dtypes = {0: torch.float32, L.OUT_BF16: torch.bfloat16, L.OUT_F16: torch.float16}
    flag = int(mode) & ~L.MODE_MASK
    if flag not in dtypes:
        raise ValueError('feature mode 0x%x: at most one of OUT_BF16 / OUT_F16 above the mode' % int(mode))
    return dtypes[flag]


def default_mel_matrix(num_mel_bins=80, num_spectrogram_bins=257, sample_rate=16000,
                       lower_edge_hertz=125.0, upper_edge_hertz=3800.0):
    """``tf.signal.linear_to_mel_weight_matrix`` (called at transforms.py:55-56), rebuilt
    op-for-op in float32 in TF 2.2's order: HTK mel ``1127*ln(1+f/700)``, linspace as
    ``start + step*i``, triangles in the mel domain, DC row zero."""
    f32 = np.float32

    def linspace(start, stop, num):
        start, stop = f32(start), f32(stop)
        step = f32((stop - start) / f32(num - 1))
        return (start + step * np.arange(num, dtype=np.float32)).astype(np.float32)

    def h2m(f):
        return (f32(1127.0) * np.log(f32(1.0) + np.asarray(f, np.float32) / f32(700.0))
                ).astype(np.float32)

    lin = linspace(0.0, f32(sample_rate) / f32(2.0), num_spectrogram_bins)[1:]
    spec_mel = h2m(lin)[:, None]
    edges = linspace(h2m(f32(lower_edge_hertz)), h2m(f32(upper_edge_hertz)), num_mel_bins + 2)
    lower, center, upper = edges[None, :-2], edges[None, 1:-1], edges[None, 2:]
    w = np.maximum(f32(0), np.minimum((spec_mel - lower) / (center - lower),
                                      (upper - spec_mel) / (upper - center)))
    return np.pad(w.astype(np.float32), [[1, 0], [0, 0]])


def bank_item(item):
    """One waveform-bank item -> (float32 ``[C, N]`` array, sample rate): ``(waveform, sample_rate)``, the
    in-memory form ``load_wav`` takes, or a plain array, which is 16 kHz audio."""
    if isinstance(item, tuple):
        wav, rate = item
        return np.ascontiguousarray(wav, np.float32), int(rate)
    return np.ascontiguousarray(item, np.float32), 16000


def is_spec_bank(items):
    """Whether bank ``items`` are spectrograms ``[257, t, 2C]`` rather than waveforms (arrays ``[C, N]`` or
    ``(waveform, sample_rate)`` tuples)."""
    return not isinstance(items[0], tuple) and np.asarray(items[0]).ndim == 3


def pack_waveforms(items):
    """Waveform-bank items (see :func:`bank_item`) -> (packed float32 samples, offsets int64 ``[n + 1]`` of the
    per-channel sample counts at each item's own rate, sample rates int32 ``[n]``, channels): the arguments
    of ``iris_bank_register(_audio)``."""
    waves, rates = zip(*(bank_item(x) for x in items))
    n_chan = waves[0].shape[0]
    assert all(w.ndim == 2 and w.shape[0] == n_chan for w in waves), \
        'each waveform must be [chan, samples]'
    offsets = np.zeros(len(waves) + 1, np.int64)
    offsets[1:] = np.cumsum([w.shape[1] for w in waves])
    packed = np.concatenate([w.reshape(-1) for w in waves])
    return packed, offsets, np.asarray(rates, np.int32), n_chan


class Engine:
    """One engine (= one ``iris_ctx``) per CUDA device."""

    def __init__(self, device=0):
        torch = _torch()
        self.lib = L.load()
        if not torch.cuda.is_available():
            raise L.IrisError('no CUDA device visible: libiris has no CPU fallback')
        self.device = torch.device('cuda', int(device))
        self._ctx = C.c_void_p()
        L.check(self.lib.iris_ctx_create(int(device), C.byref(self._ctx)))
        self.n_mel = 0
        self.mel_matrix = None
        self.bank_frames = {}
        self.bank_chan = None
        self.n_classes = 0
        self._plan = None

    def close(self):
        for p, n in getattr(self, '_host_allocs', []):
            self.lib.iris_host_free(self._ctx, p, n)
        self._host_allocs = []
        if self._ctx:
            self.lib.iris_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers ----
    def _stream(self):
        torch = _torch()
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _empty(self, shape, dtype=None):
        torch = _torch()
        return torch.empty(shape, dtype=dtype or torch.float32, device=self.device)

    @staticmethod
    def _ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    # ---- configuration ----
    def set_mel(self, num_mel_bins=80, num_spectrogram_bins=257, sample_rate=16000,
                mel_matrix=None, **kwargs):
        w = mel_matrix if mel_matrix is not None else default_mel_matrix(
            num_mel_bins, num_spectrogram_bins, sample_rate, **kwargs)
        w = np.ascontiguousarray(w, np.float32)
        L.check(self.lib.iris_set_mel(self._ctx, w.shape[1], w.shape[0], w.ctypes.data))
        self.n_mel = w.shape[1]
        self.mel_matrix = w

    def register_spec_bank(self, kind, specs, labels=None):
        """``specs``: list of pre-computed complex spectrograms ``[257, t_i, 2*chan]`` -- the
        reference's own bank format (``utils.load_data`` pickles, consumed by
        pipeline.py:113-175).  Mixed in the spectrogram domain (k_spec.cu)."""
        items = [np.ascontiguousarray(x, np.float32) for x in specs]
        F, W = items[0].shape[0], items[0].shape[2]
        assert all(x.ndim == 3 and x.shape[0] == F and x.shape[2] == W for x in items), \
            'each spec must be a 3D-tensor [freq, time, chan*2]'
        offsets = np.zeros(len(items) + 1, np.int64)
        offsets[1:] = np.cumsum([x.shape[1] for x in items])
        packed = np.concatenate([x.reshape(-1) for x in items])
        lab, n_classes = None, 0
        if labels is not None:
            lab = np.ascontiguousarray(labels, np.float32)
            assert lab.shape[0] == len(items)
            n_classes = lab.shape[1]
        L.check(self.lib.iris_specbank_register(
            self._ctx, kind, len(items), F, W, packed.ctypes.data, offsets.ctypes.data,
            lab.ctypes.data if lab is not None else None, n_classes, self._stream()))
        frames = np.zeros(len(items), np.int32)
        L.check(self.lib.iris_bank_info(self._ctx, kind, None, None, frames.ctypes.data))
        self.bank_frames[kind] = frames
        self.bank_chan = W // 2
        if kind == L.BANK_VOICE:
            self.n_classes = n_classes
        return frames

    def register_bank(self, kind, waveforms, labels=None, normalize=True):
        """``waveforms``: list of float32 ``[C, N_i]`` arrays of 16 kHz audio or ``(waveform, sample_rate)``
        tuples at any rate, mixed freely (the audio load_wav reads, data_utils.py:19-22; items not at 16 kHz
        are resampled on the device with load_wav's filter), or spectrograms ``[257, t, 2C]``
        (:meth:`register_spec_bank`).  ``labels``: ``[n_items, K]`` one-hot rows (voice bank)."""
        if is_spec_bank(waveforms):
            return self.register_spec_bank(kind, waveforms, labels=labels)
        packed, offsets, rates, n_chan = pack_waveforms(waveforms)
        n = len(rates)
        lab = None
        n_classes = 0
        if labels is not None:
            lab = np.ascontiguousarray(labels, np.float32)
            assert lab.shape[0] == n
            n_classes = lab.shape[1]
        lab_p = lab.ctypes.data if lab is not None else None
        if (rates == 16000).all():
            L.check(self.lib.iris_bank_register(
                self._ctx, kind, n, n_chan, packed.ctypes.data, offsets.ctypes.data, lab_p, n_classes,
                int(bool(normalize)), self._stream()))
        else:
            if not hasattr(self.lib, 'iris_bank_register_audio'):
                raise NotImplementedError('this libiris predates iris_bank_register_audio: resample the items '
                                          'to 16 kHz first')
            L.check(self.lib.iris_bank_register_audio(
                self._ctx, kind, n, n_chan, packed.ctypes.data, offsets.ctypes.data, rates.ctypes.data, lab_p,
                n_classes, int(bool(normalize)), self._stream()))
        frames = np.zeros(n, np.int32)
        L.check(self.lib.iris_bank_info(self._ctx, kind, None, None, frames.ctypes.data))
        self.bank_frames[kind] = frames
        self.bank_chan = n_chan
        if kind == L.BANK_VOICE:
            self.n_classes = n_classes
        return frames

    def voice_activity(self, item):
        n = int(self.bank_frames[L.BANK_VOICE][item])
        out = np.zeros(n, np.uint8)
        L.check(self.lib.iris_bank_activity(self._ctx, int(item), out.ctypes.data))
        return out

    # ---- per-step ----
    def upload_plan(self, d: BatchDraws, stft_filter=0, chan_remap=L.REMAP_NONE, n_out_chan=0):
        def i32(a):
            return None if a is None else np.ascontiguousarray(a, np.int32)

        def f32(a):
            return None if a is None else np.ascontiguousarray(a, np.float32)

        keep = dict(bg_id=i32(d.bg_id), bg_offset=i32(d.bg_offset), n_voices=i32(d.n_voices),
                    voice_id=i32(d.voice_id), voice_gain=f32(d.voice_gain),
                    voice_offset=i32(d.voice_offset), n_noises=i32(d.n_noises),
                    noise_id=i32(d.noise_id), noise_gain=f32(d.noise_gain),
                    noise_offset=i32(d.noise_offset), time_masks=i32(d.time_masks),
                    freq_masks=i32(d.freq_masks), merge_factor=f32(d.merge_factor))
        p = L.IrisPlan()
        p.batch, p.n_frame = int(d.batch), int(d.n_frame)
        p.max_voices, p.max_noises = int(d.max_voices), int(d.max_noises)
        p.min_ratio, p.min_noise_ratio = float(d.min_ratio), float(d.min_noise_ratio)
        for k, v in keep.items():
            if v is None:
                continue
            ptr_t = L._f32p if v.dtype == np.float32 else L._i32p
            setattr(p, k, v.ctypes.data_as(ptr_t))
        p.n_time_masks = 0 if d.time_masks is None else d.time_masks.shape[1]
        p.n_freq_masks = 0 if d.freq_masks is None else d.freq_masks.shape[1]
        p.stft_filter = int(stft_filter)
        p.chan_remap = int(chan_remap)
        p.n_out_chan = int(n_out_chan)
        L.check(self.lib.iris_plan_upload(self._ctx, C.byref(p), self._stream()))
        self._plan = dict(B=int(d.batch), T=int(d.n_frame), V=int(d.max_voices), remap=int(chan_remap),
                          c_out=self._remap_channels(chan_remap, n_out_chan),
                          bytes=sum(v.nbytes for v in keep.values() if v is not None))
        return self._plan

    def _remap_channels(self, chan_remap, n_out_chan):
        """C' of include/iris.h: the channels after a channel remap of the banks' channels."""
        if chan_remap == L.REMAP_NONE:
            return self.bank_chan
        return {L.REMAP_STEREO_MONO: 3, L.REMAP_MONO_CHAN: 2}.get(chan_remap, int(n_out_chan))

    def labels(self, want_vtk=False, want_keep=True):
        """-> (frame_labels [B,T,K], labels [B,V,T,K] or None, keep [B,V] uint8 or None)."""
        torch = _torch()
        pl = self._plan
        B, T, V, K = pl['B'], pl['T'], pl['V'], self.n_classes
        if V == 0:
            raise ValueError('the uploaded plan has no voices, hence no labels')
        frame = self._empty((B, T, K))
        vtk = self._empty((B, V, T, K)) if want_vtk else None
        keep = self._empty((B, V), torch.uint8) if want_keep else None
        L.check(self.lib.iris_labels(self._ctx, self._ptr(vtk), self._ptr(frame),
                                     self._ptr(keep), self._stream()))
        return frame, vtk, keep

    def feature_shape(self, mode):
        """Shape of the features of ``mode``; for FEAT_SE the shapes of its three blocks (x, only_voice,
        only_noise)."""
        pl = self._plan
        if int(mode) & L.MODE_MASK == L.FEAT_SE:
            C = self.bank_chan
            return tuple((pl['B'], 256, pl['T'], c) for c in (C, C // 2, C // 2))
        if int(mode) & L.MODE_MASK >= L.FEAT_MEL:
            return (pl['B'], self.n_mel, pl['T'], pl['c_out'])   # channels after the remap
        if int(mode) & L.MODE_MASK == L.FEAT_COMPLEX and pl['remap'] == L.REMAP_MONO_CHAN:
            return (pl['B'], 257, pl['T'], 3)                    # mono_chan's own columns
        return (pl['B'], 257, pl['T'], 2 * pl['c_out'])

    def _feature_buffer(self, mode, out, dtype):
        """-> (buffer the library writes, what the caller gets).  FEAT_SE: one flat buffer, returned as the
        contiguous views (x, only_voice, only_noise); ``out`` is then a flat tensor of their total size."""
        shape = self.feature_shape(mode)
        if int(mode) & L.MODE_MASK != L.FEAT_SE:
            if out is None:
                out = self._empty(shape, dtype)
            else:
                assert tuple(out.shape) == shape and out.is_contiguous() and out.is_cuda and out.dtype == dtype
            return out, out
        sizes = [int(np.prod(s)) for s in shape]
        if out is None:
            out = self._empty((sum(sizes),), dtype)
        else:
            assert out.numel() == sum(sizes) and out.is_contiguous() and out.is_cuda and out.dtype == dtype
        flat = out.view(-1)
        return out, tuple(v.view(s) for v, s in zip(flat.split(sizes), shape))

    def features(self, mode, out=None, select=L.SELECT_ALL, dtype=None):
        """``select``: SELECT_VOICES / SELECT_BG_NOISE give ``only_voice`` / ``only_noise`` of
        ``merge_complex_specs(seperate_noise_voice=True)`` (plain complex spectrograms).  ``dtype``:
        torch.float32 (default), torch.bfloat16 or torch.float16 -- the float32 features rounded to
        nearest even by the kernel's store; default: the dtype of ``out``, else float32.  FEAT_SE returns
        the tuple (x [B,256,T,C], only_voice [B,256,T,C//2], only_noise [B,256,T,C//2]) of views of one
        buffer (float32 only)."""
        torch = _torch()
        pl = self._plan
        if dtype is None:
            dtype = out.dtype if out is not None else torch.float32
        mode = int(mode) | out_flag(dtype)
        if select == L.SELECT_ALL:
            out, res = self._feature_buffer(mode, out, dtype)
        else:
            shape = (pl['B'], 257, pl['T'], 2 * self.bank_chan)
            if out is None:
                out = self._empty(shape, dtype)
            else:
                assert tuple(out.shape) == shape and out.is_contiguous() and out.is_cuda and out.dtype == dtype
            res = out
        L.check(self.lib.iris_features_select(self._ctx, mode, int(select), self._ptr(out), self._stream()))
        return res

    # ---- one call per batch (iris_step) ----
    def step_config(self, draw_cfg, mode, stft_filter=0, chan_remap=L.REMAP_NONE, n_out_chan=0, out_dtype=None):
        """``out_dtype``: torch.float32 (default), torch.bfloat16 or torch.float16 features."""
        flag = 0 if out_dtype is None else out_flag(out_dtype)
        return L.IrisStepConfig(draw_cfg, int(stft_filter), int(chan_remap), int(n_out_chan), int(mode) | flag)

    def step(self, scfg, uniforms, streams=None, out=None, frame=None, want_frame=True, vtk=None,
             keep=None, y_pred=None, triples=None, counts=None, comm=None, counts_reduced=None,
             triples_send=None, triples_global=None, global_batch=0, threshold=0.5):
        """ONE C call: draws from ``uniforms`` -> plan upload -> labels -> features, plus the metric
        leg (counting, count all-reduce) on the context's side stream when ``y_pred`` is given.
        -> (features, frame_labels or None); for FEAT_SE the features are the tuple of ``features``.
        ``streams``: ``plan.stream_handles(...)``."""
        torch = _torch()
        g = scfg.draw
        B, T, V = g.batch, g.n_frame, g.max_voices
        self._plan = dict(B=B, T=T, V=V, remap=int(scfg.chan_remap),
                          c_out=self._remap_channels(scfg.chan_remap, scfg.n_out_chan), bytes=0)
        mode = scfg.feature_mode
        out, res = self._feature_buffer(mode, out, out_dtype(mode))
        if frame is None and want_frame and V > 0:
            frame = self._empty((B, T, self.n_classes))
        u = uniforms if uniforms.flags['C_CONTIGUOUS'] and uniforms.dtype == np.float64 \
            else np.ascontiguousarray(uniforms, np.float64)
        io = L.IrisStepIO()
        io.uniforms = u.ctypes.data
        if streams is not None:
            io.streams = streams
        io.d_features = out.data_ptr()
        io.d_frame_labels = frame.data_ptr() if frame is not None else None
        io.d_labels_vtk = vtk.data_ptr() if vtk is not None else None
        io.d_keep = keep.data_ptr() if keep is not None else None
        if y_pred is not None:
            io.d_y_pred = y_pred.data_ptr()
            io.threshold = float(threshold)
            io.d_triples = triples.data_ptr()
            io.d_counts = counts.data_ptr() if counts is not None else None
            if comm is not None:
                io.comm = comm
                io.d_counts_reduced = counts_reduced.data_ptr()
                io.d_triples_send = triples_send.data_ptr() if triples_send is not None else None
                io.d_triples_global = triples_global.data_ptr() if triples_global is not None else None
                io.global_batch = int(global_batch)
        L.check(self.lib.iris_step(self._ctx, C.byref(scfg), C.byref(io), self._stream()))
        return res, frame

    def counts_wait(self, lag=0):
        """The current stream waits for the metric leg issued ``lag`` steps ago."""
        L.check(self.lib.iris_counts_wait(self._ctx, int(lag), self._stream()))

    def step_draws(self, scfg):
        """The draws of the last ``step`` as a :class:`BatchDraws` (copies)."""
        g = scfg.draw
        B, V, M = g.batch, g.max_voices, g.max_noises
        raw = L.IrisDraws()
        L.check(self.lib.iris_step_draws(self._ctx, C.byref(raw)))

        def arr(name, shape):
            ptr = getattr(raw, name)
            if not ptr:
                return None
            return np.ctypeslib.as_array(ptr, shape=shape).copy()
        d = BatchDraws(batch=B, n_frame=g.n_frame, max_voices=V, max_noises=M, bg_id=arr('bg_id', (B,)),
                       bg_offset=arr('bg_offset', (B,)), min_ratio=g.min_ratio,
                       min_noise_ratio=g.min_noise_ratio)
        if V > 0:
            d.n_voices, d.voice_id = arr('n_voices', (B,)), arr('voice_id', (B, V))
            d.voice_u, d.voice_gain = arr('voice_u', (B, V)), arr('voice_gain', (B, V))
            d.voice_offset = arr('voice_offset', (B, V))
        if M > 0:
            d.n_noises, d.noise_id = arr('n_noises', (B,)), arr('noise_id', (B, M))
            d.noise_u, d.noise_gain = arr('noise_u', (B, M)), arr('noise_gain', (B, M))
            d.noise_offset = arr('noise_offset', (B, M))
        if g.n_time_masks:
            d.time_masks = arr('time_masks', (B, g.n_time_masks, 2))
        if g.n_freq_masks:
            d.freq_masks = arr('freq_masks', (B, g.n_freq_masks, 2))
        if g.merge_extra:
            d.merge_factor = arr('merge_factor', (B, g.merge_extra))
        return d

    def plan_upload_bytes(self):
        return int(self.lib.iris_plan_upload_bytes(self._ctx))

    def mel_fusable(self):
        return bool(self.lib.iris_mel_fusable(self._ctx))

    # ---- DLPack hand-over ----
    def features_dlpack(self, mode, capsule):
        """``iris_features`` into the tensor behind a DLPack capsule (``to_dlpack(t)``).  Without an
        IRIS_OUT_* flag in ``mode`` the flag of the tensor's dtype (bfloat16 / float16) is added."""
        ptr = L.dlpack_pointer(capsule)
        mode = int(mode)
        if not mode & ~L.MODE_MASK:
            mode |= L.dlpack_out_flag(ptr)
        L.check(self.lib.iris_features_dlpack(self._ctx, mode, ptr, self._stream()))

    def step_dlpack(self, scfg, uniforms, features_capsule, frame_capsule=None, streams=None):
        """``iris_step`` into DLPack tensors; without an IRIS_OUT_* flag in ``scfg.feature_mode`` the flag
        of the feature tensor's dtype is added."""
        u = np.ascontiguousarray(uniforms, np.float64)
        fptr = L.dlpack_pointer(features_capsule)
        if not scfg.feature_mode & ~L.MODE_MASK:
            scfg = L.IrisStepConfig(scfg.draw, scfg.stft_filter, scfg.chan_remap, scfg.n_out_chan,
                                    scfg.feature_mode | L.dlpack_out_flag(fptr))
        g = scfg.draw
        self._plan = dict(B=g.batch, T=g.n_frame, V=g.max_voices, remap=int(scfg.chan_remap),
                          c_out=self._remap_channels(scfg.chan_remap, scfg.n_out_chan), bytes=0)
        L.check(self.lib.iris_step_dlpack(
            self._ctx, C.byref(scfg), u.ctypes.data, streams, fptr,
            L.dlpack_pointer(frame_capsule) if frame_capsule is not None else None, self._stream()))

    # ---- multi-GPU: the count all-reduce (NCCL inside libiris) ----
    def nccl_unique_id(self):
        buf = C.create_string_buffer(128)
        L.check(self.lib.iris_nccl_unique_id(buf))
        return buf.raw

    def nccl_comm(self, unique_id, rank, world_size):
        comm = C.c_void_p()
        L.check(self.lib.iris_nccl_comm_create(self._ctx, unique_id, int(rank), int(world_size), C.byref(comm)))
        return comm

    def nccl_comm_destroy(self, comm):
        L.check(self.lib.iris_nccl_comm_destroy(comm))

    def allreduce_counts(self, comm, counts_send, counts_recv, triples_send=None, triples_recv=None,
                         global_batch=0):
        L.check(self.lib.iris_allreduce_counts(
            self._ctx, comm, self._ptr(counts_send), self._ptr(counts_recv), self._ptr(triples_send),
            self._ptr(triples_recv), int(global_batch), self._stream()))

    def er_from_triples(self, triples):
        """metrics.py:268-273 on (reduced) triples ``[n,3]`` int32 -> er ``[n]``."""
        er = self._empty((triples.shape[0],))
        L.check(self.lib.iris_er_from_triples(self._ctx, self._ptr(triples), int(triples.shape[0]),
                                              self._ptr(er), self._stream()))
        return er

    def host_alloc(self, shape, dtype=np.float32):
        """Pinned host array on the NUMA node of this GPU (``iris_host_alloc``) -> (ndarray, node)."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p, node = C.c_void_p(), C.c_int(-1)
        L.check(self.lib.iris_host_alloc(self._ctx, n, C.byref(p), C.byref(node)))
        buf = (C.c_char * n).from_address(p.value)
        a = np.frombuffer(buf, dtype=dtype).reshape(shape)
        self._host_allocs = getattr(self, '_host_allocs', [])
        self._host_allocs.append((p, n))
        return a, node.value

    def plan_bytes(self, mode, keep=None, clips=None):
        """Algorithmic bytes (in, out) of the uploaded plan, optionally of the clips ``[lo, hi)``."""
        bi, bo = C.c_int64(), C.c_int64()
        k = None if keep is None else np.ascontiguousarray(keep, np.uint8)
        lo, hi = clips if clips is not None else (0, self._plan['B'])
        L.check(self.lib.iris_plan_bytes_clips(self._ctx, int(mode),
                                               k.ctypes.data if k is not None else None, int(lo), int(hi),
                                               C.byref(bi), C.byref(bo)))
        return bi.value, bo.value

    def profile_clips(self):
        return int(self.lib.iris_profile_clips(self._ctx))

    def profile(self, enable=True):
        L.check(self.lib.iris_profile_enable(self._ctx, int(bool(enable))))

    def profile_read(self, reset=True):
        """-> (summed device ms of the fused-kernel launches, number of launches)."""
        ms, n = C.c_double(), C.c_int32()
        L.check(self.lib.iris_profile_read(self._ctx, C.byref(ms), C.byref(n), int(bool(reset))))
        return ms.value, n.value

    def stft(self, wav, normalize=True):
        """``load_wav`` on an in-memory waveform ``[C, N]`` -> ``[257, T, 2C]`` (device)."""
        torch = _torch()
        if isinstance(wav, torch.Tensor):
            w = wav.to(torch.float32).contiguous()
            ptr = w.data_ptr()
        else:
            w = np.ascontiguousarray(wav, np.float32)
            ptr = w.ctypes.data
        n_chan, n = w.shape
        out = self._empty((257, 1 + n // 256, 2 * n_chan))
        L.check(self.lib.iris_stft(self._ctx, C.c_void_p(ptr), n_chan, n, int(bool(normalize)),
                                   self._ptr(out), self._stream()))
        return out

    def resample(self, wav, orig_freq, new_freq=16000):
        """``torchaudio.compliance.kaldi.resample_waveform`` (data_utils.py:20-21) on an in-memory
        waveform ``[C, N]`` (host or device) -> ``[C, N']`` (device)."""
        torch = _torch()
        if isinstance(wav, torch.Tensor):
            w = wav.to(torch.float32).contiguous()
            ptr = w.data_ptr()
        else:
            w = np.ascontiguousarray(wav, np.float32)
            ptr = w.ctypes.data
        n_chan, n = w.shape
        n_out = int(self.lib.iris_resample_len(n, int(orig_freq), int(new_freq)))
        out = self._empty((n_chan, n_out))
        L.check(self.lib.iris_resample(self._ctx, C.c_void_p(ptr), n_chan, n, int(orig_freq),
                                       int(new_freq), self._ptr(out), self._stream()))
        return out

    def metric_counts(self, y_true, y_pred, threshold=0.5, tpfpfn=None, want_er=True, counts=None):
        """-> (triples [B,3] int32, tpfpfn [3] int64 accumulated, er [B] float or None).

        ``counts``: optional int64 ``[6]`` device tensor ``[TP, FP, FN, sum n_true, sum n_pred,
        sum correct]`` accumulated in place (the multi-GPU all-reduce payload); it then also
        serves as ``tpfpfn``."""
        torch = _torch()
        yt = torch.as_tensor(y_true, dtype=torch.float32, device=self.device).contiguous()
        yp = torch.as_tensor(y_pred, dtype=torch.float32, device=self.device).contiguous()
        B, T, K = yt.shape
        assert yp.shape == yt.shape
        triples = self._empty((B, 3), torch.int32)
        sums = None
        if counts is not None:
            assert counts.dtype == torch.int64 and counts.numel() == 6 and counts.is_contiguous()
            tpfpfn, sums = counts[:3], counts[3:]
        elif tpfpfn is None:
            tpfpfn = torch.zeros(3, dtype=torch.int64, device=self.device)
        er = self._empty((B,)) if want_er else None
        L.check(self.lib.iris_metric_counts(self._ctx, self._ptr(yt), self._ptr(yp), B, T, K,
                                            float(threshold), self._ptr(triples),
                                            self._ptr(tpfpfn), self._ptr(sums), self._ptr(er),
                                            self._stream()))
        return triples, tpfpfn, er


    def er_counts_pooled(self, y_true, y_pred_pooled, threshold=0.5):
        """``er_score(smoothing=True)`` core: ``y_pred_pooled`` is on the pooled time base
        (metrics.py:222-224).  -> (triples [B,3] int32, er [B] float)."""
        torch = _torch()
        yt = torch.as_tensor(y_true, dtype=torch.float32, device=self.device).contiguous()
        yp = torch.as_tensor(y_pred_pooled, dtype=torch.float32, device=self.device).contiguous()
        B, T, K = yt.shape
        assert yp.shape[0] == B and yp.shape[2] == K
        triples = self._empty((B, 3), torch.int32)
        er = self._empty((B,))
        L.check(self.lib.iris_er_counts_pooled(self._ctx, self._ptr(yt), T, self._ptr(yp),
                                               int(yp.shape[1]), B, K, float(threshold),
                                               self._ptr(triples), self._ptr(er), self._stream()))
        return triples, er


_engines = {}


def get_engine(device=None):
    """Process-wide engine of a device (default: torch's current CUDA device)."""
    torch = _torch()
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    device = int(device)
    if device not in _engines:
        _engines[device] = Engine(device)
    return _engines[device]
