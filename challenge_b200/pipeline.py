"""Drop-in mirror of the reference's ``pipeline.py``: ``make_pipeline`` / ``merge_complex_specs``.

The reference zips three shuffled ``tf.data`` streams of PRE-COMPUTED complex spectrograms and
maps ``merge_complex_specs`` over them, one sample at a time on one host thread
(pipeline.py:113-175).  Here the banks are registered once in HBM, in either format:

* WAVEFORMS ``[chan, samples]`` -- the fast path: the STFT of ``data_utils.load_wav`` moves into
  the per-step fused kernel (time-domain mix, one FFT per output frame);
* the reference's own SPECTROGRAMS ``[257, time, chan*2]`` (``utils.load_data`` pickles): mixed in
  the spectrogram domain by a streaming kernel with the reference's arithmetic (k_spec.cu).

The host only draws the randomness of a whole batch in the reference's draw order
(``plan.draw_batch``) and one launch produces ``batch`` samples.

``make_pipeline`` returns an :class:`IrisDataset` with the slice of the ``tf.data`` surface
that ``sj_train.make_dataset`` (sj_train.py:92-130) uses -- ``map``, ``batch``, ``prefetch``,
``take``, ``repeat``, iteration.  Chaining the drop-in functions in sj_train's order
(``to_frame_labels``, ``augment``, ``stereo_mono`` | ``random_merge_aug(n)`` | ``mono_chan``,
``stft_filter(k)``, ``batch``, ``complex_to_magphase``, ``magphase_to_mel(n)``, ``minmax``,
``log_on_mel``) is recognised and lowered to ONE fused launch per batch (``mono_chan`` of 2-channel
banks only); so is the 'se' chain
(``seperate_noise_voice=True``, [``augment``, ``stft_filter(k)``,] ``speech_enhancement_preprocess``,
``batch``, sj_train.py:99-106) of 2-channel banks.  Any other callable runs after it on the un-fused
tensors (the stand-alone kernels), so arbitrary chains work.
"""
import numpy as np

from . import _lib as L
from . import _ops as O
from .engine import Engine, get_engine, is_spec_bank
from .plan import ShuffleStream, draw_batch, draw_config, stream_handles, uniforms_per_clip

AUTOTUNE = -1   # tf.data.experimental.AUTOTUNE stand-in for .prefetch()


def _is_waveform_bank(items):
    return isinstance(items[0], tuple) or np.asarray(items[0]).ndim == 2


class IrisDataset:
    """Lazy description of ``make_pipeline(...)`` followed by ``map`` / ``batch`` / ``take`` stages.

    Every pipeline owns its engine (= its ``iris_ctx`` and bank set), so a train and a test
    pipeline built back to back (sj_train.py:472-473, trainer.py:261-262) stay independent."""

    def __init__(self, source, stages=(), batch_size=None, limit=None, elem_limit=None,
                 drop_remainder=False):
        self._src = source
        self._stages = tuple(stages)        # callables; ('batch', n) marks the batch point
        self._batch = batch_size
        self._limit = limit                 # take() after batch(): batches
        self._elem_limit = elem_limit       # take() before batch(): elements, as in tf.data
        self._drop_remainder = drop_remainder

    def _with(self, **kw):
        args = dict(source=self._src, stages=self._stages, batch_size=self._batch, limit=self._limit,
                    elem_limit=self._elem_limit, drop_remainder=self._drop_remainder)
        args.update(kw)
        return IrisDataset(**args)

    # ---- tf.data surface used by sj_train.make_dataset ----
    def map(self, fn, num_parallel_calls=None):
        return self._with(stages=self._stages + (fn,))

    def batch(self, batch_size, drop_remainder=False):
        if self._batch is not None:
            raise ValueError('IrisDataset is already batched')
        return self._with(stages=self._stages + (('batch', int(batch_size)),), batch_size=int(batch_size),
                          drop_remainder=bool(drop_remainder))

    def prefetch(self, buffer_size=None):
        return self

    def repeat(self, count=None):
        return self

    def shuffle(self, buffer_size, **kwargs):
        return self      # the source streams are already shuffled (pipeline.py:147,154,164)

    def take(self, count):
        count = int(count)
        if self._batch is None:             # elements, like tf.data; batch() then sees `count` of them
            cur = self._elem_limit
            return self._with(elem_limit=count if cur is None else min(cur, count))
        cur = self._limit
        return self._with(limit=count if cur is None else min(cur, count))

    @property
    def engine(self):
        return self._src['engine']

    # ---- lowering ----
    def _lower(self, allow_mel=True):
        """Split the stage list into what the fused kernel absorbs and the remainder."""
        fused = dict(frame_labels=False, density_labels=False, augment=False, remap=L.REMAP_NONE, n_out=0, filt=0,
                     mode=L.FEAT_COMPLEX, n_mels=0, mel_matrix=None, out_flag=0)
        rest = []
        state = 'pre'       # pre-batch element stages -> post-batch feature stages
        order = {'to_frame_labels': 0, 'density_labels': 0, 'augment': 1, 'stereo_mono': 2, 'merge_aug': 2,
                 'mono_chan': 2, 'stft_filter': 3}
        last = -1
        stages = list(self._stages)
        i = 0
        while i < len(stages):
            st = stages[i]
            tag = getattr(st, '_iris_stage', None) if callable(st) else st
            if rest:
                rest.append(st)
            elif state == 'pre' and tag and tag[0] in order and order[tag[0]] > last \
                    and (tag[0] != 'mono_chan' or self._src.get('n_chan') == 2):
                last = order[tag[0]]
                if tag[0] == 'to_frame_labels':
                    fused['frame_labels'] = True
                elif tag[0] == 'density_labels':            # trainer.to_density_labels (labels only)
                    fused['density_labels'] = True
                elif tag[0] == 'augment':
                    fused['augment'] = True
                elif tag[0] == 'stereo_mono':
                    fused['remap'], fused['n_out'] = L.REMAP_STEREO_MONO, 3
                elif tag[0] == 'merge_aug':
                    fused['remap'], fused['n_out'] = L.REMAP_MERGE_AUG, int(tag[1])
                elif tag[0] == 'mono_chan':                 # 2-channel banks only (IRIS_REMAP_MONO_CHAN)
                    fused['remap'], fused['n_out'] = L.REMAP_MONO_CHAN, 2
                elif tag[0] == 'stft_filter':
                    fused['filt'] = int(tag[1])
            elif state == 'pre' and tag and tag[0] == 'se' and self._se_fusable(fused, last, i):
                fused['mode'] = L.FEAT_SE      # x, (frame labels, only_voice, only_noise) in one step
                last = len(order)              # no pre-batch stage is absorbed behind it
            elif state == 'pre' and tag and tag[0] == 'batch':
                state = 'post'
            elif state == 'post' and tag and tag[0] == 'magphase' and fused['mode'] == L.FEAT_COMPLEX:
                fused['mode'] = L.FEAT_MAGPHASE
            elif state == 'post' and allow_mel and tag and tag[0] == 'mel' and fused['mode'] == L.FEAT_MAGPHASE:
                fused['mode'], fused['n_mels'], fused['mel_matrix'] = L.FEAT_MEL, tag[1], tag[2]
            elif state == 'post' and tag and tag[0] == 'minmax' and fused['mode'] == L.FEAT_MEL \
                    and i + 1 < len(stages) and getattr(stages[i + 1], '_iris_stage', (None,))[0] == 'log_on_mel':
                fused['mode'] = L.FEAT_LOGMEL_MINMAX
                i += 1
            elif state == 'post' and tag and tag[0] == 'minmax_log' and fused['mode'] == L.FEAT_MEL:
                fused['mode'] = L.FEAT_LOGMEL_MINMAX          # trainer.minmax_log_on_mel
            elif state == 'post' and tag and tag[0] == 'log_on_mel' and fused['mode'] == L.FEAT_MEL:
                fused['mode'] = L.FEAT_LOGMEL
            elif state == 'post' and tag and tag[0] == 'cast' and fused['out_flag'] == 0 \
                    and fused['mode'] != L.FEAT_SE:
                fused['out_flag'] = tag[1]                    # data_utils.cast_features: the kernels store it
            else:
                rest.append(st)
            i += 1
        return fused, rest

    def _se_fusable(self, fused, last, i):
        """``speech_enhancement_preprocess`` at stage ``i`` lowers to FEAT_SE: a ``seperate_noise_voice`` source
        of 2-channel banks, the stage first before ``.batch()`` or behind ``augment`` / ``stft_filter`` only,
        and, unbatched, the last stage."""
        src = self._src
        return bool(src.get('separate')) and src.get('n_chan') == 2 and last in (-1, 1, 3) \
            and not fused['frame_labels'] and not fused['density_labels'] and fused['remap'] == L.REMAP_NONE \
            and (self._batch is not None or i + 1 == len(self._stages))

    def _prepare(self):
        """Lower the stage list once per iteration: fused step configuration + leftover stages."""
        src = self._src
        eng = src['engine']
        fused, rest = self._lower()
        if L.FEAT_MEL <= fused['mode'] <= L.FEAT_LOGMEL_MINMAX:
            cur = eng.mel_matrix
            if cur is None or cur.shape != fused['mel_matrix'].shape \
                    or not np.array_equal(cur, fused['mel_matrix']):
                eng.set_mel(mel_matrix=fused['mel_matrix'])
            if not src['spec_banks'] and not eng.mel_fusable():
                # a filter wider than the fused epilogue takes (e.g. n_mels = 20): the fused kernel
                # stops at magnitude + phase and the mel stage runs as the stand-alone kernel
                fused, rest = self._lower(allow_mel=False)
        # stages the fused launch did not absorb: the ones mapped BEFORE .batch() see single
        # elements in the reference, so they run per element here (then the batch is re-stacked)
        pre, post = [], []
        seen_batch = not any(isinstance(st, tuple) and st[0] == 'batch' for st in rest)
        for st in rest:
            if isinstance(st, tuple) and st[0] == 'batch':
                seen_batch = True
                continue
            (post if seen_batch and self._batch is not None else pre).append(st)
        return fused, pre, post

    def _step_config(self, fused, B):
        src = self._src
        cfg = draw_config(B, src['n_frame'], src['max_voices'], src['max_noises'], src['snr'],
                          src['min_ratio'], src['min_noise_ratio'],
                          6 if fused['augment'] else 0, 24, 1 if fused['augment'] else 0, 16, 257,
                          max(fused['n_out'] - 2, 0) if fused['remap'] == L.REMAP_MERGE_AUG else 0)
        return src['engine'].step_config(cfg, fused['mode'] | fused['out_flag'], stft_filter=fused['filt'],
                                         chan_remap=fused['remap'], n_out_chan=fused['n_out'])

    def __iter__(self):
        src = self._src
        eng = src['engine']
        fused, pre, post = self._prepare()
        B = self._batch or 1
        handles = stream_handles(src['streams'])
        configs = {}

        def config_for(b):
            if b not in configs:
                sc = self._step_config(fused, b)
                configs[b] = (sc, uniforms_per_clip(sc.draw))
            return configs[b]

        def _el(t, i):
            return tuple(u[i] for u in t) if isinstance(t, tuple) else t[i]

        def _stack(items):
            import torch
            if isinstance(items[0], tuple):
                return tuple(torch.stack([it[k] for it in items]) for k in range(len(items[0])))
            return torch.stack(list(items))

        n_batches = 0
        elems_left = self._elem_limit
        while self._limit is None or n_batches < self._limit:
            b = B
            if elems_left is not None:
                if elems_left <= 0 or (elems_left < B and self._drop_remainder):
                    break
                b = min(B, elems_left)
                elems_left -= b
            scfg, n_u = config_for(b)
            se = fused['mode'] == L.FEAT_SE
            want_frame = fused['frame_labels'] or se
            want_vtk = not want_frame or fused['density_labels']
            vtk = eng._empty((b, src['max_voices'], src['n_frame'], eng.n_classes)) if want_vtk else None
            # ONE C call: draws -> plan -> labels -> features (include/iris.h iris_step)
            x, frame = eng.step(scfg, O.rng().random((b, n_u)), streams=handles, vtk=vtk,
                                want_frame=want_frame)
            y = frame if fused['frame_labels'] else vtk
            if fused['density_labels']:
                from .trainer import to_density_labels
                _, y = to_density_labels(None, vtk)
            if se:                    # speech_enhancement_preprocess's (x, (frame labels, only_voice, only_noise))
                x, y = x[0], (frame, x[1], x[2])
            elif src.get('separate'):   # (label, only_voice, only_noise), pipeline.py:107-108
                y = (y, eng.features(L.FEAT_COMPLEX, select=L.SELECT_VOICES),
                     eng.features(L.FEAT_COMPLEX, select=L.SELECT_BG_NOISE))
            if pre:
                xs, ys = [], []
                for i in range(b):
                    xi, yi = _el(x, i), _el(y, i)
                    for st in pre:
                        res = st(xi, yi)
                        xi, yi = res if isinstance(res, tuple) and len(res) == 2 else (res, yi)
                    xs.append(xi)
                    ys.append(yi)
                x, y = _stack(xs), _stack(ys)
            if self._batch is None:
                x, y = _el(x, 0), _el(y, 0)
            for st in post:
                res = st(x, y)
                x, y = res if isinstance(res, tuple) and len(res) == 2 else (res, y)
            n_batches += 1
            yield x, y


_merge_engines = {}


def _merge_engine():
    """Engine of the single-sample ``merge_complex_specs`` calls (one per device)."""
    import torch
    dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if dev not in _merge_engines:
        _merge_engines[dev] = Engine(dev)
    return _merge_engines[dev]


def merge_complex_specs(background, voices_and_labels, noises=None, n_frame=300, n_classes=3,
                        t_axis=1, min_ratio=2 / 3, min_noise_ratio=1 / 2, snr=-20,
                        seperate_noise_voice=False, *, draws=None):
    '''
    pipeline.py:6-110 for ONE sample.  ``background`` [freq, time, chan2] (the reference's
    format) or a waveform [chan, samples]; ``voices_and_labels`` = (the whole padded_batch
    group of voices in the same format, labels [n, n_classes]); ``noises`` likewise or None.

    OUTPUT:
        complex_spec: (freq, time, chan2)
        labels: (n_voices, time, n_classes)
    '''
    voices, labels = voices_and_labels
    if not isinstance(background, tuple) and np.asarray(background).ndim not in (2, 3):
        raise ValueError('background must be a spectrogram [freq, time, chan2] or a waveform [chan, samples]')
    if t_axis != 1:
        raise NotImplementedError('merge_complex_specs: t_axis must be 1 (the only value the reference uses)')
    eng = _merge_engine()     # not a pipeline's engine: live datasets keep their banks
    bf = eng.register_bank(L.BANK_BG, [background])
    vf = eng.register_bank(L.BANK_VOICE, list(voices), labels=np.asarray(labels, np.float32))
    nf = eng.register_bank(L.BANK_NOISE, list(noises)) if noises is not None else None
    V, M = len(voices), (len(noises) if noises is not None else 0)
    if draws is None:
        draws = draw_batch(O.rng(), 1, n_frame, bf, vf, nf, max_voices=V, max_noises=M, snr=snr,
                           min_ratio=min_ratio, min_noise_ratio=min_noise_ratio)
        draws.voice_id[:] = np.arange(V)
        if M:
            draws.noise_id[:] = np.arange(M)
    eng.upload_plan(draws)
    _, vtk, _ = eng.labels(want_vtk=True, want_keep=False)
    spec = eng.features(L.FEAT_COMPLEX)
    if seperate_noise_voice:     # pipeline.py:37-38, 82-83, 104-108
        only_voice = eng.features(L.FEAT_COMPLEX, select=L.SELECT_VOICES)
        only_noise = eng.features(L.FEAT_COMPLEX, select=L.SELECT_BG_NOISE)
        return spec[0], (vtk[0], only_voice[0], only_noise[0])
    return spec[0], vtk[0]


def make_pipeline(backgrounds,  # a list of background noises  (waveforms [chan, samples])
                  voices,       # a list of human voices
                  labels,       # a list of labels of human voices
                  noises=None,  # a list of additional noises
                  n_frame=300,  # number of frames per sample
                  max_voices=10,
                  max_noises=10,
                  n_classes=3,
                  **kwargs):
    '''
    OUTPUT
        dataset: IrisDataset yielding
                 complex spectrogram: [freq_bins, n_frame, chan*2]
                     [..., :chan] = real
                     [..., chan:] = imag
                 labels: [max_voices, n_frame, n_classes]
    (pipeline.py:113-175; kwargs = merge_complex_specs' min_ratio / min_noise_ratio / snr)
    '''
    # pipeline.py:136 asserts 3-D spectrograms; waveform banks [chan, samples] are accepted too
    assert _is_waveform_bank(backgrounds) or is_spec_bank(backgrounds), 'each spec must be a 3D-tensor'
    assert len(voices) == len(labels)
    assert len(np.asarray(labels[0]).shape) == 1 and np.asarray(labels[0]).shape[0] == n_classes, \
        'labels must be in the form of [n_samples, n_classes]'
    import torch
    eng = Engine(torch.cuda.current_device() if torch.cuda.is_available() else 0)   # this pipeline's bank set
    bf = eng.register_bank(L.BANK_BG, list(backgrounds))
    vf = eng.register_bank(L.BANK_VOICE, list(voices), labels=np.asarray(labels, np.float32))
    nf = eng.register_bank(L.BANK_NOISE, list(noises)) if noises is not None else None
    spec_banks = not _is_waveform_bank(backgrounds)
    V, M = int(max_voices), int(max_noises) if noises is not None else 0
    if not spec_banks:
        # the fused kernel mixes at most iris_max_segments() source segments per clip: background
        # tiles (pipeline.py:29-35) + accepted voices (< max_voices) + noises (< max_noises)
        reps = -(-int(n_frame) // int(min(bf)))
        worst = (reps + 1) + max(V - 1, 1) + max(M - 1, 0)
        cap = int(eng.lib.iris_max_segments())
        if worst > cap:
            raise ValueError(
                'make_pipeline: a clip could mix %d segments (%d background tiles of the shortest '
                'background (%d frames < n_frame=%d), %d voices, %d noises); the fused kernel takes '
                '%d.  Use longer backgrounds, fewer max_voices / max_noises, or spectrogram banks.'
                % (worst, reps + 1, int(min(bf)), int(n_frame), max(V - 1, 1), max(M - 1, 0), cap))
    r = O.rng()
    streams = {'bg': ShuffleStream(len(backgrounds), r), 'voice': ShuffleStream(len(voices), r)}
    if noises is not None:
        streams['noise'] = ShuffleStream(len(noises), r)
    source = dict(engine=eng, n_frame=int(n_frame), bg_frames=bf, voice_frames=vf, noise_frames=nf,
                  max_voices=int(max_voices), max_noises=int(max_noises) if noises is not None else 0,
                  snr=kwargs.get('snr', -20), min_ratio=kwargs.get('min_ratio', 2 / 3),
                  min_noise_ratio=kwargs.get('min_noise_ratio', 1 / 2), streams=streams,
                  separate=bool(kwargs.get('seperate_noise_voice', False)), spec_banks=spec_banks,
                  n_chan=eng.bank_chan)
    return IrisDataset(source)
