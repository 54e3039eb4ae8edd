"""ctypes binding of libiris.so (include/iris.h).  There is NO CPU fallback: if the
shared library is missing or no CUDA device is present, importing the compute entry
points fails loudly."""
import ctypes as C
import os

from .errors import InvalidArgumentError, IrisError

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('IRIS_LIB') or os.path.join(_HERE, 'libiris.so')   # IRIS_LIB: experiment builds

IRIS_OK, IRIS_ERR_INVALID, IRIS_ERR_CUDA, IRIS_ERR_EMPTY_RANGE, IRIS_ERR_STATE, \
    IRIS_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
BANK_BG, BANK_VOICE, BANK_NOISE = 0, 1, 2
FEAT_COMPLEX, FEAT_MAGPHASE, FEAT_LOG_MAGPHASE, FEAT_MEL, FEAT_LOGMEL, FEAT_LOGMEL_MINMAX = range(6)
FEAT_SE = 6   # x, only_voice, only_noise of the 'se' model: three blocks of one buffer (include/iris.h)
REMAP_NONE, REMAP_STEREO_MONO, REMAP_MERGE_AUG, REMAP_MONO_CHAN = 0, 1, 2, 3
SELECT_ALL, SELECT_VOICES, SELECT_BG_NOISE = 0, 1, 2
# output element type, OR-ed into a feature mode (none: float32)
OUT_BF16, OUT_F16 = 0x100, 0x200
MODE_MASK = 0xff

_i32p = C.POINTER(C.c_int32)
_f32p = C.POINTER(C.c_float)


class IrisPlan(C.Structure):
    _fields_ = [
        ('batch', C.c_int32), ('n_frame', C.c_int32), ('max_voices', C.c_int32),
        ('max_noises', C.c_int32), ('min_ratio', C.c_float), ('min_noise_ratio', C.c_float),
        ('bg_id', _i32p), ('bg_offset', _i32p), ('n_voices', _i32p), ('voice_id', _i32p),
        ('voice_gain', _f32p), ('voice_offset', _i32p), ('n_noises', _i32p), ('noise_id', _i32p),
        ('noise_gain', _f32p), ('noise_offset', _i32p), ('n_time_masks', C.c_int32),
        ('n_freq_masks', C.c_int32), ('time_masks', _i32p), ('freq_masks', _i32p),
        ('stft_filter', C.c_int32), ('chan_remap', C.c_int32), ('n_out_chan', C.c_int32),
        ('merge_factor', _f32p),
    ]


class IrisDrawConfig(C.Structure):
    _fields_ = [
        ('batch', C.c_int32), ('n_frame', C.c_int32), ('max_voices', C.c_int32), ('max_noises', C.c_int32),
        ('min_ratio', C.c_float), ('min_noise_ratio', C.c_float), ('snr', C.c_float),
        ('n_time_masks', C.c_int32), ('time_mask_max', C.c_int32), ('n_freq_masks', C.c_int32),
        ('freq_mask_max', C.c_int32), ('n_bins', C.c_int32), ('merge_extra', C.c_int32),
    ]


class IrisDraws(C.Structure):
    _fields_ = [
        ('bg_id', _i32p), ('bg_offset', _i32p),
        ('n_voices', _i32p), ('voice_id', _i32p), ('voice_u', _f32p), ('voice_gain', _f32p), ('voice_offset', _i32p),
        ('n_noises', _i32p), ('noise_id', _i32p), ('noise_u', _f32p), ('noise_gain', _f32p), ('noise_offset', _i32p),
        ('time_masks', _i32p), ('freq_masks', _i32p), ('merge_factor', _f32p),
    ]


class IrisStepConfig(C.Structure):
    _fields_ = [('draw', IrisDrawConfig), ('stft_filter', C.c_int32), ('chan_remap', C.c_int32),
                ('n_out_chan', C.c_int32), ('feature_mode', C.c_int32)]


class IrisStepIO(C.Structure):
    _fields_ = [
        ('uniforms', C.c_void_p), ('streams', C.POINTER(C.c_void_p)),
        ('d_features', C.c_void_p), ('d_frame_labels', C.c_void_p), ('d_labels_vtk', C.c_void_p),
        ('d_keep', C.c_void_p),
        ('d_y_pred', C.c_void_p), ('threshold', C.c_float), ('d_triples', C.c_void_p),
        ('d_counts', C.c_void_p), ('comm', C.c_void_p), ('d_counts_reduced', C.c_void_p),
        ('d_triples_send', C.c_void_p), ('d_triples_global', C.c_void_p), ('global_batch', C.c_int32),
    ]


# name -> (restype, argtypes); also the list of symbols include/iris.h declares
SIGNATURES = {
    'iris_abi_version': (C.c_int, []),
    'iris_last_error': (C.c_char_p, []),
    'iris_ctx_create': (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    'iris_ctx_destroy': (C.c_int, [C.c_void_p]),
    'iris_set_mel': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    'iris_bank_register': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    'iris_bank_register_audio': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    'iris_specbank_register': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    'iris_bank_info': (C.c_int, [C.c_void_p, C.c_int, _i32p, _i32p, C.c_void_p]),
    'iris_bank_activity': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    'iris_plan_upload': (C.c_int, [C.c_void_p, C.POINTER(IrisPlan), C.c_void_p]),
    'iris_labels': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'iris_features': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'iris_features_select': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    'iris_stft': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p,
                            C.c_void_p]),
    'iris_metric_counts': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                     C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    'iris_er_counts_pooled': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                        C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    'iris_profile_enable': (C.c_int, [C.c_void_p, C.c_int]),
    'iris_profile_read': (C.c_int, [C.c_void_p, C.POINTER(C.c_double), _i32p, C.c_int]),
    'iris_plan_bytes': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int64),
                                  C.POINTER(C.c_int64)]),
    'iris_plan_bytes_clips': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                        C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    'iris_profile_clips': (C.c_int, [C.c_void_p]),
    # stand-alone stages (include/iris.h, second half)
    'iris_op_mask': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                               C.c_void_p, C.c_int, C.c_void_p]),
    'iris_op_stft_filter': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                      C.c_int, C.c_void_p]),
    'iris_op_random_shift': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                       C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    'iris_debug_claims': (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    'iris_op_normalize': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'iris_op_pointwise': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                    C.c_int, C.c_float, C.c_void_p]),
    'iris_op_chan_map': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                   C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    'iris_op_mel': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                              C.c_void_p]),
    'iris_op_minmax': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                 C.c_int, C.c_void_p]),
    'iris_op_sum_voices': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                     C.c_int64, C.c_void_p]),
    'iris_op_avg_pool_time': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_int, C.c_void_p]),
    'iris_op_cos_sim': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                  C.c_int, C.c_void_p]),
    'iris_op_phase_vocoder': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'iris_resample_len': (C.c_int64, [C.c_int64, C.c_int, C.c_int]),
    'iris_resample': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p,
                                C.c_void_p]),
    'iris_op_sum_pool2': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                    C.c_float, C.c_void_p]),
    'iris_op_density_labels': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                         C.c_int64, C.c_void_p]),
    # evaluation-side chain (metrics.evaluate)
    'iris_op_eval_windows': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                       C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    'iris_op_eval_merge': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_int, C.c_void_p]),
    'iris_op_eval_smooth': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    'iris_op_eval_events': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'iris_op_get_er': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                 C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    # one call per batch, host planner, NCCL, pinned memory, DLPack (include/iris.h, round 2)
    'iris_shuffle_create': (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'iris_shuffle_destroy': (C.c_int, [C.c_void_p]),
    'iris_shuffle_take': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    'iris_draw_uniforms_per_clip': (C.c_int, [C.POINTER(IrisDrawConfig)]),
    'iris_draw_batch': (C.c_int, [C.POINTER(IrisDrawConfig), C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                  C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p,
                                  C.POINTER(IrisDraws)]),
    'iris_step': (C.c_int, [C.c_void_p, C.POINTER(IrisStepConfig), C.POINTER(IrisStepIO), C.c_void_p]),
    'iris_counts_wait': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    'iris_step_draws': (C.c_int, [C.c_void_p, C.POINTER(IrisDraws)]),
    'iris_allreduce_counts': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_int, C.c_void_p]),
    'iris_nccl_unique_id': (C.c_int, [C.c_void_p]),
    'iris_nccl_comm_create': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'iris_nccl_comm_destroy': (C.c_int, [C.c_void_p]),
    'iris_er_from_triples': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'iris_host_alloc': (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]),
    'iris_host_free': (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    'iris_features_dlpack': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'iris_labels_dlpack': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'iris_step_dlpack': (C.c_int, [C.c_void_p, C.POINTER(IrisStepConfig), C.c_void_p, C.POINTER(C.c_void_p),
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    'iris_mel_fusable': (C.c_int, [C.c_void_p]),
    'iris_plan_upload_bytes': (C.c_int64, [C.c_void_p]),
    'iris_max_segments': (C.c_int, []),
}
# symbols added under IRIS_ABI_VERSION 2 that an older library lacks (callers probe with hasattr)
OPTIONAL = {'iris_bank_register_audio'}
PW_C2MP, PW_MP2C, PW_LOG_MAGPHASE, PW_LOG_ON_MEL, PW_MULTIPLY = range(5)
MAP_MONO_CHAN, MAP_STEREO_MONO, MAP_MERGE_AUG = range(3)

_lib = None


def load():
    """Load libiris.so (built in-tree by ``python -m challenge_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'challenge_b200/libiris.so is missing -- build it with '
            '`python -m challenge_b200.build` (needs nvcc).  There is no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        if name in OPTIONAL and not hasattr(lib, name):
            continue
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def dlpack_pointer(capsule):
    """``DLManagedTensor*`` behind a DLPack PyCapsule (name "dltensor": not consumed yet)."""
    C.pythonapi.PyCapsule_GetPointer.restype = C.c_void_p
    C.pythonapi.PyCapsule_GetPointer.argtypes = [C.py_object, C.c_char_p]
    return C.c_void_p(C.pythonapi.PyCapsule_GetPointer(capsule, b'dltensor'))


class _DLDataType(C.Structure):
    _fields_ = [('code', C.c_uint8), ('bits', C.c_uint8), ('lanes', C.c_uint16)]


class _DLTensorHead(C.Structure):   # the leading fields of DLTensor (include/iris_dlpack.h)
    _fields_ = [('data', C.c_void_p), ('device_type', C.c_int32), ('device_id', C.c_int32),
                ('ndim', C.c_int32), ('dtype', _DLDataType)]


def dlpack_out_flag(managed):
    """OUT_BF16 / OUT_F16 for a bfloat16 / float16 ``DLManagedTensor*``, else 0 (the library checks
    the dtype against the flag)."""
    dt = _DLTensorHead.from_address(managed.value).dtype
    return {(4, 16): OUT_BF16, (2, 16): OUT_F16}.get((dt.code, dt.bits), 0)


def check(rc):
    if rc == IRIS_OK:
        return
    msg = load().iris_last_error().decode('utf-8', 'replace')
    if rc == IRIS_ERR_EMPTY_RANGE:
        raise InvalidArgumentError(msg)
    if rc == IRIS_ERR_INVALID:
        raise ValueError(msg)
    if rc == IRIS_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise IrisError('libiris error %d: %s' % (rc, msg))
