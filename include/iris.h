/* libiris -- C ABI of the B200-native preprocessing hot path of IRIS-AUDIO/challenge.
 *
 * The reference has no FFI: its boundary is the Python function surface of pipeline.py,
 * transforms.py, data_utils.py and metrics.py, consumed as tf.data map callables and Keras
 * metric callables.  This header is what a maintainer's binding (ctypes / a TF custom op /
 * cffi) calls instead; every entry point names the reference code it replaces.  Plain
 * pointers and sizes only; device buffers are CALLER-allocated (framework allocator) and
 * handed over as raw pointers (DLPack `data` + `byte_offset`), outputs are written in the
 * reference's layouts, all work is enqueued on the caller's CUDA stream.  Return 0 on
 * success, a negative IRIS_ERR_* otherwise; iris_last_error() gives the thread-local text.
 * There is no CPU fallback: without a CUDA device every compute entry point fails.
 *
 * One context per device; calls on one context are serialised by the caller.
 */
#ifndef IRIS_H_
#define IRIS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IRIS_ABI_VERSION 2

typedef struct iris_ctx iris_ctx;
typedef void* iris_stream; /* cudaStream_t */

enum {
    IRIS_OK = 0,
    IRIS_ERR_INVALID = -1,     /* bad argument (reference: assert / ValueError) */
    IRIS_ERR_CUDA = -2,        /* CUDA runtime error, text in iris_last_error() */
    IRIS_ERR_EMPTY_RANGE = -3, /* reference: tf InvalidArgumentError on int-uniform with
                                  maxval <= minval (pipeline.py:68-69) */
    IRIS_ERR_STATE = -4,       /* call order (no plan / bank not registered) */
    IRIS_ERR_UNSUPPORTED = -5  /* valid in the reference, outside the fused path */
};

enum { IRIS_BANK_BG = 0, IRIS_BANK_VOICE = 1, IRIS_BANK_NOISE = 2 };

/* feature modes of iris_features(); layouts as in the reference.  C' is the channel count after the
 * plan's channel remap (3 for stereo_mono, n_out_chan for random_merge_aug, 2 for mono_chan, else the
 * bank's), in the spectrogram and the mel layouts alike: a remap is fused in front of the mel projection.
 * (A library older than that answers the mel modes of a remapped plan with IRIS_ERR_UNSUPPORTED.)  One
 * exception: IRIS_FEAT_COMPLEX of a mono_chan plan is [B,257,T,3], see IRIS_REMAP_MONO_CHAN. */
enum {
    IRIS_FEAT_COMPLEX = 0,       /* [B,257,T,2C']  make_pipeline output (pipeline.py:131-133)  */
    IRIS_FEAT_MAGPHASE = 1,      /* [B,257,T,2C']  complex_to_magphase (transforms.py:111-123)  */
    IRIS_FEAT_LOG_MAGPHASE = 2,  /* [B,257,T,2C']  + log_magphase (transforms.py:80-86)         */
    IRIS_FEAT_MEL = 3,           /* [B,n_mel,T,C'] magphase_to_mel (transforms.py:51-77)        */
    IRIS_FEAT_LOGMEL = 4,        /* [B,n_mel,T,C'] + log_on_mel ('nominmax', sj_train.py:121)   */
    IRIS_FEAT_LOGMEL_MINMAX = 5, /* [B,n_mel,T,C'] + minmax + log_on_mel (sj_train.py:119-123)  */
    IRIS_FEAT_SE = 6             /* the batch of the 'se' model, see below                      */
};

/* IRIS_FEAT_SE: merge_complex_specs(seperate_noise_voice=True) followed by
 * speech_enhancement_preprocess (pipeline.py:37-38, 82-83, 104-108; data_utils.py:139-148), the chain of
 * the 'se' model (sj_train.py:99-106), for a 2-channel plan without a channel remap.  The feature buffer
 * holds three C-contiguous float32 blocks back to back, each starting 16-byte aligned:
 *   x          [B,256,T,C]    real parts of bins 1..256 of the mix, after the plan's masks and stft_filter
 *   only_voice [B,256,T,C/2]  real part of channel 0 of the sum of the kept voices
 *   only_noise [B,256,T,C/2]  real part of channel 0 of background + noises
 * (C/2 channels: the reference cuts the two label spectrograms after x was halved.)  Masks and
 * stft_filter act on x only.  Other channel counts and remapped plans are IRIS_ERR_UNSUPPORTED; an
 * IRIS_OUT_* flag, a selection other than IRIS_SELECT_ALL and the DLPack entry points are
 * IRIS_ERR_INVALID (as is the mode itself for a library that predates it, so callers can probe for it).
 * The frame labels of the batch come from iris_labels / iris_step as for every mode. */

/* Output element type, OR-ed into the mode of iris_features, iris_features_select,
 * iris_features_dlpack, iris_plan_bytes(_clips) and into iris_step_config.feature_mode.  Without a
 * flag the features are float32.  With one, the output buffer holds 2-byte elements in the same
 * layout, equal bit for bit to the float32 features converted with round-to-nearest-even (torch's
 * .to(torch.bfloat16 / torch.float16); float16 overflow gives +-inf).  All arithmetic stays float32.
 * Both flags at once, or any other bit above the low 8, is IRIS_ERR_INVALID (as it is for a library
 * that predates the flags, so callers can detect support). */
enum { IRIS_OUT_BF16 = 0x100, IRIS_OUT_F16 = 0x200 };

enum { IRIS_REMAP_NONE = 0, IRIS_REMAP_STEREO_MONO = 1, IRIS_REMAP_MERGE_AUG = 2, IRIS_REMAP_MONO_CHAN = 3 };
/* IRIS_REMAP_MONO_CHAN: data_utils.mono_chan (data_utils.py:73-76) of a 2-channel plan, n_out_chan = 2.  Its
 * broadcast quirk x[..., :1] + x[..., 1:] makes the complex spectrogram the 3 columns [re0 + re1, re0 + im0,
 * re0 + im1] (IRIS_FEAT_COMPLEX: [B,257,T,3]); complex_to_magphase then broadcasts the one real column
 * against the two imaginary ones (transforms.py:111-123), so every later mode sees C' = 2 pseudo-channels
 * z_j = (re0 + re1) + i (re0 + im_j): magnitude + phase [B,257,T,4], mel [B,n_mel,T,2].  Masks act on the
 * inputs, stft_filter on the sums.  A library without it answers the plan with IRIS_ERR_INVALID (n_out_chan
 * below 3), so callers can probe for it. */

int iris_abi_version(void);
const char* iris_last_error(void);

int iris_ctx_create(int device, iris_ctx** out);
int iris_ctx_destroy(iris_ctx* ctx);

/* Mel weights: dense [n_bins=257, n_mel] row-major host array, i.e. the matrix
 * tf.signal.linear_to_mel_weight_matrix returns at transforms.py:55-56.  Stored sparse. */
int iris_set_mel(iris_ctx* ctx, int n_mel, int n_bins, const float* dense_w);

/* The reference's own bank format (utils.load_data, utils.py:88-94; consumed by
 * pipeline.make_pipeline, pipeline.py:113-175): a list of pre-computed complex spectrograms
 * [257, t_i, 2 * chan] ([..., :chan] = re, [..., chan:] = im), packed back to back in `specs`
 * (host or device memory); frame_offsets [n_items + 1] = cumulative t_i.  Banks registered this
 * way are mixed in the spectrogram domain with pipeline.merge_complex_specs' arithmetic
 * (pipeline.py:29-106); frame activity is `max over (freq, chan2) > 0` (pipeline.py:55).  All
 * three banks of a plan must be of the same format. */
int iris_specbank_register(iris_ctx* ctx, int kind, int n_items, int n_freq, int n_chan2,
                           const float* specs, const int64_t* frame_offsets, const float* labels,
                           int n_classes, iris_stream stream);
/* Register a bank of WAVEFORMS (replaces data_utils.load_wav, data_utils.py:9-29, for every
 * source: normalize (32-34) + reflect padding now, STFT inside iris_features).
 *   packed_wav : item i is the [n_chan, len_i] row-major block starting at float
 *                n_chan * offsets[i]; host or device pointer.
 *   offsets    : [n_items+1] cumulative per-channel sample counts (host).
 *   labels     : [n_items, n_classes] host floats (one-hot rows) for the VOICE bank, else NULL.
 * For the VOICE bank the per-frame activity flags (reduce_max(voice) > 0, pipeline.py:55)
 * are computed here by one STFT pass.  Synchronises the stream before returning. */
int iris_bank_register(iris_ctx* ctx, int kind, int n_items, int n_chan, const float* packed_wav,
                       const int64_t* offsets, const float* labels, int n_classes, int normalize,
                       iris_stream stream);
/* The same from audio at any sample rate, as load_wav reads it (data_utils.py:19-22): item i is
 * [n_chan, len_i] at sample_rates[i] Hz (host, >= 1), packed and counted by `offsets` as above.  Every
 * item not at 16 kHz is resampled to 16 kHz with iris_resample's filter (Kaldi LinearResample) by one
 * device pass over the bank; the 16 kHz items are then registered exactly as iris_bank_register
 * registers them (normalize over the resampled item, layout, activity), so iris_bank_info reports the
 * frames of the iris_resample_len lengths and a bank whose rates are all 16000 is registered bit for
 * bit as by iris_bank_register.  A rate pair whose filter bank exceeds 32 MB is IRIS_ERR_UNSUPPORTED.
 * Added under IRIS_ABI_VERSION 2: callers probe for the symbol. */
int iris_bank_register_audio(iris_ctx* ctx, int kind, int n_items, int n_chan, const float* packed_wav,
                             const int64_t* offsets, const int32_t* sample_rates, const float* labels,
                             int n_classes, int normalize, iris_stream stream);
int iris_bank_info(iris_ctx* ctx, int kind, int32_t* n_items, int32_t* n_chan,
                   int32_t* n_frames /* [n_items] or NULL */);
int iris_bank_activity(iris_ctx* ctx, int item, uint8_t* host_out /* [n_frames[item]] */);

/* All random draws of one batch, made by the HOST in the reference's draw order
 * (SURVEY.md 3.1): everything tf.random supplies inside merge_complex_specs
 * (pipeline.py:35,43,50,69,87,94,103), mask (transforms.py:25-26) and random_merge_aug
 * (data_utils.py:109).  Arrays are host pointers, row-major. */
typedef struct iris_plan {
    int32_t batch;        /* B */
    int32_t n_frame;      /* T   (make_pipeline n_frame)                                   */
    int32_t max_voices;   /* V   padded_batch group size (pipeline.py:155); 0 = no voices  */
    int32_t max_noises;   /* M   (pipeline.py:165); 0 = no noises                          */
    float min_ratio;      /* merge_complex_specs min_ratio (sj_train passes 1)             */
    float min_noise_ratio;
    const int32_t* bg_id;        /* [B]                                                    */
    const int32_t* bg_offset;    /* [B]   random_crop offset into the tiled background     */
    const int32_t* n_voices;     /* [B]   in [1, V)  (V == 1: 1)                           */
    const int32_t* voice_id;     /* [B,V] the whole group (its longest member pads all)    */
    const float* voice_gain;     /* [B,V] pow(10, -u), u ~ U[0, -snr/10)                   */
    const int32_t* voice_offset; /* [B,V] in [0, len - T)                                  */
    const int32_t* n_noises;     /* [B]   in [0, M)                                        */
    const int32_t* noise_id;     /* [B,M]                                                  */
    const float* noise_gain;     /* [B,M] pow(10, -u), u ~ U[0, 2)                         */
    const int32_t* noise_offset; /* [B,M] in [0, len - T]                                  */
    int32_t n_time_masks;        /* augment: 6 (data_utils.py:59)                          */
    int32_t n_freq_masks;        /* augment: 1 (data_utils.py:60)                          */
    const int32_t* time_masks;   /* [B,n_time_masks,2] (size, offset) or NULL              */
    const int32_t* freq_masks;   /* [B,n_freq_masks,2] (size, offset) or NULL              */
    int32_t stft_filter;         /* zero bins 1..k (data_utils.py:126-136); 0 = off        */
    int32_t chan_remap;          /* IRIS_REMAP_*  (data_utils.py:79-82, 100-117)           */
    int32_t n_out_chan;          /* channels after remap (3 for stereo_mono, 2 for mono_chan) */
    const float* merge_factor;   /* [B, n_out_chan-2] U(0.1, 0.9), REMAP_MERGE_AUG only    */
} iris_plan;

/* Validates the draws against the registered banks with the reference's placement
 * arithmetic (pipeline.py:29-35, 58-74, 95-103) and uploads the batch plan. */
int iris_plan_upload(iris_ctx* ctx, const iris_plan* plan, iris_stream stream);

/* Labels of merge_complex_specs (pipeline.py:41-84): same-class overlap rejection and
 * per-voice frame labels, then to_frame_labels (data_utils.py:64-70).
 *   d_labels_vtk   : [B,V,T,K] float or NULL      (make_pipeline's label output)
 *   d_frame_labels : [B,T,K]   float or NULL      (after to_frame_labels)
 *   d_keep         : [B,V]     uint8 or NULL      (no_overlap flag per voice slot) */
int iris_labels(iris_ctx* ctx, float* d_labels_vtk, float* d_frame_labels, uint8_t* d_keep,
                iris_stream stream);

/* The fused feature kernel for the uploaded plan; d_out sized per the mode's layout, 16-byte aligned.
 * mode: IRIS_FEAT_* | optional IRIS_OUT_BF16 / IRIS_OUT_F16, in which case d_out points at 2-byte
 * elements (bfloat16 / float16) in the same layout. */
int iris_features(iris_ctx* ctx, int mode, float* d_out, iris_stream stream);

/* merge_complex_specs(seperate_noise_voice=True) (pipeline.py:37-38, 82-83, 104-108): the same
 * mix restricted to a subset of the sources, as a plain complex spectrogram [B,257,T,2C] (no
 * masks, remap or filter: these are labels of the 'se' model, sj_train.py:99-105).
 *   IRIS_SELECT_VOICES   only_voice = sum of the accepted voices
 *   IRIS_SELECT_BG_NOISE only_noise = background + noises
 * IRIS_SELECT_ALL is iris_features().  mode (IRIS_FEAT_COMPLEX for a selection) takes the
 * IRIS_OUT_* flags as iris_features does, d_out then holding 2-byte elements. */
enum { IRIS_SELECT_ALL = 0, IRIS_SELECT_VOICES = 1, IRIS_SELECT_BG_NOISE = 2 };
int iris_features_select(iris_ctx* ctx, int mode, int select, float* d_out, iris_stream stream);

/* data_utils.load_wav on one in-memory waveform (data_utils.py:9-29 minus decode/resample):
 * wav [n_chan, n_samples] (host or device) -> d_out [257, 1 + n_samples/256, 2*n_chan]. */
int iris_stft(iris_ctx* ctx, const float* wav, int n_chan, int64_t n_samples, int normalize,
              float* d_out, iris_stream stream);

/* metrics.er_score(smoothing=False) integer core (metrics.py:217-266) and tfa F1Score
 * micro counts (metrics.py:290-298) for y_true, y_pred [B,T,K] device floats.
 *   d_triples : [B,3] int32  (n_true, n_pred, correct)
 *   d_tpfpfn  : [3]   uint64 ACCUMULATED (the reference's F1 metric is never reset), or NULL
 *   d_sums    : [3]   uint64 ACCUMULATED batch totals of the triples (together with d_tpfpfn
 *                     the payload of the multi-GPU count all-reduce), or NULL
 *   d_er      : [B]   float  score per sample (metrics.py:268-273), or NULL */
int iris_metric_counts(iris_ctx* ctx, const float* d_y_true, const float* d_y_pred, int batch,
                       int n_frame, int n_classes, float threshold, int32_t* d_triples,
                       uint64_t* d_tpfpfn, uint64_t* d_sums, float* d_er, iris_stream stream);

/* metrics.er_score(smoothing=True) (metrics.py:217-274): y_pred has already been average-pooled
 * with AveragePooling1D(31, padding='same') -- strides default to the pool size, so it holds
 * n_frame_pred = ceil(n_frame / 31) frames -- and the reference matches the midpoints of the
 * pooled events against the un-pooled true events by their raw frame indices (metrics.py:256-266).
 * Same integer core as iris_metric_counts with the two time bases kept apart; no F1 counts.
 *   d_y_true [B, n_frame, K], d_y_pred [B, n_frame_pred, K]; d_triples [B,3]; d_er [B] or NULL */
int iris_er_counts_pooled(iris_ctx* ctx, const float* d_y_true, int n_frame, const float* d_y_pred,
                          int n_frame_pred, int batch, int n_classes, float threshold,
                          int32_t* d_triples, float* d_er, iris_stream stream);

/* Algorithmic HBM bytes of the last uploaded plan for `mode` (SURVEY.md 8d): 4 * samples of
 * every kept source frame range read, plus 4 (2 with an IRIS_OUT_* flag in `mode`) * output
 * elements; used by bench.py's roofline. */
int iris_plan_bytes(iris_ctx* ctx, int mode, const uint8_t* host_keep, int64_t* bytes_in,
                    int64_t* bytes_out);
/* The same for the clips [clip_lo, clip_hi) of the plan. */
int iris_plan_bytes_clips(iris_ctx* ctx, int mode, const uint8_t* host_keep, int clip_lo, int clip_hi,
                          int64_t* bytes_in, int64_t* bytes_out);

/* Debug / test hook (no device needed): the work-claim schedule a k_fused launch of n_tiles tiles on `grid`
 * persistent CTAs gets -- schedule5 = {chunk, chunk_mid, chunk_tail, n_big, n_mid} -- and the tile range of
 * claim q under it (first >= n_tiles: no work left).  tests/test_host_logic.py checks that the claims
 * cover every tile exactly once. */
int iris_debug_claims(int64_t n_tiles, int grid, int chunk, int pair_merge, int64_t q, int32_t* schedule5,
                      int64_t* first, int32_t* len);
/* Measurement hook for bench.py's roofline: when enabled, every launch of the fused
 * feature kernel inside iris_features() is bracketed by cudaEvents on the launching stream;
 * iris_profile_read() synchronises them and returns the summed device time. */
int iris_profile_enable(iris_ctx* ctx, int enable);
int iris_profile_read(iris_ctx* ctx, double* total_ms, int32_t* n_launches, int reset);
/* Clips of the launch the hook timed last (the whole batch of that feature launch). */
int iris_profile_clips(iris_ctx* ctx);

/* ---------------------------------------------------------------------------------------
 * Stand-alone stages: the reference's public functions applied one at a time (what a
 * tf.data `.map(fn)` of a single function binds to).  The fused iris_features() path above
 * is the hot path; these are its stages un-fused, for callers that compose the reference's
 * functions in an order the fused kernel does not cover.  x / out are DEVICE fp32 tensors,
 * C-contiguous, out may alias x unless noted.  Small parameter arrays are HOST pointers.
 * --------------------------------------------------------------------------------------- */

/* transforms.mask (transforms.py:12-40): x viewed as [outer, n_axis, inner]; masks = n_mask
 * host pairs (size, offset) in draw order (transforms.py:25-26); out = x * mask (product,
 * signed zeros kept).  Also data_utils.augment (data_utils.py:58-61) = two calls. */
int iris_op_mask(iris_ctx* ctx, const float* d_x, float* d_out, int64_t outer, int64_t n_axis,
                 int64_t inner, const int32_t* masks, int n_mask, iris_stream stream);
/* data_utils.stft_filter(k) (data_utils.py:126-136): x [n_bins, inner], bins 1..k times 0. */
int iris_op_stft_filter(iris_ctx* ctx, const float* d_x, float* d_out, int64_t n_bins,
                        int64_t inner, int k, iris_stream stream);
/* transforms.random_shift (transforms.py:43-47): zero-pad `width` both sides of the axis and
 * crop at `offset` in [0, 2*width].  out must NOT alias x. */
int iris_op_random_shift(iris_ctx* ctx, const float* d_x, float* d_out, int64_t outer,
                         int64_t n_axis, int64_t inner, int width, int offset, iris_stream stream);
/* Row-wise stages on [rows, 2*n_chan] (first half real / magnitude, second imag / phase). */
enum {
    IRIS_PW_COMPLEX_TO_MAGPHASE = 0, /* transforms.py:111-123; width 3 (mono_chan's [re, im0, im1]) is
                                        TF's broadcast of re against both: rows of 4 (out must NOT
                                        alias x), other odd widths are IRIS_ERR_INVALID */
    IRIS_PW_MAGPHASE_TO_COMPLEX = 1, /* transforms.py:126-134 */
    IRIS_PW_LOG_MAGPHASE = 2,        /* transforms.py:80-86; `param_i` = n_chan argument      */
    IRIS_PW_LOG_ON_MEL = 3,          /* data_utils.py:50-55; any shape, pass width = 1        */
    IRIS_PW_MULTIPLY = 4             /* data_utils.py:120-123; `param_f` = multiply_factor    */
};
/* data_utils.normalize (data_utils.py:32-34): d_out = d_x / (10 * sqrt(mean(d_x^2))) over all n
 * elements (every channel and sample of one clip); squares summed in fp64, the rest in fp32 as in
 * the bank registration.  In place is allowed. */
int iris_op_normalize(iris_ctx* ctx, const float* d_x, float* d_out, int64_t n, iris_stream stream);
int iris_op_pointwise(iris_ctx* ctx, int op, const float* d_x, float* d_out, int64_t rows,
                      int width, int param_i, float param_f, iris_stream stream);
/* Channel remaps on [rows, w_in] -> [rows, w_out] (out must NOT alias x):
 *   mono_chan (data_utils.py:73-76; w_out = w_in - 1, the reference's broadcast quirk),
 *   stereo_mono (79-82; 4 -> 6), random_merge_aug(number) (100-117; 4 -> 2*number, `factor`
 *   = host [n_samples, number-2] draws of U(0.1, 0.9), rows_per_sample rows per sample). */
enum { IRIS_MAP_MONO_CHAN = 0, IRIS_MAP_STEREO_MONO = 1, IRIS_MAP_MERGE_AUG = 2 };
int iris_op_chan_map(iris_ctx* ctx, int kind, const float* d_x, float* d_out, int64_t rows,
                     int w_in, int w_out, const float* factor, int64_t n_samples,
                     int64_t rows_per_sample, iris_stream stream);
/* transforms.magphase_to_mel (transforms.py:51-77) with the matrix of iris_set_mel (any
 * matrix): x [B, n_bins, T, 2C] -> out [B, n_mel, T, C] (unbatched: B = 1). */
int iris_op_mel(iris_ctx* ctx, const float* d_x, float* d_out, int B, int T, int n_chan,
                iris_stream stream);
/* data_utils.minmax (data_utils.py:37-47, safe_div utils.py:114-116): variant 0, one group;
 * transforms.minmax_norm_magphase (transforms.py:89-107): variant 1, the two halves of the
 * last axis (width) normalised separately.  x [n_samples, per_sample]. */
int iris_op_minmax(iris_ctx* ctx, int variant, const float* d_x, float* d_out, int64_t n_samples,
                   int64_t per_sample, int width, iris_stream stream);
/* data_utils.to_frame_labels (data_utils.py:64-70): y [outer, V, inner] -> [outer, inner]. */
int iris_op_sum_voices(iris_ctx* ctx, const float* d_y, float* d_out, int64_t outer, int V,
                       int64_t inner, iris_stream stream);
/* AveragePooling1D(r, r, 'same') over time of y [B, T, K] -> [B, ceil(T/r), K];
 * binarize != 0 adds the `>= 0.5` of data_utils.label_downsample (data_utils.py:85-97; the
 * `[:resolution]` batch slice is the caller's), binarize == 0 is the smoothing pool of
 * metrics.er_score (metrics.py:222-224). */
int iris_op_avg_pool_time(iris_ctx* ctx, const float* d_y, float* d_out, int B, int T, int K, int r,
                          int binarize, iris_stream stream);
/* metrics.cos_sim (metrics.py:277-287): y_true, y_pred [B, T, K<=8] -> out [B]. */
int iris_op_cos_sim(iris_ctx* ctx, const float* d_y_true, const float* d_y_pred, float* d_out,
                    int B, int T, int K, iris_stream stream);


/* transforms.phase_vocoder (transforms.py:137-195), SURVEY.md 8f rank 3: x [n_freq, T, 2*chan]
 * -> out [n_freq, T_out, 2*chan].  idx0 / idx1 / alpha are HOST arrays [T_out] with the
 * reference's time-step arithmetic: steps = tf.range(0, T, rate), idx0 = int32(steps),
 * idx1 = int32(steps + 1) (frames T, T + 1 are the zero padding), alpha = steps % 1. */
int iris_op_phase_vocoder(iris_ctx* ctx, const float* d_x, float* d_out, int n_freq, int T, int n_chan,
                          int T_out, const int32_t* idx0, const int32_t* idx1, const float* alpha,
                          iris_stream stream);

/* torchaudio.compliance.kaldi.resample_waveform(wav, orig_freq, new_freq) as load_wav calls it
 * (data_utils.py:20-21; Kaldi LinearResample, lowpass_filter_width 6, cutoff 0.99 * Nyquist of the
 * lower rate).  wav [n_chan, n_in] host or device -> d_out [n_chan, iris_resample_len(...)]. */
int64_t iris_resample_len(int64_t n_in, int orig_freq, int new_freq);
int iris_resample(iris_ctx* ctx, const float* wav, int n_chan, int64_t n_in, int orig_freq, int new_freq,
                  float* d_out, iris_stream stream);

/* ---- trainer.py label variants (trainer.py:86-104), SURVEY.md 8f rank 4 ---- */
/* One stage of trainer.preprocess_labels: avg_pool1d(y, 2, 2, 'SAME') * 2 (* scale) on
 * y [B, T, K] -> out [B, ceil(T/2), K]; a lone last cell is doubled (TF averages over the
 * valid cells). */
int iris_op_sum_pool2(iris_ctx* ctx, const float* d_y, float* d_out, int B, int T, int K, float scale,
                      iris_stream stream);
/* trainer.to_density_labels: y [outer, V, inner = T*K] -> out [outer, inner]: every voice
 * divided by max(its total, 1e-8) (utils.safe_div), summed over the voices. */
int iris_op_density_labels(iris_ctx* ctx, const float* d_y, float* d_out, int64_t outer, int V,
                           int64_t inner, iris_stream stream);

/* ---- evaluation-side chain of metrics.evaluate (metrics.py:40-90), SURVEY.md 8f rank 1 ---- */
/* metrics.py:60-61: tf.signal.frame(x, frame_len, step, pad_end=True, axis=-2) + transpose
 * (1, 0, 2, 3).  x [outer, T, inner] -> out [n_win, outer, frame_len, inner] with
 * n_win = ceil(T / step) (checked), zeros past the end. */
int iris_op_eval_windows(iris_ctx* ctx, const float* d_x, float* d_out, int64_t outer, int64_t T,
                         int64_t inner, int frame_len, int step, int n_win, iris_stream stream);
/* metrics.py:67-75: UpSampling1D(up) + overlap_and_add(preds) / overlap_and_add(ones) +
 * [..., :L].  preds [n_win, n_p, K] -> out [L, K]; L <= (n_win - 1) * step + n_p * up. */
int iris_op_eval_merge(iris_ctx* ctx, const float* d_preds, float* d_out, int n_win, int n_p, int K,
                       int up, int step, int L, iris_stream stream);
/* metrics.py:77-81: AveragePooling1D(k_avg, 1, 'same') -> MaxPooling1D(k_max, 1, 'same') ->
 * `>= threshold` as 0/1 floats.  x, out [L, K]; d_tmp [L, K] scratch. */
int iris_op_eval_smooth(iris_ctx* ctx, const float* d_x, float* d_tmp, float* d_out, int L, int K,
                        int k_avg, int k_max, float threshold, iris_stream stream);
/* Challenge_Metric.get_start_end_frame + output_to_metric (metrics.py:109-133, 196-214).
 * y [L, K<=8].  d_rows int32 [max_rows, 4] = (class, start, end, int32(((start + end) / 2) *
 * hop / sr)) ordered by class then time; d_n_rows int32 [1 + K] = total events (may exceed
 * max_rows: rows beyond it are dropped), events per class. */
int iris_op_eval_events(iris_ctx* ctx, const float* d_y, int L, int K, int hop, int sr,
                        int32_t* d_rows, int max_rows, int32_t* d_n_rows, iris_stream stream);
/* metrics.get_er (metrics.py:176-193).  d_gt int32 [m, 3] (class, start, end); d_pred int32 rows
 * of pred_stride ints with the class in column 0 and the time in column pred_time_col
 * ([n, 2] tensor: stride 2, column 1; rows of iris_op_eval_events: stride 4, column 3);
 * n = *d_n_pred (clamped to n_pred_max) or n_pred_max if d_n_pred is NULL.
 * d_out int32 [3] = (N = n + m, answer = 2 * matches, m); ER = (N - answer) / m. */
int iris_op_get_er(iris_ctx* ctx, const int32_t* d_gt, int m, const int32_t* d_pred, int pred_stride,
                   int pred_time_col, const int32_t* d_n_pred, int n_pred_max, int32_t* d_out,
                   iris_stream stream);

/* ---------------------------------------------------------------------------------------
 * One call per batch (round 2).  The reference builds a batch with ~B * (V + M + 10) tf.random
 * draws inside merge_complex_specs / mask / random_merge_aug and ~10 Python-level tf.data stages
 * (pipeline.py:113-175, sj_train.py:92-130).  Here the caller supplies ONE block of host
 * uniforms per batch (randomness stays host-generated and explicit); iris_draw_batch turns it
 * into the draws of an iris_plan with the reference's placement arithmetic, and iris_step runs
 * draws -> plan upload -> labels -> features (-> metric counts -> count all-reduce) from C.
 * --------------------------------------------------------------------------------------- */

/* Dataset.from_generator(items).repeat().shuffle(buffer_size) as a stream of item ids
 * (pipeline.py:143-147, 149-154, 159-164): a buffer fed by the endlessly repeated sequence
 * 0..n-1; every draw emits slot floor(u * buffer_size) and refills it.  Host-only state. */
typedef struct iris_shuffle iris_shuffle;
int iris_shuffle_create(int n_items, int buffer_size, iris_shuffle** out);
int iris_shuffle_destroy(iris_shuffle* s);
int iris_shuffle_take(iris_shuffle* s, const double* uniforms, int k, int32_t* out_ids);

typedef struct iris_draw_config {
    int32_t batch;            /* B */
    int32_t n_frame;          /* T */
    int32_t max_voices;       /* V (0: none) */
    int32_t max_noises;       /* M (0: none) */
    float min_ratio;          /* merge_complex_specs min_ratio (pipeline.py:12) */
    float min_noise_ratio;    /* (pipeline.py:13) */
    float snr;                /* (pipeline.py:14): voice gain 10^-u, u ~ U[0, -snr/10) */
    int32_t n_time_masks;     /* augment: 6 masks below time_mask_max = 24 (data_utils.py:59) */
    int32_t time_mask_max;
    int32_t n_freq_masks;     /* augment: 1 mask below freq_mask_max = 16 (data_utils.py:60) */
    int32_t freq_mask_max;
    int32_t n_bins;           /* 257 */
    int32_t merge_extra;      /* random_merge_aug(number): number - 2 factors (data_utils.py:109) */
} iris_draw_config;

/* Uniforms one clip consumes, in the reference's per-clip draw order (SURVEY.md 3.1):
 *   bg id, bg crop offset (pipeline.py:35), V voice ids, n_voices (43), V x {gain u (50),
 *   offset (69)}, M noise ids, n_noises (87), M x {gain u (94), crop offset (103)},
 *   n_time_masks x {size (transforms.py:25), offset (26)}, n_freq_masks x {size, offset},
 *   merge_extra factors.  Integers are floor(u * range); ids come from the shuffle streams
 *   when given. */
int iris_draw_uniforms_per_clip(const iris_draw_config* cfg);

/* Caller-allocated HOST outputs of iris_draw_batch; shapes as in iris_plan.  voice_u / noise_u
 * are the raw fp32 exponent draws (gain = powf(10, -u)); rows behind n_voices / n_noises are
 * zero (gain 1).  Pointers of absent parts (V == 0, no masks, ...) may be NULL. */
typedef struct iris_draws {
    int32_t* bg_id;        int32_t* bg_offset;
    int32_t* n_voices;     int32_t* voice_id;   float* voice_u;  float* voice_gain;  int32_t* voice_offset;
    int32_t* n_noises;     int32_t* noise_id;   float* noise_u;  float* noise_gain;  int32_t* noise_offset;
    int32_t* time_masks;   int32_t* freq_masks;
    float* merge_factor;
} iris_draws;

/* Host-only (no device needed): uniforms [batch, iris_draw_uniforms_per_clip] in [0, 1) ->
 * draws.  *_frames are the frame counts of the bank items (1 + n_samples / 256, or the
 * spectrogram lengths); streams[kind] may be NULL (ids = floor(u * n_items)).  Returns
 * IRIS_ERR_EMPTY_RANGE where the reference's int-uniform would raise (pipeline.py:68-69). */
int iris_draw_batch(const iris_draw_config* cfg, const int32_t* bg_frames, int n_bg,
                    const int32_t* voice_frames, int n_voice, const int32_t* noise_frames, int n_noise,
                    iris_shuffle* const* streams /* [3] or NULL */, const double* uniforms,
                    iris_draws* out);

typedef struct iris_step_config {
    iris_draw_config draw;
    int32_t stft_filter;      /* data_utils.stft_filter(k); 0 = off */
    int32_t chan_remap;       /* IRIS_REMAP_* */
    int32_t n_out_chan;       /* channels after remap */
    int32_t feature_mode;     /* IRIS_FEAT_* | optional IRIS_OUT_BF16 / IRIS_OUT_F16 */
} iris_step_config;

typedef void* iris_nccl_comm; /* ncclComm_t */

typedef struct iris_step_io {
    const double* uniforms;   /* HOST [batch, iris_draw_uniforms_per_clip(&cfg->draw)] */
    iris_shuffle* const* streams; /* [3] (bg, voice, noise) or NULL */
    float* d_features;        /* DEVICE, layout of cfg->feature_mode, 16-byte aligned; 2-byte
                                 elements with an IRIS_OUT_* flag */
    float* d_frame_labels;    /* DEVICE [B,T,K] or NULL (to_frame_labels, data_utils.py:64-70) */
    float* d_labels_vtk;      /* DEVICE [B,V,T,K] or NULL (make_pipeline's label output) */
    uint8_t* d_keep;          /* DEVICE [B,V] or NULL */
    /* optional metric leg on this step's frame labels (metrics.py:217-298), enqueued on the
     * context's own side stream.  For IRIS_FEAT_LOGMEL_MINMAX it forks behind the feature kernel and
     * runs beside the second pass (the labels and the feature kernel stay adjacent in `stream`, and the
     * persistent feature grid finds every SM free); for the other modes it forks right behind the
     * labels kernel and runs beside the feature kernel: */
    const float* d_y_pred;    /* DEVICE [B,T,K] model output, or NULL: no metric leg */
    float threshold;          /* 0.5 */
    int32_t* d_triples;       /* DEVICE [B,3] (n_true, n_pred, correct) of the local clips; with a
                                 communicator: this rank's slice of a [B_global,3] send buffer whose
                                 other rows stay zero (pass send + 3 * clip_lo) */
    uint64_t* d_counts;       /* DEVICE [6] TP, FP, FN, sum n_true, sum n_pred, sum correct (accumulated) */
    iris_nccl_comm comm;      /* not NULL: iris_allreduce_counts on the side stream after the counting */
    int64_t* d_counts_reduced;   /* DEVICE [6] all-reduced copy of d_counts (with comm) */
    const int32_t* d_triples_send;  /* DEVICE [B_global,3] (see d_triples) or NULL */
    int32_t* d_triples_global;      /* DEVICE [B_global,3] all-reduced triples or NULL */
    int32_t global_batch;
} iris_step_io;

/* One batch.  Everything is enqueued on `stream` (the metric leg on the context's side stream,
 * ordered behind the labels kernel); returns when the launches are queued.  The labels kernel also
 * builds the per-tile stage lists of the feature kernel (the keep flags it decides are their only
 * input that is not in the plan), so a step is plan upload -> k_labels -> k_fused (-> k_logmel_post).  The host blocks only
 * when it is more than four batches ahead of the device (ring of pinned plan buffers). */
int iris_step(iris_ctx* ctx, const iris_step_config* cfg, const iris_step_io* io, iris_stream stream);
/* Make `stream` wait for the metric leg (counts and their all-reduce) issued `lag` iris_step
 * calls ago (0 = the latest).  The reduced counts are a logged metric (the reference reads them
 * once per epoch, sj_train.py:454-462), so a training loop waits with lag >= 1 and the collective
 * never stalls the feature kernels. */
int iris_counts_wait(iris_ctx* ctx, int lag, iris_stream stream);
/* The draws iris_step made for its last batch (host pointers owned by the context, valid until
 * the next iris_step): what the parity oracle consumes. */
int iris_step_draws(iris_ctx* ctx, iris_draws* out);

/* The path's only exchange (SURVEY.md 8e): NCCL sum over NVLink / NVSwitch of the int64 count
 * vector [TP, FP, FN, sum n_true, sum n_pred, sum correct] and -- because the reference's ER is a
 * mean of per-sample ratios clipped at the batch-global max(n_true) (metrics.py:268-273) -- of the
 * per-sample triples: every rank fills its slice of a zero-initialised [B_global,3] int32 buffer
 * (sum over disjoint slices == all-gather, ragged shards included).  Both reductions are one NCCL
 * group on `stream`.  d_triples_* may be NULL.  NCCL is resolved at run time from the process
 * (the library the framework already loaded) or from libnccl.so.2. */
int iris_allreduce_counts(iris_ctx* ctx, iris_nccl_comm comm, const int64_t* d_counts_send,
                          int64_t* d_counts_recv, const int32_t* d_triples_send,
                          int32_t* d_triples_recv, int global_batch, iris_stream stream);
/* Communicator plumbing for callers that do not own an ncclComm_t: rank 0 makes an id
 * (128 bytes), every rank joins with it. */
int iris_nccl_unique_id(void* out_id_128);
int iris_nccl_comm_create(iris_ctx* ctx, const void* id_128, int rank, int world_size, iris_nccl_comm* out);
int iris_nccl_comm_destroy(iris_nccl_comm comm);
/* metrics.py:268-273 on already reduced triples [n,3] -> er [n] (the denominator clips at the
 * batch-global max(n_true)). */
int iris_er_from_triples(iris_ctx* ctx, const int32_t* d_triples, int n, float* d_er, iris_stream stream);

/* Pinned host memory on the NUMA node of the context's GPU (mmap + mbind + cudaHostRegister):
 * staging for the device -> host read-back of features on multi-socket boxes where every rank's
 * default allocations land on one node.  *numa_node receives the node used (-1: not bound). */
int iris_host_alloc(iris_ctx* ctx, size_t bytes, void** out, int* numa_node);
int iris_host_free(iris_ctx* ctx, void* p, size_t bytes);

/* ---- DLPack hand-over (the exchange format north_star names) ----
 * `managed` points at a DLManagedTensor (dlpack.h ABI: the struct behind the "dltensor"
 * capsule of torch.utils.dlpack.to_dlpack / tf.experimental.dlpack.to_dlpack).  The entry points
 * check device, dtype, contiguity and shape against the plan and then write through
 * data + byte_offset: the tensor stays owned by the producing framework, nothing is copied.  The
 * dtype is float32 except for features with an IRIS_OUT_* flag in `mode` / cfg->feature_mode:
 * bfloat16 (kDLBfloat, 16 bits) for IRIS_OUT_BF16, float16 (kDLFloat, 16 bits) for IRIS_OUT_F16.  A
 * dtype that does not match the flag is IRIS_ERR_INVALID and nothing is written. */
int iris_features_dlpack(iris_ctx* ctx, int mode, void* managed, iris_stream stream);
int iris_labels_dlpack(iris_ctx* ctx, void* managed_vtk, void* managed_frame, iris_stream stream);
int iris_step_dlpack(iris_ctx* ctx, const iris_step_config* cfg, const double* uniforms,
                     iris_shuffle* const* streams, void* managed_features, void* managed_frame_labels,
                     iris_stream stream);
/* Whether iris_set_mel's matrix runs in the fused epilogue (else: IRIS_FEAT_MAGPHASE +
 * iris_op_mel), and the most mixing segments one clip may have in the fused kernel. */
int iris_mel_fusable(iris_ctx* ctx);
/* Bytes of the last plan blob copied host -> device (iris_plan_upload / iris_step). */
int64_t iris_plan_upload_bytes(iris_ctx* ctx);
int iris_max_segments(void);

#ifdef __cplusplus
}
#endif
#endif /* IRIS_H_ */
