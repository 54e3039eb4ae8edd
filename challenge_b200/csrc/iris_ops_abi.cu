// extern "C" surface of the stand-alone stages (include/iris.h, second half): argument
// checks, tiny host->device parameter uploads, kernel launches (k_ops.cu).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "iris_ctx.h"

using namespace iris;

namespace {

// small per-call parameters go through a pinned-free path: cudaMemcpyAsync from pageable host
// memory stages the bytes before returning, so stack / vector sources are safe
int upload_small(iris_ctx* c, const void* h, size_t bytes, cudaStream_t st, void** d) {
    // ring of 64 KB slices so that back-to-back ops on one stream do not overwrite each other
    const size_t slice = 64 * 1024, n_slices = 16;
    if (bytes > slice) return fail(IRIS_ERR_UNSUPPORTED, "parameter block larger than 64 KB");
    CU(c->op_small.reserve(slice * n_slices));
    static thread_local unsigned cursor = 0;
    char* p = c->op_small.as<char>() + slice * (cursor++ % n_slices);
    CU(cudaMemcpyAsync(p, h, bytes, cudaMemcpyHostToDevice, st));
    *d = p;
    return IRIS_OK;
}

int begin(iris_ctx* c) {
    if (!c) return fail(IRIS_ERR_INVALID, "NULL ctx");
    return iris_set_device(c);
}

}  // namespace

extern "C" {

int iris_op_mask(iris_ctx* c, const float* x, float* out, int64_t outer, int64_t n_axis,
                 int64_t inner, const int32_t* masks, int n_mask, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || outer < 0 || n_axis < 1 || inner < 1 || n_mask < 0 || (n_mask && !masks))
        return fail(IRIS_ERR_INVALID, "iris_op_mask: bad argument");
    if (n_axis > 16000) return fail(IRIS_ERR_UNSUPPORTED, "iris_op_mask: axis longer than 16000");
    std::vector<float> m(size_t(n_axis), 1.f);
    for (int i = 0; i < n_mask; ++i) {
        const int64_t size = masks[2 * i], off = masks[2 * i + 1];
        // tf.random.uniform(maxval=total-size) raises on an empty range (transforms.py:26)
        if (size < 0 || size >= n_axis + 1 || off < 0 || off + size > n_axis)
            return fail(IRIS_ERR_INVALID, "iris_op_mask: mask outside the axis");
        for (int64_t a = off; a < off + size; ++a) m[size_t(a)] *= 0.f;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    void* dm;
    rc = upload_small(c, m.data(), m.size() * 4, st, &dm);
    if (rc) return rc;
    CU(launch_axis_scale(x, static_cast<float*>(dm), out, size_t(outer), size_t(n_axis), size_t(inner), st));
    return IRIS_OK;
}

int iris_op_stft_filter(iris_ctx* c, const float* x, float* out, int64_t n_bins, int64_t inner, int k,
                        iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || n_bins < 1 || inner < 1 || k < 0 || k + 1 > n_bins)
        return fail(IRIS_ERR_INVALID, "iris_op_stft_filter: bad argument");
    if (n_bins > 16000) return fail(IRIS_ERR_UNSUPPORTED, "iris_op_stft_filter: too many bins");
    std::vector<float> m(size_t(n_bins), 1.f);
    for (int f = 1; f <= k; ++f) m[f] = 0.f;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    void* dm;
    rc = upload_small(c, m.data(), m.size() * 4, st, &dm);
    if (rc) return rc;
    CU(launch_axis_scale(x, static_cast<float*>(dm), out, 1, size_t(n_bins), size_t(inner), st));
    return IRIS_OK;
}

int iris_op_random_shift(iris_ctx* c, const float* x, float* out, int64_t outer, int64_t n_axis,
                         int64_t inner, int width, int offset, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || x == out || outer < 0 || n_axis < 1 || inner < 1 || width < 0 || offset < 0 ||
        offset > 2 * width)
        return fail(IRIS_ERR_INVALID, "iris_op_random_shift: bad argument");
    CU(launch_axis_shift(x, out, size_t(outer), size_t(n_axis), size_t(inner), offset - width,
                         static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_pointwise(iris_ctx* c, int op, const float* x, float* out, int64_t rows, int width,
                      int param_i, float param_f, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || rows < 0 || width < 1 || op < 0 || op > 4)
        return fail(IRIS_ERR_INVALID, "iris_op_pointwise: bad argument");
    // complex_to_magphase of mono_chan's 3 columns: real [..., :1] broadcast against imag [..., 1:]
    // (transforms.py:111-123) -> rows of 4; every other odd width is an error, as in TF
    const bool bcast = op == IRIS_PW_COMPLEX_TO_MAGPHASE && width == 3;
    if (op <= IRIS_PW_MAGPHASE_TO_COMPLEX && (width & 1) && !bcast)
        return fail(IRIS_ERR_INVALID, "iris_op_pointwise: last axis must be 2 * n_chan");
    if (bcast && x == out) return fail(IRIS_ERR_INVALID, "iris_op_pointwise: rows of 3 -> 4 cannot be in place");
    CU(launch_pointwise(op, x, out, size_t(rows), bcast ? 2 : width / 2, width, param_i, param_f,
                        static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_normalize(iris_ctx* c, const float* x, float* out, int64_t n, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || n < 1) return fail(IRIS_ERR_INVALID, "iris_op_normalize: bad argument");
    CU(c->op_small.reserve(256));
    CU(launch_normalize(x, out, size_t(n), c->op_small.as<double>(), static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_chan_map(iris_ctx* c, int kind, const float* x, float* out, int64_t rows, int w_in,
                     int w_out, const float* factor, int64_t n_samples, int64_t rows_per_sample,
                     iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || x == out || rows < 0 || w_in < 2)
        return fail(IRIS_ERR_INVALID, "iris_op_chan_map: bad argument");
    std::vector<int32_t> idx;
    std::vector<float> coef;
    int64_t S = 1;
    size_t rps = size_t(rows > 0 ? rows : 1);
    auto put = [&](int i0, int i1) { idx.push_back(i0); idx.push_back(i1); };
    if (kind == IRIS_MAP_MONO_CHAN) {
        // x[..., :1] + x[..., 1:]  (broadcast: every other column gets column 0 added)
        if (w_out != w_in - 1) return fail(IRIS_ERR_INVALID, "mono_chan: w_out must be w_in - 1");
        for (int j = 0; j < w_out; ++j) { put(0, j + 1); coef.push_back(1.f); coef.push_back(1.f); }
    } else if (kind == IRIS_MAP_STEREO_MONO) {
        // concat(x[:2], x[0]+x[1], x[2:4], x[2]+x[3])   (data_utils.py:79-82)
        if (w_in < 4 || w_out != 6) return fail(IRIS_ERR_INVALID, "stereo_mono: needs [.., >=4] -> [.., 6]");
        const int a[6] = {0, 1, 0, 2, 3, 2}, b[6] = {-1, -1, 1, -1, -1, 3};
        for (int j = 0; j < 6; ++j) { put(a[j], b[j]); coef.push_back(1.f); coef.push_back(1.f); }
    } else if (kind == IRIS_MAP_MERGE_AUG) {
        // data_utils.py:104 -- ValueError('This augment can be used in 2 channel audio')
        if (w_in != 4) return fail(IRIS_ERR_INVALID, "This augment can be used in 2 channel audio");
        const int number = w_out / 2, extra = number - 2;
        if ((w_out & 1) || extra < 0 || (extra > 0 && !factor) || n_samples < 1 || rows_per_sample < 1 ||
            n_samples * rows_per_sample != rows)
            return fail(IRIS_ERR_INVALID, "random_merge_aug: bad shape");
        S = n_samples;
        rps = size_t(rows_per_sample);
        // real: [re0, re1, f*re0 + sqrt(1-f)*re1 ...]; imag: [im0, im1, im0 + im1 ...]
        for (int j = 0; j < number; ++j) put(j < 2 ? j : 0, j < 2 ? -1 : 1);
        for (int j = 0; j < number; ++j) put(j < 2 ? 2 + j : 2, j < 2 ? -1 : 3);
        coef.resize(size_t(S) * w_out * 2);
        for (int64_t s = 0; s < S; ++s)
            for (int j = 0; j < w_out; ++j) {
                float c0 = 1.f, c1 = 1.f;
                if (j >= 2 && j < number) {
                    const float f = factor[s * extra + (j - 2)];
                    c0 = f;
                    c1 = sqrtf(1.f - f);
                }
                coef[(size_t(s) * w_out + j) * 2] = c0;
                coef[(size_t(s) * w_out + j) * 2 + 1] = c1;
            }
    } else {
        return fail(IRIS_ERR_INVALID, "iris_op_chan_map: bad kind");
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    std::vector<char> blob(idx.size() * 4 + coef.size() * 4);
    memcpy(blob.data(), idx.data(), idx.size() * 4);
    memcpy(blob.data() + idx.size() * 4, coef.data(), coef.size() * 4);
    void* d;
    rc = upload_small(c, blob.data(), blob.size(), st, &d);
    if (rc) return rc;
    CU(launch_chan_map(x, out, size_t(rows), w_in, w_out, static_cast<int32_t*>(d),
                       reinterpret_cast<float*>(static_cast<char*>(d) + idx.size() * 4), rps, st));
    return IRIS_OK;
}

int iris_op_mel(iris_ctx* c, const float* x, float* out, int B, int T, int n_chan, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || x == out || B < 0 || T < 0 || n_chan < 1)
        return fail(IRIS_ERR_INVALID, "iris_op_mel: bad argument");
    if (c->n_mel == 0) return fail(IRIS_ERR_STATE, "iris_set_mel not called");
    CU(launch_mel_project(x, c->mel_dense.as<float>(), c->mel_lo.as<int32_t>(), c->mel_len.as<int32_t>(),
                          out, B, c->mel_bins, T, n_chan, c->n_mel, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_minmax(iris_ctx* c, int variant, const float* x, float* out, int64_t n_samples,
                   int64_t per_sample, int width, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || n_samples < 0 || per_sample < 1 || variant < 0 || variant > 1 || width < 1 ||
        per_sample % width)
        return fail(IRIS_ERR_INVALID, "iris_op_minmax: bad argument");
    if (variant == 1 && (width & 1)) return fail(IRIS_ERR_INVALID, "minmax_norm_magphase: odd last axis");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CU(c->minmax_ops.reserve(size_t(n_samples) * 16));
    // (min key, max key) per sample and group, identity = (0xffffffff, 0)
    std::vector<uint32_t> init(size_t(n_samples) * 4);
    for (size_t i = 0; i < init.size(); i += 2) { init[i] = 0xffffffffu; init[i + 1] = 0u; }
    CU(cudaMemcpyAsync(c->minmax_ops.p, init.data(), init.size() * 4, cudaMemcpyHostToDevice, st));
    CU(launch_minmax(x, out, c->minmax_ops.as<uint32_t>(), size_t(n_samples), size_t(per_sample), width,
                     variant == 1 ? width / 2 : width, variant, st));
    return IRIS_OK;
}

int iris_op_sum_voices(iris_ctx* c, const float* y, float* out, int64_t outer, int V, int64_t inner,
                       iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!y || !out || outer < 0 || V < 0 || inner < 1)
        return fail(IRIS_ERR_INVALID, "iris_op_sum_voices: bad argument");
    CU(launch_sum_axis(y, out, size_t(outer), V, size_t(inner), static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_avg_pool_time(iris_ctx* c, const float* y, float* out, int B, int T, int K, int r,
                          int binarize, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!y || !out || B < 0 || T < 1 || K < 1 || r < 1)
        return fail(IRIS_ERR_INVALID, "iris_op_avg_pool_time: bad argument");
    const int out_len = (T + r - 1) / r;
    int total_pad = (out_len - 1) * r + r - T;
    if (total_pad < 0) total_pad = 0;
    CU(launch_avg_pool_time(y, out, B, T, K, r, out_len, total_pad / 2, binarize,
                            static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_cos_sim(iris_ctx* c, const float* y_true, const float* y_pred, float* out, int B, int T,
                    int K, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!y_true || !y_pred || !out || B < 0 || T < 1 || K < 1)
        return fail(IRIS_ERR_INVALID, "iris_op_cos_sim: bad argument");
    if (K > 8) return fail(IRIS_ERR_UNSUPPORTED, "iris_op_cos_sim: more than 8 classes");
    CU(launch_cos_sim(y_true, y_pred, out, B, T, K, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}


// ---- evaluation-side chain (k_eval.cu) ----
int iris_op_eval_windows(iris_ctx* c, const float* x, float* out, int64_t outer, int64_t T, int64_t inner,
                         int frame_len, int step, int n_win, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || outer < 1 || T < 1 || inner < 1 || frame_len < 1 || step < 1)
        return fail(IRIS_ERR_INVALID, "iris_op_eval_windows: bad argument");
    if (int64_t(n_win) != (T + step - 1) / step)
        return fail(IRIS_ERR_INVALID, "iris_op_eval_windows: n_win must be ceil(T / step) (pad_end=True)");
    CU(launch_eval_windows(x, out, outer, T, inner, frame_len, step, n_win, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_eval_merge(iris_ctx* c, const float* preds, float* out, int n_win, int n_p, int K, int up,
                       int step, int L, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!preds || !out || n_win < 1 || n_p < 1 || K < 1 || up < 1 || step < 1 || L < 1)
        return fail(IRIS_ERR_INVALID, "iris_op_eval_merge: bad argument");
    if (int64_t(L) > int64_t(n_win - 1) * step + int64_t(n_p) * up)
        return fail(IRIS_ERR_INVALID, "iris_op_eval_merge: L exceeds the overlap-added length");
    CU(launch_eval_merge(preds, out, n_win, n_p, K, up, step, L, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_eval_smooth(iris_ctx* c, const float* x, float* tmp, float* out, int L, int K, int k_avg,
                        int k_max, float threshold, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !tmp || !out || L < 1 || K < 1 || k_avg < 1 || k_max < 1 || tmp == x || tmp == out)
        return fail(IRIS_ERR_INVALID, "iris_op_eval_smooth: bad argument");
    CU(launch_eval_smooth(x, tmp, out, L, K, k_avg, k_max, threshold, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_eval_events(iris_ctx* c, const float* y, int L, int K, int hop, int sr, int32_t* rows,
                        int max_rows, int32_t* n_rows, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!y || !rows || !n_rows || L < 1 || K < 1 || K > 8 || hop < 1 || sr < 1 || max_rows < 0)
        return fail(IRIS_ERR_INVALID, "iris_op_eval_events: bad argument");
    CU(launch_eval_events(y, L, K, hop, sr, rows, max_rows, n_rows, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_get_er(iris_ctx* c, const int32_t* gt, int m, const int32_t* pred, int pred_stride,
                   int pred_time_col, const int32_t* n_pred, int n_pred_max, int32_t* out,
                   iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!out || m < 0 || n_pred_max < 0 || (m && !gt) || (n_pred_max && !pred) || pred_stride < 2 ||
        pred_time_col < 1 || pred_time_col >= pred_stride)
        return fail(IRIS_ERR_INVALID, "iris_op_get_er: bad argument");
    if (m > (1 << 20) || n_pred_max > (1 << 20))
        return fail(IRIS_ERR_UNSUPPORTED, "iris_op_get_er: more than 2^20 events");
    // sort orders of the two lists
    CU(c->eval_scratch.reserve(size_t(m + n_pred_max + 2) * 4));
    int32_t* order_p = c->eval_scratch.as<int32_t>();
    int32_t* order_g = order_p + n_pred_max + 1;
    CU(launch_get_er(gt, m, pred, pred_stride, pred_time_col, n_pred, n_pred_max, order_p, order_g, out,
                     static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

// ---- trainer.py label variants (SURVEY.md 8f rank 4) ----
int iris_op_sum_pool2(iris_ctx* c, const float* y, float* out, int B, int T, int K, float scale,
                      iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!y || !out || y == out || B < 0 || T < 1 || K < 1)
        return fail(IRIS_ERR_INVALID, "iris_op_sum_pool2: bad argument");
    CU(launch_sum_pool2(y, out, B, T, K, scale, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

int iris_op_density_labels(iris_ctx* c, const float* y, float* out, int64_t outer, int V, int64_t inner,
                           iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!y || !out || y == out || outer < 0 || V < 1 || inner < 1 || inner > 0x7fffffff)
        return fail(IRIS_ERR_INVALID, "iris_op_density_labels: bad argument");
    if (V > 64) return fail(IRIS_ERR_UNSUPPORTED, "iris_op_density_labels: more than 64 voices");
    CU(launch_density_labels(y, out, size_t(outer), V, int(inner), static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

// transforms.phase_vocoder (transforms.py:137-195)
int iris_op_phase_vocoder(iris_ctx* c, const float* x, float* out, int n_freq, int T, int n_chan, int T_out,
                          const int32_t* idx0, const int32_t* idx1, const float* alpha, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!x || !out || x == out || n_freq < 2 || T < 1 || n_chan < 1 || T_out < 1 || !idx0 || !idx1 || !alpha)
        return fail(IRIS_ERR_INVALID, "iris_op_phase_vocoder: bad argument");
    if (size_t(T_out) * 12 > 64 * 1024) return fail(IRIS_ERR_UNSUPPORTED, "iris_op_phase_vocoder: more than 5461 output frames");
    for (int j = 0; j < T_out; ++j)
        if (idx0[j] < 0 || idx1[j] < 0 || idx0[j] > T + 1 || idx1[j] > T + 1)
            return fail(IRIS_ERR_INVALID, "iris_op_phase_vocoder: frame index outside the padded spectrogram");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    std::vector<int32_t> blob(size_t(T_out) * 3);
    memcpy(blob.data(), idx0, size_t(T_out) * 4);
    memcpy(blob.data() + T_out, idx1, size_t(T_out) * 4);
    memcpy(blob.data() + 2 * size_t(T_out), alpha, size_t(T_out) * 4);
    void* d;
    rc = upload_small(c, blob.data(), blob.size() * 4, st, &d);
    if (rc) return rc;
    const int32_t* di = static_cast<const int32_t*>(d);
    // phase_advance = tf.linspace(0, pi * hop, n_freq) with hop = n_freq - 1, in float32
    const float stop = float(M_PI) * float(n_freq - 1);
    const float step = stop / float(n_freq - 1);
    CU(launch_phase_vocoder(x, out, n_freq, T, n_chan, T_out, di, di + T_out,
                            reinterpret_cast<const float*>(di + 2 * size_t(T_out)), step, st));
    return IRIS_OK;
}

}  // extern "C"

// torchaudio.compliance.kaldi.resample_waveform (data_utils.py:20-21): Kaldi's LinearResample.
// The per-phase window starts and windowed-sinc weights are computed here in float32 in the
// port's op order (kaldi.py::_get_LR_indices_and_weights), the FIR runs in k_resample.cu.
namespace iris {
namespace {

// The filter bank of orig -> new_freq: first[u_out] window starts, then weights[u_out * W], appended to
// `blob`.  false: it would exceed 32 MB (nothing appended).
bool append_kaldi_table(int orig_freq, int new_freq, std::vector<char>& blob, int* u_in, int* u_out, int* W) {
    int g = orig_freq;
    for (int b = new_freq; b;) { const int t = g % b; g = b; b = t; }
    *u_in = orig_freq / g;
    *u_out = new_freq / g;
    const int uo = *u_out;
    const int min_freq = orig_freq < new_freq ? orig_freq : new_freq;
    const double cutoff = 0.99 * 0.5 * min_freq;              // lowpass_cutoff
    const double width = 6.0 / (2.0 * cutoff);                // window_width, lowpass_filter_width = 6
    const float ww = float(width), fo = float(orig_freq), fn = float(new_freq);
    std::vector<int32_t> first(uo);
    std::vector<float> mn(uo);
    int w_max = 0;
    for (int i = 0; i < uo; ++i) {
        const float t = float(i) / fn;
        mn[i] = ceilf((t - ww) * fo);
        const float mx = floorf((t + ww) * fo);
        first[i] = int32_t(mn[i]);
        w_max = std::max(w_max, int(mx - mn[i] + 1.f));
    }
    *W = w_max;
    if (size_t(uo) * w_max > (8u << 20)) return false;
    std::vector<float> wt(size_t(uo) * w_max);
    const float cw = float(2 * M_PI * cutoff / 6.0), cs = float(2 * M_PI * cutoff), pi = float(M_PI);
    for (int i = 0; i < uo; ++i) {
        const float t = float(i) / fn;
        for (int j = 0; j < w_max; ++j) {
            const float dt = (mn[i] + float(j)) / fo - t;
            float w = 0.f;
            if (fabsf(dt) < ww) w = 0.5f * (1.f + cosf(cw * dt));     // raised-cosine window
            if (dt != 0.f) w *= sinf(cs * dt) / (pi * dt);              // sinc
            else w *= float(2 * cutoff);
            wt[size_t(i) * w_max + j] = w / fo;
        }
    }
    const size_t at = align_up(blob.size(), 16);
    blob.resize(at + size_t(uo) * 4 + wt.size() * 4);
    memcpy(blob.data() + at, first.data(), size_t(uo) * 4);
    memcpy(blob.data() + at + size_t(uo) * 4, wt.data(), wt.size() * 4);
    return true;
}

}  // namespace

int resample_plan(const char* who, int n_items, int n_chan, const int64_t* n_in, const int32_t* orig,
                  int new_freq, ResamplePlan* plan) {
    std::vector<ResampleItem> items(n_items);
    std::vector<int32_t> rates;           // distinct rate pairs orig -> new_freq, in order of appearance
    std::vector<ResampleItem> tabs;       // their table, u_in, u_out, W
    std::vector<char>& blob = plan->blob;
    blob.assign(size_t(n_items) * sizeof(ResampleItem), 0);
    plan->n_out.assign(n_items, 0);
    plan->copy_only = true;
    plan->smem_floats = 0;
    long long in_off = 0, out_off = 0, total = 0;
    for (int i = 0; i < n_items; ++i) {
        ResampleItem& it = items[i];
        it.in_off = in_off;
        it.out_off = out_off;
        it.n_in = n_in[i];
        it.n_out = orig[i] == new_freq ? n_in[i] : iris_resample_len(n_in[i], orig[i], new_freq);
        it.table = -1;
        it.u_in = it.u_out = it.W = 1;
        if (orig[i] != new_freq) {
            plan->copy_only = false;
            size_t r = std::find(rates.begin(), rates.end(), orig[i]) - rates.begin();
            if (r == rates.size()) {
                ResampleItem t{};
                t.table = (long long)align_up(blob.size(), 16);
                if (!append_kaldi_table(orig[i], new_freq, blob, &t.u_in, &t.u_out, &t.W))
                    return fail(IRIS_ERR_UNSUPPORTED, std::string(who) + ": rate pair needs a filter bank above 32 MB");
                if (size_t(t.u_out) * t.W * 4 <= 96 * 1024)      // staged in shared memory
                    plan->smem_floats = std::max(plan->smem_floats, t.u_out * t.W);
                rates.push_back(orig[i]);
                tabs.push_back(t);
            }
            it.table = tabs[r].table;
            it.u_in = tabs[r].u_in;
            it.u_out = tabs[r].u_out;
            it.W = tabs[r].W;
        }
        plan->n_out[i] = it.n_out;
        in_off += it.n_in * n_chan;
        out_off += it.n_out * n_chan;
        total += it.n_out;
    }
    // outputs per CTA: 4096 amortise a table load over 4096 * n_chan outputs; smaller inputs get smaller
    // chunks so that the launch still spreads over the GPU (256: one output per thread)
    int chunk = 4096;
    while (chunk > 256 && total / chunk < 1024) chunk >>= 1;
    long long cta = 0;
    for (ResampleItem& it : items) {
        it.cta0 = cta;
        cta += (it.n_out + chunk - 1) / chunk;
    }
    if (cta >= (1ll << 31)) return fail(IRIS_ERR_UNSUPPORTED, std::string(who) + ": more than 2^31 CTAs of output");
    memcpy(blob.data(), items.data(), items.size() * sizeof(ResampleItem));
    plan->chunk = chunk;
    plan->n_ctas = cta;
    return IRIS_OK;
}

}  // namespace iris

extern "C" {
int64_t iris_resample_len(int64_t n_in, int orig_freq, int new_freq) {
    if (n_in <= 0 || orig_freq <= 0 || new_freq <= 0) return 0;
    // kaldi.py::_get_num_LR_output_samples: outputs whose time lies in [0, n_in / orig_freq)
    int64_t a = orig_freq, b = new_freq;
    while (b) { const int64_t t = a % b; a = b; b = t; }
    const int64_t tick = int64_t(orig_freq) / a * new_freq;
    const int64_t ticks_in = tick / orig_freq, ticks_out = tick / new_freq;
    const int64_t interval = n_in * ticks_in;
    int64_t last = interval / ticks_out;
    if (last * ticks_out == interval) --last;
    return last + 1;
}

int iris_resample(iris_ctx* c, const float* wav, int n_chan, int64_t n_in, int orig_freq, int new_freq,
                  float* d_out, iris_stream stream) {
    int rc = begin(c);
    if (rc) return rc;
    if (!wav || !d_out || n_chan < 1 || n_in < 1 || orig_freq < 1 || new_freq < 1)
        return fail(IRIS_ERR_INVALID, "iris_resample: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (orig_freq == new_freq) {
        CU(cudaMemcpyAsync(d_out, wav, size_t(n_in) * n_chan * 4, cudaMemcpyDefault, st));
        return IRIS_OK;
    }
    ResamplePlan plan;
    const int32_t rate = orig_freq;
    rc = resample_plan("iris_resample", 1, n_chan, &n_in, &rate, new_freq, &plan);
    if (rc) return rc;
    const size_t tab = plan.blob.size(), raw = size_t(n_in) * n_chan * 4;
    CU(c->spec_scratch.reserve(align_up(tab, 256) + raw));
    char* base = c->spec_scratch.as<char>();
    CU(cudaMemcpyAsync(base, plan.blob.data(), tab, cudaMemcpyHostToDevice, st));
    float* d_wav = reinterpret_cast<float*>(base + align_up(tab, 256));
    CU(cudaMemcpyAsync(d_wav, wav, raw, cudaMemcpyDefault, st));
    CU(cudaStreamSynchronize(st));   // the host blob is freed when this call returns
    CU(launch_resample(d_wav, d_out, n_chan, base, 1, plan.n_ctas, plan.chunk, plan.smem_floats, st));
    return IRIS_OK;
}
}  // extern "C"
