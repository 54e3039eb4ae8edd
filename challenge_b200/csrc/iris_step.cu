// One call per batch: host planner (uniforms -> draws with the reference's placement
// arithmetic), iris_step (draws -> plan upload -> labels -> features, metric leg on a side
// stream), the count all-reduce over NCCL, NUMA-local pinned host memory, DLPack entry points.
// Host-side logic only; the kernels live in k_*.cu.
#include <dlfcn.h>
#include <nccl.h>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/iris_dlpack.h"
#include "iris_ctx.h"

using namespace iris;

// ---------------------------------------------------------------------------------------
// shuffle stream (pipeline.py:143-147): buffer fed by the endlessly repeated 0..n-1
// ---------------------------------------------------------------------------------------
struct iris_shuffle {
    int n = 0;
    int next_up = 0;
    std::vector<int32_t> buf;
    int pull() {
        const int v = next_up;
        next_up = (next_up + 1) % n;
        return v;
    }
    int32_t take(double u) {
        size_t j = size_t(u * double(buf.size()));
        if (j >= buf.size()) j = buf.size() - 1;
        const int32_t v = buf[j];
        buf[j] = pull();
        return v;
    }
};

namespace {

inline int64_t rand_below(double u, int64_t range) {   // floor(u * range), u in [0, 1)
    if (range <= 1) return 0;
    int64_t v = int64_t(u * double(range));
    return v >= range ? range - 1 : v;
}
inline float unit_f32(double u) {                       // fp32 uniform in [0, 1)
    const float f = float(u);
    return f >= 1.f ? 0x1.fffffep-1f : f;
}

struct DrawLayout {
    int o_bg_id, o_bg_off, o_vid, o_nv, o_v, o_nid, o_nn, o_n, o_tm, o_fm, o_mf, n_u;
};
DrawLayout layout_of(const iris_draw_config& g) {
    DrawLayout L{};
    int o = 0;
    L.o_bg_id = o++;
    L.o_bg_off = o++;
    const int V = std::max(g.max_voices, 0), M = std::max(g.max_noises, 0);
    L.o_vid = o; o += V;
    L.o_nv = o; o += V > 0 ? 1 : 0;
    L.o_v = o; o += 2 * V;
    L.o_nid = o; o += M;
    L.o_nn = o; o += M > 0 ? 1 : 0;
    L.o_n = o; o += 2 * M;
    L.o_tm = o; o += 2 * std::max(g.n_time_masks, 0);
    L.o_fm = o; o += 2 * std::max(g.n_freq_masks, 0);
    L.o_mf = o; o += std::max(g.merge_extra, 0);
    L.n_u = o;
    return L;
}

// ---- NCCL, resolved at run time ----
struct NcclApi {
    bool tried = false, ok = false;
    std::string why;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi& nccl() {
    static NcclApi api;
    if (api.tried) return api;
    api.tried = true;
    // the copy the process already carries (torch bundles one) wins; else the system library
    void* h = nullptr;
    if (dlsym(RTLD_DEFAULT, "ncclAllReduce")) h = RTLD_DEFAULT;
    if (!h) {
        const char* names[] = {getenv("IRIS_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n || !*n) continue;
            h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
    }
    if (!h) {
        api.why = "NCCL not found (dlopen libnccl.so.2 failed; set IRIS_NCCL_LIB)";
        return api;
    }
    auto sym = [&](const char* n) { return dlsym(h, n); };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.GroupStart &&
             api.GroupEnd && api.GetErrorString;
    if (!api.ok) api.why = "NCCL library lacks a required symbol";
    return api;
}
#define NC(x)                                                                                  \
    do {                                                                                       \
        ncclResult_t r_ = (x);                                                                 \
        if (r_ != ncclSuccess)                                                                 \
            return fail(IRIS_ERR_CUDA, std::string(#x ": ") + nccl().GetErrorString(r_));       \
    } while (0)

int ensure_step_state(iris_ctx* c) {
    if (c->side) return IRIS_OK;
    CU(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&c->ev_labels, cudaEventDisableTiming));
    for (auto& l : c->legs) CU(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
    return IRIS_OK;
}

// DLManagedTensor -> device pointer after checking device / dtype / layout / shape; dtype: float32, or
// for features the OutType of the mode's IRIS_OUT_* flag
int dl_device_ptr(iris_ctx* c, void* managed, const int64_t* want_shape, int want_ndim, const char* what,
                  float** out, int out_type = OUT_F32) {
    if (!managed) return fail(IRIS_ERR_INVALID, std::string(what) + ": NULL DLManagedTensor");
    const DLTensor& t = static_cast<DLManagedTensor*>(managed)->dl_tensor;
    if (t.device.device_type != kDLCUDA)
        return fail(IRIS_ERR_INVALID, std::string(what) + ": DLPack tensor is not in CUDA device memory");
    if (t.device.device_id != c->device)
        return fail(IRIS_ERR_INVALID, std::string(what) + ": DLPack tensor lives on another device than the context");
    static const struct { int code, bits; const char* name; } kWant[3] = {
        {kDLFloat, 32, "float32"}, {kDLBfloat, 16, "bfloat16 (IRIS_OUT_BF16)"}, {kDLFloat, 16, "float16 (IRIS_OUT_F16)"}};
    if (t.dtype.code != kWant[out_type].code || t.dtype.bits != kWant[out_type].bits || t.dtype.lanes != 1)
        return fail(IRIS_ERR_INVALID, std::string(what) + ": DLPack tensor must be " + kWant[out_type].name);
    if (t.ndim != want_ndim) return fail(IRIS_ERR_INVALID, std::string(what) + ": wrong rank");
    int64_t stride = 1;
    for (int i = t.ndim - 1; i >= 0; --i) {
        if (t.shape[i] != want_shape[i]) {
            char msg[200];
            snprintf(msg, sizeof msg, "%s: axis %d has %lld elements, the plan needs %lld", what, i,
                     (long long)t.shape[i], (long long)want_shape[i]);
            return fail(IRIS_ERR_INVALID, msg);
        }
        if (t.strides && t.shape[i] > 1 && t.strides[i] != stride)
            return fail(IRIS_ERR_INVALID, std::string(what) + ": DLPack tensor must be C-contiguous");
        stride *= t.shape[i];
    }
    if (!t.data) return fail(IRIS_ERR_INVALID, std::string(what) + ": NULL data");
    *out = reinterpret_cast<float*>(static_cast<char*>(t.data) + t.byte_offset);
    return IRIS_OK;
}

// mode: the base mode (IRIS_FEAT_*)
void feature_shape(const iris_ctx* c, int mode, int64_t (&shape)[4]) {
    shape[0] = c->B;
    if (mode >= IRIS_FEAT_MEL) { shape[1] = c->n_mel; shape[2] = c->T; shape[3] = c->c_out; }   // after the remap
    else { shape[1] = kBins; shape[2] = c->T; shape[3] = spec_width(mode, c->remap, c->c_out); }
}

}  // namespace

void iris_step_release(iris_ctx* c) {
    if (c->side) cudaStreamDestroy(c->side);
    if (c->ev_labels) cudaEventDestroy(c->ev_labels);
    for (auto& l : c->legs)
        if (l.done) cudaEventDestroy(l.done);
    c->side = nullptr;
    c->ev_labels = nullptr;
}

extern "C" {

int iris_shuffle_create(int n_items, int buffer_size, iris_shuffle** out) {
    if (!out || n_items < 1) return fail(IRIS_ERR_INVALID, "iris_shuffle_create: need n_items >= 1");
    if (buffer_size <= 0) buffer_size = n_items;
    iris_shuffle* s = new iris_shuffle();
    s->n = n_items;
    s->buf.resize(size_t(buffer_size));
    for (auto& v : s->buf) v = s->pull();
    *out = s;
    return IRIS_OK;
}
int iris_shuffle_destroy(iris_shuffle* s) {
    delete s;
    return IRIS_OK;
}
int iris_shuffle_take(iris_shuffle* s, const double* u, int k, int32_t* out) {
    if (!s || !u || !out || k < 0) return fail(IRIS_ERR_INVALID, "iris_shuffle_take: bad argument");
    for (int i = 0; i < k; ++i) out[i] = s->take(u[i]);
    return IRIS_OK;
}

int iris_draw_uniforms_per_clip(const iris_draw_config* cfg) {
    if (!cfg) return fail(IRIS_ERR_INVALID, "NULL config");
    return layout_of(*cfg).n_u;
}

int iris_draw_batch(const iris_draw_config* cfg, const int32_t* bg_frames, int n_bg, const int32_t* voice_frames,
                    int n_voice, const int32_t* noise_frames, int n_noise, iris_shuffle* const* streams,
                    const double* uniforms, iris_draws* out) {
    if (!cfg || !uniforms || !out || !bg_frames) return fail(IRIS_ERR_INVALID, "iris_draw_batch: NULL argument");
    const iris_draw_config& g = *cfg;
    const int B = g.batch, T = g.n_frame, V = std::max(g.max_voices, 0), M = std::max(g.max_noises, 0);
    if (B < 1 || T < 1 || n_bg < 1) return fail(IRIS_ERR_INVALID, "iris_draw_batch: bad sizes");
    if (V > 0 && (!voice_frames || n_voice < 1)) return fail(IRIS_ERR_INVALID, "voice draws need the voice bank's frame counts");
    if (M > 0 && (!noise_frames || n_noise < 1)) return fail(IRIS_ERR_INVALID, "noise draws need the noise bank's frame counts");
    if (!out->bg_id || !out->bg_offset) return fail(IRIS_ERR_INVALID, "bg_id / bg_offset outputs NULL");
    if (V > 0 && (!out->n_voices || !out->voice_id || !out->voice_gain || !out->voice_offset))
        return fail(IRIS_ERR_INVALID, "voice outputs NULL");
    if (M > 0 && (!out->n_noises || !out->noise_id || !out->noise_gain || !out->noise_offset))
        return fail(IRIS_ERR_INVALID, "noise outputs NULL");
    const int n_tm = std::max(g.n_time_masks, 0), n_fm = std::max(g.n_freq_masks, 0), n_mf = std::max(g.merge_extra, 0);
    if ((n_tm && !out->time_masks) || (n_fm && !out->freq_masks) || (n_mf && !out->merge_factor))
        return fail(IRIS_ERR_INVALID, "mask / merge outputs NULL");
    const int n_bins = g.n_bins > 0 ? g.n_bins : kBins;
    iris_shuffle* s_bg = streams ? streams[0] : nullptr;
    iris_shuffle* s_v = streams ? streams[1] : nullptr;
    iris_shuffle* s_n = streams ? streams[2] : nullptr;
    const DrawLayout L = layout_of(g);
    const float snr_span = float(-double(g.snr) / 10.0);   // u ~ U[0, -snr/10)      (pipeline.py:50)
    char msg[200];
    for (int b = 0; b < B; ++b) {
        const double* u = uniforms + size_t(b) * L.n_u;
        // background: id, then the random_crop offset into the tiled background (pipeline.py:29-35)
        const int id = s_bg ? s_bg->take(u[L.o_bg_id]) : int(rand_below(u[L.o_bg_id], n_bg));
        out->bg_id[b] = id;
        const int64_t bgT = bg_frames[id];
        const int64_t tiled = bgT * ((T + bgT - 1) / bgT);
        out->bg_offset[b] = int32_t(rand_below(u[L.o_bg_off], tiled - T + 1));
        if (V > 0) {
            int vP = 0;   // padded_batch: the group's longest member (pipeline.py:155-156)
            for (int v = 0; v < V; ++v) {
                const int vid = s_v ? s_v->take(u[L.o_vid + v]) : int(rand_below(u[L.o_vid + v], n_voice));
                out->voice_id[size_t(b) * V + v] = vid;
                vP = std::max(vP, int(voice_frames[vid]));
            }
            const int nv = V > 1 ? 1 + int(rand_below(u[L.o_nv], V - 1)) : 1;              // (43)
            out->n_voices[b] = nv;
            const int pad = T - int(int32_t(float(g.min_ratio) * float(vP)));              // (58-59)
            const int len = pad > 0 ? vP + 2 * pad : vP;
            if (len - T <= 0) {
                snprintf(msg, sizeof msg,
                         "clip %d: voice group of padded length %d leaves an empty offset range for "
                         "n_frame=%d (pipeline.py:68-69)", b, vP, T);
                return fail(IRIS_ERR_EMPTY_RANGE, msg);
            }
            for (int v = 0; v < V; ++v) {
                const size_t k = size_t(b) * V + v;
                const bool live = v < nv;
                const float uu = live ? unit_f32(u[L.o_v + 2 * v]) * snr_span : 0.f;        // (50)
                if (out->voice_u) out->voice_u[k] = uu;
                out->voice_gain[k] = powf(10.f, -uu);
                out->voice_offset[k] = live ? int32_t(rand_below(u[L.o_v + 2 * v + 1], len - T)) : 0;   // (69)
            }
        }
        if (M > 0) {
            int nP = 0;
            for (int n = 0; n < M; ++n) {
                const int nid = s_n ? s_n->take(u[L.o_nid + n]) : int(rand_below(u[L.o_nid + n], n_noise));
                out->noise_id[size_t(b) * M + n] = nid;
                nP = std::max(nP, int(noise_frames[nid]));
            }
            const int nn = int(rand_below(u[L.o_nn], M));                                  // (87)
            out->n_noises[b] = nn;
            const int pad = T - int(int32_t(float(g.min_noise_ratio) * float(nP)));        // (95-96)
            const int len = pad > 0 ? nP + 2 * pad : nP;
            if (len < T) {
                snprintf(msg, sizeof msg, "clip %d: noise group shorter than n_frame after padding (pipeline.py:103)", b);
                return fail(IRIS_ERR_EMPTY_RANGE, msg);
            }
            for (int n = 0; n < M; ++n) {
                const size_t k = size_t(b) * M + n;
                const bool live = n < nn;
                const float uu = live ? unit_f32(u[L.o_n + 2 * n]) * 2.f : 0.f;             // (94)
                if (out->noise_u) out->noise_u[k] = uu;
                out->noise_gain[k] = powf(10.f, -uu);
                out->noise_offset[k] = live ? int32_t(rand_below(u[L.o_n + 2 * n + 1], len - T + 1)) : 0;   // (103)
            }
        }
        for (int i = 0; i < n_tm; ++i) {                                                   // transforms.py:25-26
            const int size = int(rand_below(u[L.o_tm + 2 * i], g.time_mask_max));
            int32_t* m = out->time_masks + (size_t(b) * n_tm + i) * 2;
            m[0] = size;
            m[1] = int32_t(rand_below(u[L.o_tm + 2 * i + 1], T - size));
        }
        for (int i = 0; i < n_fm; ++i) {
            const int size = int(rand_below(u[L.o_fm + 2 * i], g.freq_mask_max));
            int32_t* m = out->freq_masks + (size_t(b) * n_fm + i) * 2;
            m[0] = size;
            m[1] = int32_t(rand_below(u[L.o_fm + 2 * i + 1], n_bins - size));
        }
        for (int i = 0; i < n_mf; ++i)                                                     // data_utils.py:109
            out->merge_factor[size_t(b) * n_mf + i] = 0.1f + unit_f32(u[L.o_mf + i]) * 0.8f;
    }
    return IRIS_OK;
}

int iris_step(iris_ctx* c, const iris_step_config* cfg, const iris_step_io* io, iris_stream stream) {
    if (!c || !cfg || !io || !io->uniforms || !io->d_features) return fail(IRIS_ERR_INVALID, "iris_step: NULL argument");
    int base_mode = 0, out_type = OUT_F32;   // the output flag is iris_features' business; the rest needs the mode
    if (!split_feature_mode(cfg->feature_mode, &base_mode, &out_type))
        return fail(IRIS_ERR_INVALID, "iris_step: at most one of IRIS_OUT_BF16 / IRIS_OUT_F16 above the feature mode");
    int rc = iris_set_device(c);
    if (rc) return rc;
    rc = ensure_step_state(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const iris_draw_config& g = cfg->draw;
    const int B = g.batch, V = std::max(g.max_voices, 0), M = std::max(g.max_noises, 0);
    const int n_tm = std::max(g.n_time_masks, 0), n_fm = std::max(g.n_freq_masks, 0), n_mf = std::max(g.merge_extra, 0);
    if (B < 1) return fail(IRIS_ERR_INVALID, "iris_step: batch < 1");
    const Bank& bg = c->banks[IRIS_BANK_BG];
    const Bank& vb = c->banks[IRIS_BANK_VOICE];
    const Bank& nb = c->banks[IRIS_BANK_NOISE];
    if (!bg.ready) return fail(IRIS_ERR_STATE, "background bank not registered");
    if (V > 0 && !vb.ready) return fail(IRIS_ERR_STATE, "voice bank not registered");
    if (M > 0 && !nb.ready) return fail(IRIS_ERR_STATE, "noise bank not registered");

    // ---- draws (host) ----
    const size_t nB = size_t(B);
    c->draw_i32.resize(nB * (2 + 1 + V + V + 1 + M + M + 2 * n_tm + 2 * n_fm) + 16);
    c->draw_f32.resize(nB * (2 * V + 2 * M + n_mf) + 16);
    int32_t* pi = c->draw_i32.data();
    float* pf = c->draw_f32.data();
    iris_draws& d = c->draws;
    memset(&d, 0, sizeof d);
    d.bg_id = pi; pi += nB;
    d.bg_offset = pi; pi += nB;
    if (V > 0) {
        d.n_voices = pi; pi += nB;
        d.voice_id = pi; pi += nB * V;
        d.voice_offset = pi; pi += nB * V;
        d.voice_u = pf; pf += nB * V;
        d.voice_gain = pf; pf += nB * V;
    }
    if (M > 0) {
        d.n_noises = pi; pi += nB;
        d.noise_id = pi; pi += nB * M;
        d.noise_offset = pi; pi += nB * M;
        d.noise_u = pf; pf += nB * M;
        d.noise_gain = pf; pf += nB * M;
    }
    if (n_tm) { d.time_masks = pi; pi += nB * n_tm * 2; }
    if (n_fm) { d.freq_masks = pi; pi += nB * n_fm * 2; }
    if (n_mf) { d.merge_factor = pf; pf += nB * n_mf; }
    rc = iris_draw_batch(&g, bg.n_frames.data(), bg.n_items, V > 0 ? vb.n_frames.data() : nullptr, vb.n_items,
                         M > 0 ? nb.n_frames.data() : nullptr, nb.n_items, io->streams, io->uniforms, &d);
    if (rc) return rc;

    // ---- plan: validation + segment lists + one H2D copy (iris_plan_upload) ----
    iris_plan pl;
    memset(&pl, 0, sizeof pl);
    pl.batch = B; pl.n_frame = g.n_frame; pl.max_voices = V; pl.max_noises = M;
    pl.min_ratio = g.min_ratio; pl.min_noise_ratio = g.min_noise_ratio;
    pl.bg_id = d.bg_id; pl.bg_offset = d.bg_offset;
    pl.n_voices = d.n_voices; pl.voice_id = d.voice_id; pl.voice_gain = d.voice_gain; pl.voice_offset = d.voice_offset;
    pl.n_noises = d.n_noises; pl.noise_id = d.noise_id; pl.noise_gain = d.noise_gain; pl.noise_offset = d.noise_offset;
    pl.n_time_masks = n_tm; pl.n_freq_masks = n_fm;
    pl.time_masks = d.time_masks; pl.freq_masks = d.freq_masks;
    pl.stft_filter = cfg->stft_filter; pl.chan_remap = cfg->chan_remap; pl.n_out_chan = cfg->n_out_chan;
    pl.merge_factor = d.merge_factor;
    rc = iris_plan_upload(c, &pl, stream);
    if (rc) return rc;

    // ---- labels, then the metric leg beside the feature kernel ----
    const bool metric = io->d_y_pred != nullptr;
    if (metric && (!io->d_frame_labels || !io->d_triples || V == 0))
        return fail(IRIS_ERR_INVALID, "the metric leg needs voices, d_frame_labels and d_triples");
    ++c->step_seq;
    if (io->d_frame_labels)   // a leg of an earlier step may still read this buffer on the side stream
        for (auto& l : c->legs)
            if (l.seq && l.labels == io->d_frame_labels) CU(cudaStreamWaitEvent(st, l.done, 0));
    if (V > 0) {
        c->feat_hint = base_mode;   // k_labels also builds the tile blocks of the feature launch
        rc = iris_labels(c, io->d_labels_vtk, io->d_frame_labels, io->d_keep, stream);
        if (rc) return rc;
    }
    // The metric leg needs the labels only.  For the min-max log-mel features it is forked BEHIND
    // k_fused and runs beside k_logmel_post (31 us, the leg takes ~10): k_labels -> k_fused stay
    // adjacent in the stream, so k_fused's programmatic launch overlaps its prologue with k_labels.
    // Other modes have no second pass to hide the leg behind: it forks right behind k_labels.
    const bool late = metric && base_mode == IRIS_FEAT_LOGMEL_MINMAX && !c->spec_mode;
    if (late) {
        c->ev_after_fused = c->ev_labels;
        rc = iris_features(c, cfg->feature_mode, io->d_features, stream);
        if (rc) return rc;
        if (c->ev_after_fused) {   // the feature path did not go through run_fused
            c->ev_after_fused = nullptr;
            CU(cudaEventRecord(c->ev_labels, st));
        }
    }
    if (metric) {
        if (!late) CU(cudaEventRecord(c->ev_labels, st));
        CU(cudaStreamWaitEvent(c->side, c->ev_labels, 0));
        const int K = vb.n_classes;
        CU(launch_metric_counts(io->d_frame_labels, io->d_y_pred, B, c->T, c->T, K,
                                io->threshold > 0.f ? io->threshold : 0.5f, io->d_triples,
                                reinterpret_cast<unsigned long long*>(io->d_counts),
                                io->d_counts ? reinterpret_cast<unsigned long long*>(io->d_counts) + 3 : nullptr,
                                c->side));
        if (io->comm) {
            if (!io->d_counts || !io->d_counts_reduced)
                return fail(IRIS_ERR_INVALID, "the count all-reduce needs d_counts and d_counts_reduced");
            rc = iris_allreduce_counts(c, io->comm, reinterpret_cast<const int64_t*>(io->d_counts),
                                       io->d_counts_reduced, io->d_triples_send, io->d_triples_global,
                                       io->global_batch, c->side);
            if (rc) return rc;
        }
        iris_ctx::MetricLeg& leg = c->legs[c->step_seq % iris_ctx::kLegRing];
        CU(cudaEventRecord(leg.done, c->side));
        leg.labels = io->d_frame_labels;
        leg.seq = c->step_seq;
    }
    if (late) return IRIS_OK;
    return iris_features(c, cfg->feature_mode, io->d_features, stream);
}

int iris_counts_wait(iris_ctx* c, int lag, iris_stream stream) {
    if (!c || lag < 0) return fail(IRIS_ERR_INVALID, "iris_counts_wait: bad argument");
    if (uint64_t(lag) >= c->step_seq || lag >= iris_ctx::kLegRing) return IRIS_OK;   // nothing that old
    const uint64_t want = c->step_seq - uint64_t(lag);
    const iris_ctx::MetricLeg& leg = c->legs[want % iris_ctx::kLegRing];
    if (leg.seq == want) CU(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), leg.done, 0));
    return IRIS_OK;
}

int iris_step_draws(iris_ctx* c, iris_draws* out) {
    if (!c || !out) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (c->step_seq == 0) return fail(IRIS_ERR_STATE, "iris_step has not run");
    *out = c->draws;
    return IRIS_OK;
}

int iris_allreduce_counts(iris_ctx* c, iris_nccl_comm comm, const int64_t* d_send, int64_t* d_recv,
                          const int32_t* d_tr_send, int32_t* d_tr_recv, int global_batch, iris_stream stream) {
    if (!c || !comm || !d_send || !d_recv) return fail(IRIS_ERR_INVALID, "iris_allreduce_counts: NULL argument");
    if ((d_tr_send == nullptr) != (d_tr_recv == nullptr) || (d_tr_send && global_batch < 1))
        return fail(IRIS_ERR_INVALID, "iris_allreduce_counts: triples need send, recv and global_batch");
    NcclApi& n = nccl();
    if (!n.ok) return fail(IRIS_ERR_STATE, n.why);
    int rc = iris_set_device(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ncclComm_t cm = static_cast<ncclComm_t>(comm);
    NC(n.GroupStart());
    ncclResult_t r1 = n.AllReduce(d_send, d_recv, 6, ncclInt64, ncclSum, cm, st);
    ncclResult_t r2 = ncclSuccess;
    if (d_tr_send) r2 = n.AllReduce(d_tr_send, d_tr_recv, size_t(global_batch) * 3, ncclInt32, ncclSum, cm, st);
    ncclResult_t r3 = n.GroupEnd();
    NC(r1);
    NC(r2);
    NC(r3);
    return IRIS_OK;
}

int iris_nccl_unique_id(void* out) {
    if (!out) return fail(IRIS_ERR_INVALID, "NULL argument");
    NcclApi& n = nccl();
    if (!n.ok) return fail(IRIS_ERR_STATE, n.why);
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NC(n.GetUniqueId(&id));
    memcpy(out, &id, sizeof id);
    return IRIS_OK;
}

int iris_nccl_comm_create(iris_ctx* c, const void* id128, int rank, int world, iris_nccl_comm* out) {
    if (!c || !id128 || !out || world < 1 || rank < 0 || rank >= world)
        return fail(IRIS_ERR_INVALID, "iris_nccl_comm_create: bad argument");
    NcclApi& n = nccl();
    if (!n.ok) return fail(IRIS_ERR_STATE, n.why);
    int rc = iris_set_device(c);
    if (rc) return rc;
    ncclUniqueId id;
    memcpy(&id, id128, sizeof id);
    ncclComm_t cm = nullptr;
    NC(n.CommInitRank(&cm, world, id, rank));
    *out = cm;
    return IRIS_OK;
}

int iris_nccl_comm_destroy(iris_nccl_comm comm) {
    if (!comm) return IRIS_OK;
    NcclApi& n = nccl();
    if (!n.ok) return fail(IRIS_ERR_STATE, n.why);
    NC(n.CommDestroy(static_cast<ncclComm_t>(comm)));
    return IRIS_OK;
}

int iris_er_from_triples(iris_ctx* c, const int32_t* d_triples, int n, float* d_er, iris_stream stream) {
    if (!c || !d_triples || !d_er || n < 1) return fail(IRIS_ERR_INVALID, "iris_er_from_triples: bad argument");
    int rc = iris_set_device(c);
    if (rc) return rc;
    CU(launch_er_finalize(d_triples, n, d_er, static_cast<cudaStream_t>(stream)));
    return IRIS_OK;
}

// ---- NUMA-local pinned host memory ----
int iris_host_alloc(iris_ctx* c, size_t bytes, void** out, int* numa_node) {
    if (!c || !out || bytes == 0) return fail(IRIS_ERR_INVALID, "iris_host_alloc: bad argument");
    int rc = iris_set_device(c);
    if (rc) return rc;
    int node = -1;
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, c->device) == cudaSuccess) {
        for (char* p = bus; *p; ++p) *p = char(tolower(*p));
        std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
        if (FILE* f = fopen(path.c_str(), "r")) {
            if (fscanf(f, "%d", &node) != 1) node = -1;
            fclose(f);
        }
    }
    const size_t page = size_t(sysconf(_SC_PAGESIZE));
    const size_t len = (bytes + page - 1) / page * page;
    void* p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) return fail(IRIS_ERR_CUDA, "iris_host_alloc: mmap failed");
    if (node >= 0 && node < 1024) {
        unsigned long mask[16] = {0};
        mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
#ifdef SYS_mbind
        if (syscall(SYS_mbind, p, len, 2 /* MPOL_BIND */, mask, sizeof(mask) * 8, 0) != 0) node = -1;
#else
        node = -1;
#endif
    }
    memset(p, 0, len);   // fault the pages in on the chosen node before they are pinned
    cudaError_t e = cudaHostRegister(p, len, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        munmap(p, len);
        return cuda_fail(e, "cudaHostRegister");
    }
    *out = p;
    if (numa_node) *numa_node = node;
    return IRIS_OK;
}

int iris_host_free(iris_ctx* c, void* p, size_t bytes) {
    if (!p) return IRIS_OK;
    if (c) iris_set_device(c);
    cudaHostUnregister(p);
    const size_t page = size_t(sysconf(_SC_PAGESIZE));
    munmap(p, (bytes + page - 1) / page * page);
    return IRIS_OK;
}

// ---- DLPack entry points ----
int iris_features_dlpack(iris_ctx* c, int mode, void* managed, iris_stream stream) {
    if (!c) return fail(IRIS_ERR_INVALID, "NULL ctx");
    if (!c->has_plan) return fail(IRIS_ERR_STATE, "no plan uploaded");
    int base = 0, out_type = OUT_F32;
    if (!split_feature_mode(mode, &base, &out_type) || base < IRIS_FEAT_COMPLEX || base > IRIS_FEAT_LOGMEL_MINMAX)
        return fail(IRIS_ERR_INVALID, base == IRIS_FEAT_SE ? "IRIS_FEAT_SE has three output blocks: one DLPack tensor cannot "
                                                             "describe them (use iris_features)" : "bad feature mode");
    int64_t shape[4];
    feature_shape(c, base, shape);
    float* out = nullptr;
    int rc = dl_device_ptr(c, managed, shape, 4, "features", &out, out_type);
    if (rc) return rc;
    return iris_features(c, mode, out, stream);
}

int iris_labels_dlpack(iris_ctx* c, void* managed_vtk, void* managed_frame, iris_stream stream) {
    if (!c) return fail(IRIS_ERR_INVALID, "NULL ctx");
    if (!c->has_plan) return fail(IRIS_ERR_STATE, "no plan uploaded");
    const int K = c->banks[IRIS_BANK_VOICE].n_classes;
    float *vtk = nullptr, *frame = nullptr;
    int rc;
    if (managed_vtk) {
        const int64_t s4[4] = {c->B, c->V, c->T, K};
        if ((rc = dl_device_ptr(c, managed_vtk, s4, 4, "labels [B,V,T,K]", &vtk))) return rc;
    }
    if (managed_frame) {
        const int64_t s3[3] = {c->B, c->T, K};
        if ((rc = dl_device_ptr(c, managed_frame, s3, 3, "frame labels [B,T,K]", &frame))) return rc;
    }
    return iris_labels(c, vtk, frame, nullptr, stream);
}

int iris_step_dlpack(iris_ctx* c, const iris_step_config* cfg, const double* uniforms, iris_shuffle* const* streams,
                     void* managed_features, void* managed_frame_labels, iris_stream stream) {
    if (!c || !cfg) return fail(IRIS_ERR_INVALID, "NULL argument");
    const iris_draw_config& g = cfg->draw;
    const Bank& bg = c->banks[IRIS_BANK_BG];
    if (!bg.ready) return fail(IRIS_ERR_STATE, "background bank not registered");
    int base_mode = 0, out_type = OUT_F32;
    if (!split_feature_mode(cfg->feature_mode, &base_mode, &out_type))
        return fail(IRIS_ERR_INVALID, "iris_step_dlpack: at most one of IRIS_OUT_BF16 / IRIS_OUT_F16 above the feature mode");
    if (base_mode == IRIS_FEAT_SE)
        return fail(IRIS_ERR_INVALID, "IRIS_FEAT_SE has three output blocks: one DLPack tensor cannot describe them (use iris_step)");
    const int c_out = remap_channels(cfg->chan_remap, bg.n_chan, cfg->n_out_chan);
    int64_t fs[4] = {g.batch, kBins, g.n_frame, spec_width(base_mode, cfg->chan_remap, c_out)};
    if (base_mode >= IRIS_FEAT_MEL) { fs[1] = c->n_mel; fs[3] = c_out; }
    iris_step_io io;
    memset(&io, 0, sizeof io);
    io.uniforms = uniforms;
    io.streams = streams;
    int rc = dl_device_ptr(c, managed_features, fs, 4, "features", &io.d_features, out_type);
    if (rc) return rc;
    if (managed_frame_labels) {
        const int64_t s3[3] = {g.batch, g.n_frame, c->banks[IRIS_BANK_VOICE].n_classes};
        if ((rc = dl_device_ptr(c, managed_frame_labels, s3, 3, "frame labels [B,T,K]", &io.d_frame_labels))) return rc;
    }
    return iris_step(c, cfg, &io, stream);
}

int64_t iris_plan_upload_bytes(iris_ctx* c) { return c ? int64_t(c->last_upload_bytes) : 0; }
int iris_mel_fusable(iris_ctx* c) { return c && c->mel_fusable ? 1 : 0; }
int iris_max_segments(void) { return fused_max_segments(); }

}  // extern "C"
