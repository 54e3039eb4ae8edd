// Internal state of libiris shared by the extern "C" translation units (not a public header).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <utility>
#include <vector>

#include "../../include/iris.h"
#include "iris_common.cuh"
#include "iris_launch.h"

namespace iris {

std::string& last_error();   // thread-local text behind iris_last_error()

inline int fail(int code, const std::string& msg) {
    last_error() = msg;
    return code;
}
inline int cuda_fail(cudaError_t e, const char* what) {
    last_error() = std::string(what) + ": " + cudaGetErrorString(e);
    return IRIS_ERR_CUDA;
}
#define CU(x)                                               \
    do {                                                    \
        cudaError_t e_ = (x);                               \
        if (e_ != cudaSuccess) return ::iris::cuda_fail(e_, #x); \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return static_cast<T*>(p); }
};

struct Bank {
    bool ready = false;
    bool spec = false;                 // items are pre-computed spectrograms [257, t, 2C] (k_spec.cu)
    int n_items = 0, n_chan = 0, n_classes = 0;
    std::vector<int64_t> offsets;      // samples per channel, cumulative
    std::vector<int64_t> pad_offsets;  // padded floats per channel, cumulative
    std::vector<int32_t> n_frames;
    int max_frames = 0;
    DevBuf padded, activity, labels, d_n_frames;
    // 2-channel waveform banks: the STFT bin plane, the geometry of `padded` (one 2 KB row per frame: bins
    // 0..127 of frame h as {re0, re1, im0, im1}; the item's last row is zero), read by the mel launches
    // (fused_reads_plane); `plane_floats` of it are in use
    DevBuf plane;
    size_t plane_floats = 0;
    std::vector<uint8_t> h_activity;   // host mirror (voice bank)
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// the IRIS_FEAT_* modes with a mel projection (IRIS_FEAT_SE, numbered after them, has none)
inline bool mel_mode(int mode) { return mode >= IRIS_FEAT_MEL && mode <= IRIS_FEAT_LOGMEL_MINMAX; }

// C' of include/iris.h: the channels after a plan's channel remap of n_chan bank channels
inline int remap_channels(int remap, int n_chan, int n_out_chan) {
    if (remap == IRIS_REMAP_NONE) return n_chan;
    if (remap == IRIS_REMAP_STEREO_MONO) return 3;
    if (remap == IRIS_REMAP_MONO_CHAN) return 2;
    return n_out_chan;
}
// last axis of the spectrogram modes (base mode < IRIS_FEAT_MEL): 2 C', except the 3 columns of mono_chan's
// complex spectrogram
inline int spec_width(int mode, int remap, int c_out) {
    return mode == IRIS_FEAT_COMPLEX && remap == IRIS_REMAP_MONO_CHAN ? 3 : 2 * c_out;
}

// One k_resample launch (iris_ops_abi.cu: resample_plan): item i is [n_chan, n_in[i]] at orig[i] Hz, packed
// back to back in the input, its [n_chan, n_out[i]] result back to back in the output.  `blob` is what goes
// to the device in one copy: the ResampleItem array, then the Kaldi filter table of every distinct rate pair
// (built once per pair).
struct ResamplePlan {
    std::vector<char> blob;
    std::vector<int64_t> n_out;
    long long n_ctas = 0;
    int chunk = 0, smem_floats = 0;
    bool copy_only = true;   // every item is at the target rate
};
// Rates must be >= 1.  A rate pair whose table exceeds 32 MB is IRIS_ERR_UNSUPPORTED ("<who>: ...").
int resample_plan(const char* who, int n_items, int n_chan, const int64_t* n_in, const int32_t* orig,
                  int new_freq, ResamplePlan* plan);

// mode argument of the feature entry points: IRIS_FEAT_* in the low 8 bits, at most one IRIS_OUT_*
// flag above them.  false: any other high bit (the base mode is range-checked by the caller).
inline bool split_feature_mode(int mode, int* base, int* out_type) {
    *base = mode & 0xff;
    switch (mode & ~0xff) {
        case 0: *out_type = OUT_F32; return true;
        case IRIS_OUT_BF16: *out_type = OUT_BF16; return true;
        case IRIS_OUT_F16: *out_type = OUT_F16; return true;
        default: return false;
    }
}

}  // namespace iris

struct iris_ctx {
    using DevBuf = iris::DevBuf;
    using Bank = iris::Bank;
    using Seg = iris::Seg;
    int device = 0;
    int num_sms = 148;
    Bank banks[3];
    DevBuf tw, ts, whalf;
    // mel (CSR by mel bin)
    int n_mel = 0, mel_f_lo = 0, mel_f_n = 0, mel_taps = 0;
    int mel_L[4] = {0, 0, 0, 0};
    DevBuf mel_info, mel_w;
    // plan
    bool has_plan = false, labels_done = false;
    int B = 0, T = 0, V = 0, M = 0, C = 0;
    int n_tmask = 0, n_fmask = 0, filter_k = 0, remap = 0, c_out = 0;
    std::vector<Seg> h_segs;
    std::vector<int64_t> h_seg_len;   // true samples per channel of each segment's source
    std::vector<int32_t> h_seg_ptr;
    DevBuf keep, minmax, scratch_labels, stft_pad, stft_small;   // minmax: [B,2] + done [B]
    DevBuf tiles, sched;
    int max_segs = 1;
    // tile blocks built by k_labels for the feature launch that follows (iris_abi.cu: run_labels):
    // the layout they were built for; a feature launch with another one runs k_tiles
    struct TileSig {
        bool valid = false;
        const void *segs = nullptr, *keep = nullptr;   // the plan (a plan upload invalidates as well)
        int B = 0, T = 0;
        int fm_bits = 0, seg_select = 0, fr = 0, n_pairs = 0, max_segs = 0, stride = 0, masks = 0, filter_k = 0;
        int plane = 0;   // the stages point into the bin planes (full gains) or into the waveforms (halved)
    } tile_sig;
    int feat_hint = -1;   // feature mode of the last feature launch: what k_labels builds tile blocks for
    cudaEvent_t ev_after_fused = nullptr;   // recorded (once) right behind the next k_fused launch (iris_step)
    // pinned staging for the plan blob: a ring, so that the host can run up to kStageRing batches
    // ahead of the device before it has to wait for an upload to drain
    static constexpr int kStageRing = 4;
    void* h_stage[kStageRing] = {nullptr, nullptr, nullptr, nullptr};
    size_t h_stage_cap[kStageRing] = {0, 0, 0, 0};
    cudaEvent_t stage_free[kStageRing] = {nullptr, nullptr, nullptr, nullptr};
    int stage_next = 0;
    size_t last_upload_bytes = 0;
    DevBuf plan_blobs[kStageRing];     // device side of the ring
    cudaStream_t copy = nullptr;       // plan uploads
    cudaEvent_t blob_ready[kStageRing] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t blob_used[kStageRing] = {nullptr, nullptr, nullptr, nullptr};
    bool blob_used_valid[kStageRing] = {false, false, false, false};
    // device views into plan_blob
    Seg* d_segs = nullptr;
    int32_t *d_seg_ptr = nullptr, *d_n_voices = nullptr, *d_voice_id = nullptr,
            *d_voice_shift = nullptr, *d_voice_kt = nullptr, *d_tmask = nullptr, *d_fmask = nullptr;
    float *d_merge_f = nullptr, *d_merge_sf = nullptr;
    // roofline measurement hook
    bool profile = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    size_t prof_used = 0;
    int prof_clips = 0;               // clips of the launch the hook timed last
    // stand-alone ops (iris_ops_abi.cu): dense mel matrix + column supports, small scratch
    DevBuf mel_dense, mel_lo, mel_len, op_small, minmax_ops, eval_scratch, spec_scratch;
    // fp32 mel features [B, n_mel, T, C] of a bfloat16 / float16 launch whose last pass (k_logmel_post)
    // converts: the min-max log-mel modes and the many-channel spectrogram-bank fallback
    DevBuf mel_scratch;
    bool spec_mode = false;            // the uploaded plan mixes spectrogram banks
    int mel_bins = 0;
    bool mel_fusable = false;
    // ---- one-call step (iris_step.cu) ----
    cudaStream_t side = nullptr;       // metric leg: counting + count all-reduce beside the feature kernel
    cudaEvent_t ev_labels = nullptr;   // labels of the current step are written
    static constexpr int kLegRing = 8;
    struct MetricLeg {
        cudaEvent_t done = nullptr;
        const void* labels = nullptr;  // frame-label buffer the leg reads
        uint64_t seq = 0;              // iris_step call that issued it (1-based); 0: never used
    } legs[kLegRing];
    uint64_t step_seq = 0;
    std::vector<int32_t> draw_i32;     // host draws of the last iris_step (views in `draws`)
    std::vector<float> draw_f32;
    iris_draws draws{};
    int mel_read_wavefronts = 0;       // modelled shared-memory wavefronts per frame of the mel tap reads
};

int iris_set_device(iris_ctx* c);
void iris_step_release(iris_ctx* c);   // iris_step.cu: side stream + events
