// extern "C" surface of libiris (include/iris.h): context, bank registration, batch plan,
// and the launches of the hot-path kernels.  Host-side logic only; kernels live in k_*.cu.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "iris_ctx.h"
#include "iris_tiles.cuh"

using namespace iris;

thread_local std::string g_err;
namespace iris {
std::string& last_error() { return g_err; }
}

namespace {

int set_device(iris_ctx* c) { return iris_set_device(c); }

int build_tables(iris_ctx* c) {
    // fftwarp.cuh tables.  tw1[q][n2] = {W512^(n2*2q), W512^(n2*(2q+1))} (inter-pass twiddles);
    // ts[m][par] = {t(2m), t(2m+1)} with t(i) = par ? W32^i : 1 (radix-2 DIF of pass 2)
    std::vector<float> tw(8 * 32 * 4), ts(8 * 2 * 4), hann(512);
    for (int q = 0; q < 8; ++q)
        for (int n2 = 0; n2 < 32; ++n2)
            for (int h = 0; h < 2; ++h) {
                const double a = -2.0 * M_PI * double((2 * q + h) * n2) / 512.0;
                tw[4 * (q * 32 + n2) + 2 * h] = float(cos(a));
                tw[4 * (q * 32 + n2) + 2 * h + 1] = float(sin(a));
            }
    for (int m = 0; m < 8; ++m)
        for (int par = 0; par < 2; ++par)
            for (int h = 0; h < 2; ++h) {
                const double a = -2.0 * M_PI * double(2 * m + h) / 32.0;
                ts[4 * (m * 2 + par) + 2 * h] = par ? float(cos(a)) : 1.f;
                ts[4 * (m * 2 + par) + 2 * h + 1] = par ? float(sin(a)) : 0.f;
            }
    // periodic Hann (torch.hann_window(512)); the 1/2 of the two-channel split rides on the gains
    for (int n = 0; n < 512; ++n) hann[n] = float(0.5 - 0.5 * cos(2.0 * M_PI * n / 512.0));
    CU(c->tw.reserve(tw.size() * 4));
    CU(c->ts.reserve(ts.size() * 4));
    CU(c->whalf.reserve(hann.size() * 4));
    CU(cudaMemcpy(c->tw.p, tw.data(), tw.size() * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->ts.p, ts.data(), ts.size() * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->whalf.p, hann.data(), hann.size() * 4, cudaMemcpyHostToDevice));
    CU(c->sched.reserve(8));   // k_fused work counters: next chunk, CTAs finished
    CU(cudaMemset(c->sched.p, 0, 8));
    return IRIS_OK;
}

void fill_common(iris_ctx* c, FusedParams& p) {
    memset(&p, 0, sizeof(p));
    p.tw1 = c->tw.as<float4>();
    p.ts = c->ts.as<float4>();
    p.hann = c->whalf.as<float>();
    p.n_mel = c->n_mel;
    p.mel_f_lo = c->mel_f_lo;
    p.mel_f_n = c->mel_f_n;
    p.mel_taps = c->mel_taps;
    for (int r = 0; r < 4; ++r) p.mel_L[r] = c->mel_L[r];
    p.mel_info = c->mel_info.as<uint32_t>();
    p.mel_w = c->mel_w.as<float>();
}

// a tile of the fused kernel is `fr` frames of one (clip, channel pair)
void set_geometry(iris_ctx* c, FusedParams& p, int n_chan, bool mel) {
    p.C = n_chan;
    p.n_pairs = (n_chan + 1) / 2;
    p.c_out = n_chan;
    if (!mel) p.mel_taps = 0;   // no mel tables in shared memory
    p.fr = fused_pick_fr(p.mel_taps);
    (void)c;
}

int ensure_stage(iris_ctx* c, int slot, size_t bytes) {
    if (bytes <= c->h_stage_cap[slot]) return IRIS_OK;
    if (c->h_stage[slot]) cudaFreeHost(c->h_stage[slot]);
    c->h_stage[slot] = nullptr;
    c->h_stage_cap[slot] = 0;
    const size_t want = bytes + bytes / 4 + 4096;
    CU(cudaMallocHost(&c->h_stage[slot], want));
    c->h_stage_cap[slot] = want;
    return IRIS_OK;
}

int feature_params(iris_ctx* c, int mode, int select, FusedParams& p);
bool tile_sig_matches(const iris_ctx* c, const FusedParams& p);
void tile_sig_set(iris_ctx* c, const FusedParams& p);

// feat_hint: feature mode of the launch that will follow (-1: unknown).  With a hint the label
// kernel also builds the tile blocks of that launch (k_labels.cu), which then skips k_tiles.
int run_labels(iris_ctx* c, float* d_vtk, float* d_frame, uint8_t* d_keep_out, cudaStream_t st, int feat_hint = -1) {
    const Bank& vb = c->banks[IRIS_BANK_VOICE];
    c->tile_sig.valid = false;
    const int K = vb.ready ? vb.n_classes : 0;
    if (c->V > 0 && !vb.ready) return fail(IRIS_ERR_STATE, "voice bank not registered");
    CU(c->keep.reserve(size_t(c->B) * (c->V > 0 ? c->V : 1)));
    if (c->V == 0 || K == 0) {
        c->labels_done = true;
        return IRIS_OK;
    }
    float* frame = d_frame;
    if (!frame) {
        CU(c->scratch_labels.reserve(size_t(c->B) * c->T * K * 4));
        frame = c->scratch_labels.as<float>();
    }
    LabelParams lp;
    lp.B = c->B; lp.T = c->T; lp.V = c->V; lp.K = K;
    lp.n_voices = c->d_n_voices;
    lp.voice_id = c->d_voice_id;
    lp.voice_shift = c->d_voice_shift;
    lp.voice_kt = c->d_voice_kt;
    lp.n_frames = vb.d_n_frames.as<int32_t>();
    lp.activity = vb.activity.as<uint8_t>();
    lp.act_stride = vb.max_frames;
    lp.bank_labels = vb.labels.as<float>();
    lp.labels_vtk = d_vtk;
    lp.frame_labels = frame;
    lp.keep = c->keep.as<uint8_t>();
    FusedParams fp;
    bool tiles = false;
    if (((feat_hint >= IRIS_FEAT_COMPLEX && feat_hint <= IRIS_FEAT_LOGMEL_MINMAX) || feat_hint == IRIS_FEAT_SE) &&
        !c->spec_mode && !getenv("IRIS_NO_LABEL_TILES")) {
        const bool mel = mel_mode(feat_hint);
        if (!(mel && (c->n_mel == 0 || !c->mel_fusable)))
            tiles = feature_params(c, feat_hint, IRIS_SELECT_ALL, fp) == IRIS_OK;
    }
    CU(launch_labels(lp, st, tiles ? &fp : nullptr));
    if (tiles) tile_sig_set(c, fp);
    if (d_keep_out)
        CU(cudaMemcpyAsync(d_keep_out, c->keep.p, size_t(c->B) * c->V, cudaMemcpyDeviceToDevice, st));
    c->labels_done = true;
    return IRIS_OK;
}

// tile-block scratch + launch parameters of a launch
int prepare_fused(iris_ctx* c, FusedParams& p, int mode, int max_segs) {
    p.max_segs = max_segs < 1 ? 1 : max_segs;
    p.stage_out = fused_stages_output(mode, p.remap, p.fr) ? 1 : 0;
    p.fm_bits = (mode == FM_MEL && p.mel_f_lo + p.mel_f_n <= 128) ? 1 : 0;   // = the NJ == 4 kernels
    p.plane = fused_reads_plane(p, mode) ? 1 : 0;
    p.pair_merge = p.stage_out && p.C == 4 ? 1 : 0;
    int stride = 0;
    const size_t bytes = fused_tile_bytes(p, &stride);
    const void* before = c->tiles.p;
    CU(c->tiles.reserve(bytes));
    if (c->tiles.p != before) c->tile_sig.valid = false;
    p.tile_blocks = c->tiles.as<unsigned char>();
    p.tile_stride = stride;
    p.sched = c->sched.as<uint32_t>();
    // tiles per work claim.  With the claims shrinking towards the end of a launch (fused_schedule) larger
    // chunks no longer cost a longer tail: 4 / 6 / 8 / 16 tiles -> k_fused 173.6 / 172.4 / 172.6 / 177.6 us
    p.chunk = 6;
    if (p.pair_merge && (p.chunk & 1)) ++p.chunk;   // both pairs of a (clip, time) range in one work claim
    return IRIS_OK;
}

// k_tiles + k_fused over the whole batch
bool tile_sig_matches(const iris_ctx* c, const FusedParams& p) {
    const iris_ctx::TileSig& g = c->tile_sig;
    return g.valid && g.segs == p.segs && g.keep == p.keep && g.B == p.B && g.T == p.T && g.fm_bits == p.fm_bits && g.seg_select == p.seg_select && g.fr == p.fr &&
           g.n_pairs == p.n_pairs && g.max_segs == p.max_segs && g.stride == p.tile_stride &&
           g.masks == ((p.tmask ? 1 : 0) | (p.fmask ? 2 : 0)) && g.filter_k == p.filter_k && g.plane == p.plane;
}
void tile_sig_set(iris_ctx* c, const FusedParams& p) {
    iris_ctx::TileSig& g = c->tile_sig;
    g.valid = true;
    g.segs = p.segs; g.keep = p.keep; g.B = p.B; g.T = p.T;
    g.fm_bits = p.fm_bits; g.seg_select = p.seg_select; g.fr = p.fr; g.n_pairs = p.n_pairs;
    g.max_segs = p.max_segs; g.stride = p.tile_stride;
    g.masks = (p.tmask ? 1 : 0) | (p.fmask ? 2 : 0);
    g.filter_k = p.filter_k;
    g.plane = p.plane;
}

// k_tiles + k_fused over the whole batch; k_tiles is skipped when the tile blocks of this plan
// already exist in this layout (built by k_labels or by an earlier feature launch)
int run_fused(iris_ctx* c, FusedParams& p, int mode, int max_segs, cudaStream_t st, int out_type = OUT_F32) {
    int rc = prepare_fused(c, p, mode, max_segs);
    if (rc) return rc;
    CU(launch_fused(p, mode, c->num_sms, st, !tile_sig_matches(c, p), out_type));
    tile_sig_set(c, p);
    if (c->ev_after_fused) {   // iris_step: the metric leg starts behind the feature kernel
        CU(cudaEventRecord(c->ev_after_fused, st));
        c->ev_after_fused = nullptr;
    }
    return IRIS_OK;
}

int prof_events(iris_ctx* c, std::pair<cudaEvent_t, cudaEvent_t>** out) {
    if (c->prof_used == c->prof_events.size()) {
        cudaEvent_t a, b;
        CU(cudaEventCreate(&a));
        CU(cudaEventCreate(&b));
        c->prof_events.emplace_back(a, b);
    }
    *out = &c->prof_events[c->prof_used++];
    return IRIS_OK;
}

int timed_fused(iris_ctx* c, FusedParams& p, int mode, cudaStream_t st, int out_type) {
    if (!c->profile) return run_fused(c, p, mode, c->max_segs, st, out_type);
    std::pair<cudaEvent_t, cudaEvent_t>* ev = nullptr;
    int rc = prof_events(c, &ev);
    if (rc) return rc;
    CU(cudaEventRecord(ev->first, st));
    rc = run_fused(c, p, mode, c->max_segs, st, out_type);
    if (rc) return rc;
    CU(cudaEventRecord(ev->second, st));
    c->prof_clips = c->B;
    return IRIS_OK;
}

// min-max log-mel: k_fused (fp32 features + per-clip extrema at p.out) -> k_logmel_post (normalise + log
// in place at d_out == p.out, or for bfloat16 / float16 features from the fp32 scratch at p.out into d_out)
int run_logmel_minmax(iris_ctx* c, FusedParams& p, void* d_out, cudaStream_t st, int out_type) {
    const size_t per_clip = size_t(c->n_mel) * c->T * p.c_out;
    uint32_t* mm = c->minmax.as<uint32_t>();
    unsigned* done = reinterpret_cast<unsigned*>(mm + 2 * size_t(c->B));
    int rc = timed_fused(c, p, FM_MEL, st, OUT_F32);
    if (rc) return rc;
    CU(launch_logmel_post(p.out, d_out, out_type, mm, done, c->B, per_clip, 1, 1, st));
    return IRIS_OK;
}

// fp32 mel scratch [B, n_mel, T, c_out] of a half-width launch whose last pass converts
int mel_scratch(iris_ctx* c, float** out) {
    CU(c->mel_scratch.reserve(size_t(c->B) * c->n_mel * c->T * c->c_out * 4));
    *out = c->mel_scratch.as<float>();
    return IRIS_OK;
}

// FusedParams of a feature launch from waveform banks: everything but the output pointer and the
// min-max scratch, including the tile-block scratch and its layout (prepare_fused)
int feature_params(iris_ctx* c, int mode, int select, FusedParams& p) {
    const bool mel = mel_mode(mode);
    fill_common(c, p);
    p.segs = c->d_segs;
    p.seg_ptr = c->d_seg_ptr;
    p.keep = c->V > 0 ? c->keep.as<uint8_t>() : nullptr;
    p.B = c->B; p.T = c->T;
    set_geometry(c, p, c->C, mel);
    p.c_out = c->c_out;
    p.tmask = c->d_tmask; p.n_tmask = c->n_tmask;
    p.fmask = c->d_fmask; p.n_fmask = c->n_fmask;
    p.filter_k = c->filter_k;
    p.remap = c->remap;
    p.merge_f = c->d_merge_f; p.merge_sf = c->d_merge_sf;
    if (select) {   // only_voice / only_noise: the plain mix of a subset, no masks / remap / filter
        p.seg_select = select;
        p.tmask = nullptr; p.fmask = nullptr; p.n_tmask = 0; p.n_fmask = 0;
        p.filter_k = 0; p.remap = IRIS_REMAP_NONE; p.c_out = c->C;
        set_geometry(c, p, c->C, false);
    }
    if (mode == IRIS_FEAT_SE) {   // two virtual channel pairs over bank pair 0: voices | background + noises
        if (c->C != 2 || c->remap != IRIS_REMAP_NONE)
            return fail(IRIS_ERR_UNSUPPORTED, "IRIS_FEAT_SE takes 2-channel plans without a channel remap");
        p.seg_select = 3;
        set_geometry(c, p, 4, false);
    }
    if (mel) {
        p.do_log = mode != IRIS_FEAT_MEL;
        p.do_minmax = mode == IRIS_FEAT_LOGMEL_MINMAX;
        // the bin planes of the plan's banks, for the launches that read them (fused_reads_plane)
        bool planes = c->C == 2;
        int k = 0;
        for (int kind : {IRIS_BANK_BG, IRIS_BANK_VOICE, IRIS_BANK_NOISE}) {
            const Bank& bk = c->banks[kind];
            const bool used = kind == IRIS_BANK_BG || (kind == IRIS_BANK_VOICE ? c->V > 0 : c->M > 0);
            if (!used) continue;
            if (!bk.ready || bk.spec || bk.n_chan != 2 || !bk.plane.p) { planes = false; break; }
            p.pl_wave[k] = bk.padded.as<float>();
            p.pl_floats[k] = int64_t(bk.plane_floats);
            p.pl_delta[k] = (int64_t(uintptr_t(bk.plane.p)) - int64_t(uintptr_t(bk.padded.p))) / 4;
            ++k;
        }
        if (!planes)
            for (int i = 0; i < 3; ++i) { p.pl_wave[i] = nullptr; p.pl_floats[i] = 0; p.pl_delta[i] = 0; }
    }
    return prepare_fused(c, p, mel ? FM_MEL : mode == IRIS_FEAT_SE ? FM_SE : mode, c->max_segs);
}

// Features from spectrogram banks: the mix + per-cell epilogue is one streaming kernel
// (k_spec.cu), for the mel modes with the projection and the per-clip extrema fused in.
int spec_features(iris_ctx* c, int mode, int select, float* d_out, cudaStream_t st, int out_type) {
    const bool mel = mel_mode(mode);
    if (mel && c->mel_bins != kBins) return fail(IRIS_ERR_INVALID, "the mel matrix must have 257 rows");
    FusedParams p;
    fill_common(c, p);
    p.segs = c->d_segs;
    p.seg_ptr = c->d_seg_ptr;
    p.keep = c->V > 0 ? c->keep.as<uint8_t>() : nullptr;
    p.B = c->B; p.T = c->T; p.C = c->C;
    p.n_pairs = (c->C + 1) / 2;
    p.c_out = c->c_out;
    p.tmask = c->d_tmask; p.n_tmask = c->n_tmask;
    p.fmask = c->d_fmask; p.n_fmask = c->n_fmask;
    p.filter_k = c->filter_k;
    p.remap = c->remap;
    p.merge_f = c->d_merge_f; p.merge_sf = c->d_merge_sf;
    if (select) {   // only_voice / only_noise: the plain mix of a subset, no masks / remap / filter
        p.seg_select = select;
        p.tmask = nullptr; p.fmask = nullptr; p.n_tmask = 0; p.n_fmask = 0;
        p.filter_k = 0; p.remap = IRIS_REMAP_NONE; p.c_out = c->C;
    }
    if (!mel) {
        p.out = d_out;
        CU(launch_specmix(p, mode == IRIS_FEAT_SE ? FM_SE : mode, nullptr, nullptr, nullptr, st, out_type));
        return IRIS_OK;
    }
    const size_t per_clip = size_t(c->n_mel) * c->T * c->c_out;   // mel channels: after the remap
    if (specmix_mel_smem(c->c_out, c->mel_f_n) <= 200 * 1024) {
        // fused: mix -> |.| -> mel -> per-clip extrema in one pass; k_logmel_post normalises in L2
        p.out = d_out;
        p.do_log = mode != IRIS_FEAT_MEL;
        p.do_minmax = mode == IRIS_FEAT_LOGMEL_MINMAX;
        const bool convert = p.do_minmax && out_type != OUT_F32;   // fp32 mel in scratch, k_logmel_post converts
        if (p.do_minmax) {
            CU(c->minmax.reserve(size_t(c->B) * 12));
            CU(cudaMemsetAsync(c->minmax.p, 0, size_t(c->B) * 12, st));
            p.minmax = c->minmax.as<uint32_t>();
            if (convert) {
                int rc = mel_scratch(c, &p.out);
                if (rc) return rc;
            }
        }
        CU(launch_specmix(p, FM_MEL, c->mel_dense.as<float>(), c->mel_lo.as<int32_t>(),
                          c->mel_len.as<int32_t>(), st, convert ? OUT_F32 : out_type));
        uint32_t* mm = c->minmax.as<uint32_t>();
        unsigned* done = c->minmax.as<unsigned>() + 2 * size_t(c->B);
        if (p.do_minmax) CU(launch_logmel_post(p.out, d_out, out_type, mm, done, c->B, per_clip, 1, 1, st));
        return IRIS_OK;
    }
    // many channels: magnitudes through a scratch spectrogram (remapped by store_bin), then the stand-alone
    // kernels (fp32; for bfloat16 / float16 features the mel goes to a scratch and the last pass converts)
    CU(c->spec_scratch.reserve(size_t(c->B) * kBins * c->T * 2 * c->c_out * 4));
    p.out = c->spec_scratch.as<float>();
    CU(launch_specmix(p, FM_MAGPHASE, nullptr, nullptr, nullptr, st, OUT_F32));
    float* mel_out = d_out;
    if (out_type != OUT_F32) {
        int rc = mel_scratch(c, &mel_out);
        if (rc) return rc;
    }
    CU(launch_mel_project(p.out, c->mel_dense.as<float>(), c->mel_lo.as<int32_t>(), c->mel_len.as<int32_t>(),
                          mel_out, c->B, kBins, c->T, c->c_out, c->n_mel, st));
    if (mode == IRIS_FEAT_LOGMEL_MINMAX) {
        int rc = iris_op_minmax(c, 0, mel_out, mel_out, c->B, int64_t(per_clip), 1, st);
        if (rc) return rc;
    }
    CU(launch_logmel_post(mel_out, d_out, out_type, nullptr, nullptr, c->B, per_clip, 0, mode != IRIS_FEAT_MEL, st));
    return IRIS_OK;
}

}  // namespace

int iris_set_device(iris_ctx* c) {
    CU(cudaSetDevice(c->device));
    return IRIS_OK;
}

extern "C" {

int iris_abi_version(void) { return IRIS_ABI_VERSION; }
const char* iris_last_error(void) { return g_err.c_str(); }

int iris_ctx_create(int device, iris_ctx** out) {
    if (!out) return fail(IRIS_ERR_INVALID, "out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(IRIS_ERR_CUDA, std::string("no CUDA device (libiris has no CPU fallback): ") +
                                       cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(IRIS_ERR_INVALID, "device index out of range");
    iris_ctx* c = new iris_ctx();
    c->device = device;
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess ||
        (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        delete c;
        return cuda_fail(e, "cudaSetDevice");
    }
    if (prop.major != 10) {
        delete c;
        return fail(IRIS_ERR_UNSUPPORTED, "libiris is built for sm_100a (Blackwell B200) only");
    }
    c->num_sms = prop.multiProcessorCount;
    for (int i = 0; i < iris_ctx::kStageRing; ++i)
        if ((e = cudaEventCreateWithFlags(&c->stage_free[i], cudaEventDisableTiming)) != cudaSuccess) {
            delete c;
            return cuda_fail(e, "cudaEventCreate");
        }
    int rc = build_tables(c);
    if (rc != IRIS_OK) {
        delete c;
        return rc;
    }
    *out = c;
    return IRIS_OK;
}

int iris_ctx_destroy(iris_ctx* c) {
    if (!c) return IRIS_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto& b : c->banks) {
        b.padded.release(); b.activity.release(); b.labels.release(); b.d_n_frames.release(); b.plane.release();
    }
    for (auto& pb : c->plan_blobs) pb.release();
    if (c->copy) {
        cudaStreamDestroy(c->copy);
        for (int i = 0; i < iris_ctx::kStageRing; ++i) {
            if (c->blob_ready[i]) cudaEventDestroy(c->blob_ready[i]);
            if (c->blob_used[i]) cudaEventDestroy(c->blob_used[i]);
        }
    }
    for (DevBuf* d : {&c->tw, &c->whalf, &c->mel_info, &c->mel_w, &c->keep,
                      &c->minmax, &c->scratch_labels, &c->stft_pad, &c->stft_small, &c->tiles, &c->ts, &c->sched,
                      &c->mel_dense, &c->mel_lo, &c->mel_len, &c->op_small, &c->minmax_ops, &c->eval_scratch, &c->spec_scratch,
                      &c->mel_scratch})
        d->release();
    for (int i = 0; i < iris_ctx::kStageRing; ++i) {
        if (c->h_stage[i]) cudaFreeHost(c->h_stage[i]);
        if (c->stage_free[i]) cudaEventDestroy(c->stage_free[i]);
    }
    iris_step_release(c);
    for (auto& ev : c->prof_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    delete c;
    return IRIS_OK;
}

int iris_set_mel(iris_ctx* c, int n_mel, int n_bins, const float* w) {
    if (!c || !w) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (n_bins != kBins) return fail(IRIS_ERR_INVALID, "n_bins must be 257 (n_fft 512)");
    if (n_mel < 1 || n_mel > 128) return fail(IRIS_ERR_INVALID, "n_mel must be in [1, 128]");
    int rc = set_device(c);
    if (rc) return rc;
    // every mel filter is the contiguous bin range [lo, hi] that holds its non-zero weights
    // (the triangles of linear_to_mel_weight_matrix are contiguous)
    std::vector<int> lo_of(n_mel, -1), len_of(n_mel, 0);
    int f_lo = kBins, f_hi = -1;
    for (int m = 0; m < n_mel; ++m) {
        int lo = -1, hi = -1;
        for (int f = 0; f < n_bins; ++f)
            if (w[size_t(f) * n_mel + m] != 0.f) {
                if (lo < 0) lo = f;
                hi = f;
            }
        if (lo < 0) continue;   // empty filter
        lo_of[m] = lo;
        len_of[m] = hi - lo + 1;
        f_lo = std::min(f_lo, lo);
        f_hi = std::max(f_hi, hi);
    }
    if (f_hi < 0) { f_lo = 0; f_hi = 0; }
    const int f_n = f_hi - f_lo + 1;
    // rounds of 32 filters (filter m = lane + 32 r) share a trip count (the longest filter of
    // the round); shorter filters are zero-padded and shifted so that every tap stays inside
    // [f_lo, f_hi]
    int L[4] = {0, 0, 0, 0}, taps = 0;
    for (int m = 0; m < n_mel; ++m) L[m >> 5] = std::max(L[m >> 5], len_of[m]);
    for (int r = 0; r < 4; ++r) {
        if ((L[r] & 1) && L[r] < f_n) ++L[r];   // even trip counts: the kernel takes two taps per step
        taps += L[r];
    }
    // the stand-alone projection (iris_op_mel) takes any matrix: dense weights + column supports
    {
        std::vector<int32_t> lo32(n_mel), len32(n_mel);
        for (int m = 0; m < n_mel; ++m) { lo32[m] = lo_of[m] < 0 ? 0 : lo_of[m]; len32[m] = len_of[m]; }
        CU(c->mel_dense.reserve(size_t(n_bins) * n_mel * 4));
        CU(c->mel_lo.reserve(size_t(n_mel) * 4));
        CU(c->mel_len.reserve(size_t(n_mel) * 4));
        CU(cudaMemcpy(c->mel_dense.p, w, size_t(n_bins) * n_mel * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->mel_lo.p, lo32.data(), size_t(n_mel) * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->mel_len.p, len32.data(), size_t(n_mel) * 4, cudaMemcpyHostToDevice));
        c->mel_bins = n_bins;
        c->n_mel = n_mel;
    }
    bool odd = false;
    for (int r = 0; r < 4; ++r) odd = odd || (L[r] & 1);
    bool wide = false;
    for (int r = 0; r < 4; ++r) wide = wide || L[r] > fused_max_mel_filter();
    c->mel_fusable = taps <= fused_max_mel_taps() && !odd && !wide;
    if (!c->mel_fusable) return IRIS_OK;   // iris_features(mel modes) then reports UNSUPPORTED
    // ---- filter -> (round, lane) assignment ----
    // Lane l of round r projects filter slot[r][l] (or nothing).  Any assignment gives the same
    // numbers (every lane stores its own mel row); what it changes is the bank-conflict count of
    // the magnitude reads: the 16 lanes of a half-warp read (|ch0|, |ch1|) pairs (8 bytes) at
    // bins start + q, which is conflict-free iff their starts are distinct modulo 16 (or equal).
    // In natural order (filter m = lane + 32 r) the TF matrix costs 44 shared-memory wavefronts
    // per frame for its 12 taps; the search below brings it to ~30 (24 = no conflict at all).
    // Cost of a round = trip count x (wavefronts of half-warp 0 + half-warp 1); the sum of the
    // trip counts may not grow.  Deterministic annealing over slot swaps (LCG, fixed seed).
    const int n_slots = 128;
    std::vector<int> slot(n_slots, -1);
    for (int m = 0; m < n_mel; ++m) slot[m] = lo_of[m] < 0 ? -1 : m;
    auto round_len = [&](const std::vector<int>& s, int r) {
        int l = 0;
        for (int i = 0; i < 32; ++i)
            if (s[32 * r + i] >= 0) l = std::max(l, len_of[s[32 * r + i]]);
        if ((l & 1) && l < f_n) ++l;
        return l;
    };
    auto read_start = [&](int m, int Lr) { return std::min(lo_of[m] - f_lo, f_n - Lr); };
    auto cost = [&](const std::vector<int>& s, int* taps_out) {
        int total = 0, tp = 0;
        for (int r = 0; r < 4; ++r) {
            const int Lr = round_len(s, r);
            tp += Lr;
            if (Lr == 0) continue;
            int wf = 0;
            for (int h = 0; h < 2; ++h) {
                int seen[16][8], cnt[16] = {0};
                int worst = 1;
                for (int i = 0; i < 16; ++i) {
                    const int m = s[32 * r + 16 * h + i];
                    if (m < 0) continue;   // an idle lane copies a neighbour's address (broadcast)
                    const int st = f_lo + read_start(m, Lr), k = st & 15;
                    bool dup = false;
                    for (int j = 0; j < cnt[k]; ++j) dup = dup || seen[k][j] == st;
                    if (!dup && cnt[k] < 8) seen[k][cnt[k]++] = st;
                    worst = std::max(worst, cnt[k]);
                }
                wf += worst;
            }
            total += Lr * wf;
        }
        if (taps_out) *taps_out = tp;
        return total;
    };
    {
        int tp = 0;
        int cur = cost(slot, &tp);
        std::vector<int> best = slot;
        int best_cost = cur;
        uint32_t rng = 0x9e3779b9u;
        auto next = [&]() { rng = rng * 1664525u + 1013904223u; return rng >> 8; };
        double temp = 2.0;
        const int used_rounds = (n_mel + 31) / 32;
        for (int it = 0; it < 60000 && best_cost > 2 * taps; ++it) {
            const int a = int(next() % uint32_t(32 * used_rounds)), b = int(next() % uint32_t(32 * used_rounds));
            if (a == b || slot[a] == slot[b]) continue;
            std::swap(slot[a], slot[b]);
            int tp2 = 0;
            const int cst = cost(slot, &tp2);
            const bool ok = tp2 <= taps;
            const double u = double(next() & 0xffff) / 65536.0;
            if (ok && (cst <= cur || u < exp(double(cur - cst) / temp))) {
                cur = cst;
                if (cst < best_cost) { best_cost = cst; best = slot; }
            } else {
                std::swap(slot[a], slot[b]);
            }
            temp = std::max(0.05, temp * 0.9999);
        }
        slot = best;
        for (int r = 0; r < 4; ++r) L[r] = round_len(slot, r);
        taps = L[0] + L[1] + L[2] + L[3];
        c->mel_read_wavefronts = best_cost;
    }
    // info word of a slot: first tap (relative to f_lo) | mel row << 16; row 0xffff = idle lane
    std::vector<uint32_t> info(n_slots, 0xffff0000u);
    std::vector<float> fw(size_t(std::max(taps, 1)) * 32, 0.f);
    int row0 = 0;
    for (int r = 0; r < 4; ++r) {
        for (int h = 0; h < 2; ++h) {
            int fill = 0;   // idle lanes read where the first busy lane of their half-warp reads
            for (int i = 0; i < 16; ++i) {
                const int m = slot[32 * r + 16 * h + i];
                if (m >= 0) { fill = read_start(m, L[r]); break; }
            }
            for (int i = 0; i < 16; ++i) {
                const int l = 16 * h + i, m = slot[32 * r + l];
                if (m < 0) {
                    info[32 * r + l] = 0xffff0000u | uint32_t(L[r] ? fill : 0);
                    continue;
                }
                const int start = read_start(m, L[r]);
                info[32 * r + l] = uint32_t(start) | (uint32_t(m) << 16);
                for (int t = 0; t < len_of[m]; ++t)
                    fw[size_t(row0 + (lo_of[m] - f_lo - start) + t) * 32 + l] =
                        w[size_t(lo_of[m] + t) * n_mel + m];
            }
        }
        row0 += L[r];
    }
    CU(c->mel_info.reserve(info.size() * 4));
    CU(c->mel_w.reserve(fw.size() * 4));
    CU(cudaMemcpy(c->mel_info.p, info.data(), info.size() * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->mel_w.p, fw.data(), fw.size() * 4, cudaMemcpyHostToDevice));
    c->mel_taps = taps;
    for (int r = 0; r < 4; ++r) c->mel_L[r] = L[r];
    c->n_mel = n_mel;
    c->mel_f_lo = f_lo;
    c->mel_f_n = f_n;
    return IRIS_OK;
}

}  // extern "C"

namespace {

// Registration of a waveform bank from 16 kHz audio, shared by iris_bank_register and
// iris_bank_register_audio.  bank_layout: checks the items of `offsets` (host, cumulative per-channel
// 16 kHz samples) and lays out their frames; bank_fill: from the packed items in `wav16` (device, item i
// at n_chan * (offsets[i] - offsets[0])), normalize + reflect-padded pair layout (k_bank_prepare) and,
// for the voice bank, the activity pass.  Synchronises the stream and releases wav16.
int bank_layout(iris_ctx* c, int kind, int n_items, int n_chan, const int64_t* offsets, int n_classes) {
    Bank& b = c->banks[kind];
    b.ready = false;
    b.spec = false;
    b.n_items = n_items;
    b.n_chan = n_chan;
    b.n_classes = n_classes;
    b.offsets.assign(offsets, offsets + n_items + 1);
    b.pad_offsets.assign(n_items + 1, 0);
    b.n_frames.assign(n_items, 0);
    b.max_frames = 0;
    for (int i = 0; i < n_items; ++i) {
        const int64_t n = offsets[i + 1] - offsets[i];
        if (n <= kNFft / 2)
            return fail(IRIS_ERR_INVALID,
                        "source shorter than 257 samples (reflect padding needs pad < length)");
        const int64_t kT = 1 + n / kHop;
        if (n_chan > 2 && 2 * 256 * (kT + 1) > INT32_MAX)
            return fail(IRIS_ERR_UNSUPPORTED,
                        "a source of 3 or more channels longer than 1073741311 samples (pair stride above 2^31 - 1)");
        b.n_frames[i] = int32_t(kT);
        if (kT > b.max_frames) b.max_frames = int(kT);
        b.pad_offsets[i + 1] = b.pad_offsets[i] + 256 * (kT + 1);
    }
    if (n_chan > 32) return fail(IRIS_ERR_UNSUPPORTED, "more than 32 channels");
    return IRIS_OK;
}

int bank_fill(iris_ctx* c, int kind, DevBuf& wav16, const float* labels, int normalize, cudaStream_t st) {
    Bank& b = c->banks[kind];
    const int n_items = b.n_items, n_chan = b.n_chan, n_classes = b.n_classes;
    const int n_pairs = (n_chan + 1) / 2;
    const size_t pad_floats = size_t(b.pad_offsets[n_items]) * n_pairs * 2;
    DevBuf d_off;
    CU(d_off.reserve(size_t(n_items + 1) * 16));
    CU(b.padded.reserve(pad_floats * 4));
    CU(b.d_n_frames.reserve(size_t(n_items) * 4));
    std::vector<int64_t> rel(n_items + 1);
    for (int i = 0; i <= n_items; ++i) rel[i] = b.offsets[i] - b.offsets[0];
    int64_t* d_o = d_off.as<int64_t>();
    CU(cudaMemcpyAsync(d_o, rel.data(), size_t(n_items + 1) * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_o + n_items + 1, b.pad_offsets.data(), size_t(n_items + 1) * 8,
                       cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(b.d_n_frames.p, b.n_frames.data(), size_t(n_items) * 4,
                       cudaMemcpyHostToDevice, st));
    CU(launch_bank_prepare(wav16.as<float>(), d_o, d_o + n_items + 1, n_items, n_chan, normalize,
                           b.padded.as<float>(), st));
    b.plane_floats = 0;
    if (n_chan != 2) b.plane.release();
    if (kind == IRIS_BANK_VOICE || n_chan == 2) {
        // the STFT passes over the bank: one segment per item, gain 1 (the split of the packed two-channel
        // FFT then gives X itself)
        std::vector<Seg> segs(n_items);
        std::vector<int32_t> ptr(n_items + 1);
        for (int i = 0; i < n_items; ++i) {
            Seg& s = segs[i];
            const int64_t plen = 256 * (int64_t(b.n_frames[i]) + 1);
            s.base = b.padded.as<float>() + size_t(b.pad_offsets[i]) * n_pairs * 2;
            s.pair_stride = int32_t(2 * plen);
            s.shift = 0;
            s.t_lo = 0;
            s.t_hi = b.n_frames[i];
            s.gain = 1.f;
            s.keep_idx = -1;
            ptr[i] = i;
        }
        ptr[n_items] = n_items;
        DevBuf d_segs;
        CU(d_segs.reserve(segs.size() * sizeof(Seg) + ptr.size() * 4));
        Seg* ds = d_segs.as<Seg>();
        int32_t* dp = reinterpret_cast<int32_t*>(ds + n_items);
        CU(cudaMemcpyAsync(ds, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(dp, ptr.data(), ptr.size() * 4, cudaMemcpyHostToDevice, st));
        FusedParams p;
        fill_common(c, p);
        p.segs = ds;
        p.seg_ptr = dp;
        p.B = n_items;
        p.T = b.max_frames;
        set_geometry(c, p, n_chan, false);
        if (n_chan == 2) {
            // the bin plane: bins 0..127 of every frame, the rows behind an item's last frame zero
            CU(b.plane.reserve(pad_floats * 4));
            CU(cudaMemsetAsync(b.plane.p, 0, pad_floats * 4, st));
            p.pl_delta[0] = (int64_t(uintptr_t(b.plane.p)) - int64_t(uintptr_t(b.padded.p))) / 4;
            const int rc = run_fused(c, p, FM_PLANE, 1, st);
            c->tile_sig.valid = false;   // the segment list of this pass is freed below
            if (rc) return rc;
            b.plane_floats = pad_floats;
        }
        if (kind == IRIS_BANK_VOICE) {
            CU(b.labels.reserve(size_t(n_items) * n_classes * 4));
            CU(cudaMemcpyAsync(b.labels.p, labels, size_t(n_items) * n_classes * 4,
                               cudaMemcpyHostToDevice, st));
            // activity: frame active iff any coefficient > 0
            const size_t act_bytes = size_t(n_items) * b.max_frames;
            CU(b.activity.reserve(act_bytes));
            CU(cudaMemsetAsync(b.activity.p, 0, act_bytes, st));
            p.activity = b.activity.as<uint8_t>();
            const int rc = run_fused(c, p, FM_ACTIVITY, 1, st);
            c->tile_sig.valid = false;
            if (rc) return rc;
            b.h_activity.resize(act_bytes);
            CU(cudaMemcpyAsync(b.h_activity.data(), b.activity.p, act_bytes, cudaMemcpyDeviceToHost, st));
        }
        CU(cudaStreamSynchronize(st));
        d_segs.release();
    }
    CU(cudaStreamSynchronize(st));
    wav16.release();
    d_off.release();
    b.ready = true;
    c->has_plan = false;
    return IRIS_OK;
}

}  // namespace

extern "C" {

int iris_bank_register(iris_ctx* c, int kind, int n_items, int n_chan, const float* wav,
                       const int64_t* offsets, const float* labels, int n_classes, int normalize,
                       iris_stream stream) {
    if (!c || !wav || !offsets) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (kind < 0 || kind > 2) return fail(IRIS_ERR_INVALID, "bad bank kind");
    if (n_items < 1 || n_chan < 1) return fail(IRIS_ERR_INVALID, "empty bank");
    if (kind == IRIS_BANK_VOICE && (!labels || n_classes < 1))
        return fail(IRIS_ERR_INVALID, "voice bank needs labels [n_items, n_classes]");
    int rc = set_device(c);
    if (rc) return rc;
    rc = bank_layout(c, kind, n_items, n_chan, offsets, n_classes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t wav_floats = size_t(offsets[n_items] - offsets[0]) * n_chan;
    DevBuf raw;
    CU(raw.reserve(wav_floats * 4));
    CU(cudaMemcpyAsync(raw.p, wav + size_t(offsets[0]) * n_chan, wav_floats * 4, cudaMemcpyDefault, st));
    return bank_fill(c, kind, raw, labels, normalize, st);
}

int iris_bank_register_audio(iris_ctx* c, int kind, int n_items, int n_chan, const float* wav,
                             const int64_t* offsets, const int32_t* sample_rates, const float* labels,
                             int n_classes, int normalize, iris_stream stream) {
    if (!c || !wav || !offsets || !sample_rates) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (kind < 0 || kind > 2) return fail(IRIS_ERR_INVALID, "bad bank kind");
    if (n_items < 1 || n_chan < 1) return fail(IRIS_ERR_INVALID, "empty bank");
    if (kind == IRIS_BANK_VOICE && (!labels || n_classes < 1))
        return fail(IRIS_ERR_INVALID, "voice bank needs labels [n_items, n_classes]");
    for (int i = 0; i < n_items; ++i)
        if (sample_rates[i] < 1 || offsets[i + 1] < offsets[i])
            return fail(IRIS_ERR_INVALID, "iris_bank_register_audio: bad argument");
    int rc = set_device(c);
    if (rc) return rc;
    std::vector<int64_t> n_in(n_items);
    for (int i = 0; i < n_items; ++i) n_in[i] = offsets[i + 1] - offsets[i];
    ResamplePlan plan;
    rc = resample_plan("iris_bank_register_audio", n_items, n_chan, n_in.data(), sample_rates, 16000, &plan);
    if (rc) return rc;
    std::vector<int64_t> off16(n_items + 1, 0);   // the items' 16 kHz lengths, cumulative
    for (int i = 0; i < n_items; ++i) off16[i + 1] = off16[i] + plan.n_out[i];
    rc = bank_layout(c, kind, n_items, n_chan, off16.data(), n_classes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t raw_floats = size_t(offsets[n_items] - offsets[0]) * n_chan;
    DevBuf raw, pcm16, blob;
    CU(raw.reserve(raw_floats * 4));
    CU(cudaMemcpyAsync(raw.p, wav + size_t(offsets[0]) * n_chan, raw_floats * 4, cudaMemcpyDefault, st));
    if (plan.copy_only)   // every item is 16 kHz: registered as iris_bank_register registers it
        return bank_fill(c, kind, raw, labels, normalize, st);
    // one copy of every item descriptor and filter table, one resample launch for the whole bank
    CU(blob.reserve(plan.blob.size()));
    CU(cudaMemcpyAsync(blob.p, plan.blob.data(), plan.blob.size(), cudaMemcpyHostToDevice, st));
    CU(pcm16.reserve(size_t(off16[n_items]) * n_chan * 4));
    CU(launch_resample(raw.as<float>(), pcm16.as<float>(), n_chan, blob.as<char>(), n_items, plan.n_ctas,
                       plan.chunk, plan.smem_floats, st));
    rc = bank_fill(c, kind, pcm16, labels, normalize, st);   // synchronises the stream
    raw.release();
    blob.release();
    return rc;
}


int iris_specbank_register(iris_ctx* c, int kind, int n_items, int n_freq, int n_chan2, const float* specs,
                           const int64_t* frame_offsets, const float* labels, int n_classes,
                           iris_stream stream) {
    if (!c || !specs || !frame_offsets) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (kind < 0 || kind > 2) return fail(IRIS_ERR_INVALID, "bad bank kind");
    if (n_items < 1) return fail(IRIS_ERR_INVALID, "empty bank");
    if (n_freq != kBins) return fail(IRIS_ERR_UNSUPPORTED, "spectrogram banks must have 257 frequency bins");
    if (n_chan2 < 2 || (n_chan2 & 1) || n_chan2 > 64)
        return fail(IRIS_ERR_INVALID, "last axis of a complex spectrogram must be 2 * chan (re | im)");
    if (kind == IRIS_BANK_VOICE && (!labels || n_classes < 1))
        return fail(IRIS_ERR_INVALID, "voice bank needs labels [n_items, n_classes]");
    int rc = set_device(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Bank& b = c->banks[kind];
    b.ready = false;
    b.spec = true;
    b.plane.release();   // spectrogram banks have none (k_specmix reads their bins directly)
    b.plane_floats = 0;
    b.n_items = n_items;
    b.n_chan = n_chan2 / 2;
    b.n_classes = n_classes;
    b.offsets.assign(frame_offsets, frame_offsets + n_items + 1);      // frames, cumulative
    b.pad_offsets.assign(n_items + 1, 0);
    b.n_frames.assign(n_items, 0);
    b.max_frames = 0;
    for (int i = 0; i < n_items; ++i) {
        const int64_t t = frame_offsets[i + 1] - frame_offsets[i];
        if (t < 1 || t > (1 << 24)) return fail(IRIS_ERR_INVALID, "spectrogram with no frames");
        b.n_frames[i] = int32_t(t);
        b.max_frames = std::max(b.max_frames, int(t));
        b.pad_offsets[i + 1] = frame_offsets[i + 1] - frame_offsets[0];
    }
    const size_t floats = size_t(b.pad_offsets[n_items]) * kBins * n_chan2;
    CU(b.padded.reserve(floats * 4));
    CU(b.d_n_frames.reserve(size_t(n_items) * 4));
    CU(cudaMemcpyAsync(b.padded.p, specs + size_t(frame_offsets[0]) * kBins * n_chan2, floats * 4,
                       cudaMemcpyDefault, st));
    CU(cudaMemcpyAsync(b.d_n_frames.p, b.n_frames.data(), size_t(n_items) * 4, cudaMemcpyHostToDevice, st));
    if (kind == IRIS_BANK_VOICE) {
        CU(b.labels.reserve(size_t(n_items) * n_classes * 4));
        CU(cudaMemcpyAsync(b.labels.p, labels, size_t(n_items) * n_classes * 4, cudaMemcpyHostToDevice, st));
        const size_t act_bytes = size_t(n_items) * b.max_frames;
        CU(b.activity.reserve(act_bytes));
        CU(cudaMemsetAsync(b.activity.p, 0, act_bytes, st));
        DevBuf d_off;
        CU(d_off.reserve(size_t(n_items + 1) * 8));
        CU(cudaMemcpyAsync(d_off.p, b.pad_offsets.data(), size_t(n_items + 1) * 8, cudaMemcpyHostToDevice, st));
        CU(launch_spec_activity(b.padded.as<float>(), d_off.as<int64_t>(), n_items, kBins, n_chan2,
                                b.max_frames, b.activity.as<uint8_t>(), st));
        b.h_activity.resize(act_bytes);
        CU(cudaMemcpyAsync(b.h_activity.data(), b.activity.p, act_bytes, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        d_off.release();
    }
    CU(cudaStreamSynchronize(st));
    b.ready = true;
    c->has_plan = false;
    return IRIS_OK;
}

int iris_bank_info(iris_ctx* c, int kind, int32_t* n_items, int32_t* n_chan, int32_t* n_frames) {
    if (!c || kind < 0 || kind > 2) return fail(IRIS_ERR_INVALID, "bad argument");
    const Bank& b = c->banks[kind];
    if (!b.ready) return fail(IRIS_ERR_STATE, "bank not registered");
    if (n_items) *n_items = b.n_items;
    if (n_chan) *n_chan = b.n_chan;
    if (n_frames) memcpy(n_frames, b.n_frames.data(), size_t(b.n_items) * 4);
    return IRIS_OK;
}

int iris_bank_activity(iris_ctx* c, int item, uint8_t* host_out) {
    if (!c || !host_out) return fail(IRIS_ERR_INVALID, "NULL argument");
    const Bank& b = c->banks[IRIS_BANK_VOICE];
    if (!b.ready) return fail(IRIS_ERR_STATE, "voice bank not registered");
    if (item < 0 || item >= b.n_items) return fail(IRIS_ERR_INVALID, "item out of range");
    memcpy(host_out, b.h_activity.data() + size_t(item) * b.max_frames, size_t(b.n_frames[item]));
    return IRIS_OK;
}

int iris_plan_upload(iris_ctx* c, const iris_plan* pl, iris_stream stream) {
    if (!c || !pl) return fail(IRIS_ERR_INVALID, "NULL argument");
    int rc = set_device(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int B = pl->batch, T = pl->n_frame, V = pl->max_voices, M = pl->max_noises;
    if (B < 1 || T < 1 || V < 0 || M < 0) return fail(IRIS_ERR_INVALID, "bad plan sizes");
    const Bank& bg = c->banks[IRIS_BANK_BG];
    const Bank& vb = c->banks[IRIS_BANK_VOICE];
    const Bank& nb = c->banks[IRIS_BANK_NOISE];
    if (!bg.ready) return fail(IRIS_ERR_STATE, "background bank not registered");
    if (V > 0 && !vb.ready) return fail(IRIS_ERR_STATE, "voice bank not registered");
    if (M > 0 && !nb.ready) return fail(IRIS_ERR_STATE, "noise bank not registered");
    if (!pl->bg_id || !pl->bg_offset) return fail(IRIS_ERR_INVALID, "bg_id / bg_offset NULL");
    if (V > 0 && (!pl->n_voices || !pl->voice_id || !pl->voice_gain || !pl->voice_offset))
        return fail(IRIS_ERR_INVALID, "voice draws NULL");
    if (M > 0 && (!pl->n_noises || !pl->noise_id || !pl->noise_gain || !pl->noise_offset))
        return fail(IRIS_ERR_INVALID, "noise draws NULL");
    const int C = bg.n_chan;
    if ((V > 0 && vb.n_chan != C) || (M > 0 && nb.n_chan != C))
        return fail(IRIS_ERR_INVALID, "all banks must have the same channel count");
    if ((V > 0 && vb.spec != bg.spec) || (M > 0 && nb.spec != bg.spec))
        return fail(IRIS_ERR_INVALID, "banks must be all waveforms or all spectrograms");
    const int n_tm = pl->time_masks ? pl->n_time_masks : 0;
    const int n_fm = pl->freq_masks ? pl->n_freq_masks : 0;
    if (n_tm < 0 || n_tm > 64) return fail(IRIS_ERR_UNSUPPORTED, "more than 64 time masks");
    if (n_fm < 0 || n_fm > 4) return fail(IRIS_ERR_UNSUPPORTED, "more than 4 frequency masks");
    const int c_out = remap_channels(pl->chan_remap, C, pl->n_out_chan);
    if (pl->chan_remap != IRIS_REMAP_NONE) {
        // data_utils.py:104 -- ValueError('This augment can be used in 2 channel audio')
        if (C != 2) return fail(IRIS_ERR_INVALID, "channel remap needs 2-channel audio");
        if (pl->chan_remap == IRIS_REMAP_MONO_CHAN) {
            if (pl->n_out_chan != 2) return fail(IRIS_ERR_INVALID, "mono_chan: n_out_chan must be 2");
        } else if (c_out < 3 || c_out > 16) {
            return fail(IRIS_ERR_INVALID, "bad n_out_chan");
        }
        if (pl->chan_remap == IRIS_REMAP_MERGE_AUG && !pl->merge_factor)
            return fail(IRIS_ERR_INVALID, "merge_factor NULL");
    }

    c->h_segs.clear();
    c->h_seg_len.clear();
    c->h_seg_ptr.assign(B + 1, 0);
    std::vector<int32_t> vshift(size_t(B) * (V > 0 ? V : 1), 0);
    std::vector<int32_t> vkt(size_t(B) * (V > 0 ? V : 1), 0);   // frames of the voice; 0 behind n_voices
    auto push = [&](const Bank& bank, int id, int shift, int lo, int hi, float gain, int keep_idx) {
        if (lo >= hi) return;
        Seg s;
        if (bank.spec) {   // k_spec.cu: base = the item's [257, tI, 2C] array, pair_stride = tI
            s.base = bank.padded.as<float>() + size_t(bank.pad_offsets[id]) * kBins * 2 * bank.n_chan;
            s.pair_stride = bank.n_frames[id];
        } else {
            const int64_t plen = 256 * (int64_t(bank.n_frames[id]) + 1);
            s.base = bank.padded.as<float>() + size_t(bank.pad_offsets[id]) * ((bank.n_chan + 1) / 2) * 2;
            s.pair_stride = int32_t(2 * plen);
        }
        s.shift = shift;
        s.t_lo = lo;
        s.t_hi = hi;
        s.gain = gain;
        s.keep_idx = keep_idx;
        c->h_segs.push_back(s);
        c->h_seg_len.push_back(bank.spec ? int64_t(bank.n_frames[id]) : bank.offsets[id + 1] - bank.offsets[id]);
    };
    char msg[160];
    int max_segs = 1;
    for (int b = 0; b < B; ++b) {
        // background: tile ceil(T/bgT) times, crop at bg_offset (pipeline.py:29-35)
        const int id = pl->bg_id[b];
        if (id < 0 || id >= bg.n_items) return fail(IRIS_ERR_INVALID, "bg_id out of range");
        const int bgT = bg.n_frames[id];
        const int reps = (T + bgT - 1) / bgT;
        const int ob = pl->bg_offset[b];
        if (ob < 0 || ob > bgT * reps - T) {
            snprintf(msg, sizeof msg, "clip %d: bg_offset %d outside [0, %d]", b, ob, bgT * reps - T);
            return fail(IRIS_ERR_INVALID, msg);
        }
        for (int r = 0; r <= reps; ++r) {
            const int lo = std::max(0, r * bgT - ob), hi = std::min(T, (r + 1) * bgT - ob);
            push(bg, id, ob - r * bgT, lo, hi, 1.f, -1);
        }
        // voices (pipeline.py:41-84)
        if (V > 0) {
            int nv = pl->n_voices[b];
            if (V == 1) nv = 1;
            if (nv < 0 || (V > 1 && nv >= V)) {
                snprintf(msg, sizeof msg, "clip %d: n_voices %d outside [1, %d)", b, nv, V);
                return fail(IRIS_ERR_INVALID, msg);
            }
            int vP = 0;   // padded_batch: the group's longest member (pipeline.py:155-156)
            for (int v = 0; v < V; ++v) {
                const int vid = pl->voice_id[size_t(b) * V + v];
                if (vid < 0 || vid >= vb.n_items) return fail(IRIS_ERR_INVALID, "voice_id out of range");
                vP = std::max(vP, int(vb.n_frames[vid]));
            }
            for (int v = 0; v < nv; ++v) {
                const int vid = pl->voice_id[size_t(b) * V + v];
                // pad_size = n_frame - int32(min_ratio * float32(v_frame))   (pipeline.py:58-59)
                const int pad = T - int(int32_t(float(pl->min_ratio) * float(vP)));
                const int len = pad > 0 ? vP + 2 * pad : vP;
                const int s0 = pad > 0 ? pad : 0;
                const int maxval = len - T;
                if (maxval <= 0) {
                    snprintf(msg, sizeof msg,
                             "clip %d voice %d: empty offset range [0, %d) (pipeline.py:68-69 raises)",
                             b, v, maxval);
                    return fail(IRIS_ERR_EMPTY_RANGE, msg);
                }
                const int off = pl->voice_offset[size_t(b) * V + v];
                if (off < 0 || off >= maxval) {
                    snprintf(msg, sizeof msg, "clip %d voice %d: offset %d outside [0, %d)", b, v, off, maxval);
                    return fail(IRIS_ERR_INVALID, msg);
                }
                const int shift = off - s0;
                vshift[size_t(b) * V + v] = shift;
                const int kT = vb.n_frames[vid];
                vkt[size_t(b) * V + v] = kT;
                push(vb, vid, shift, std::max(0, -shift), std::min(T, kT - shift),
                     pl->voice_gain[size_t(b) * V + v], b * V + v);
            }
        }
        // noises (pipeline.py:86-106)
        if (M > 0) {
            const int nn = pl->n_noises[b];
            if (nn < 0 || nn >= M) {
                snprintf(msg, sizeof msg, "clip %d: n_noises %d outside [0, %d)", b, nn, M);
                return fail(IRIS_ERR_INVALID, msg);
            }
            int nP = 0;
            for (int n = 0; n < M; ++n) {
                const int nid = pl->noise_id[size_t(b) * M + n];
                if (nid < 0 || nid >= nb.n_items) return fail(IRIS_ERR_INVALID, "noise_id out of range");
                nP = std::max(nP, int(nb.n_frames[nid]));
            }
            for (int n = 0; n < nn; ++n) {
                const int nid = pl->noise_id[size_t(b) * M + n];
                const int pad = T - int(int32_t(float(pl->min_noise_ratio) * float(nP)));
                const int len = pad > 0 ? nP + 2 * pad : nP;
                const int s0 = pad > 0 ? pad : 0;
                const int off = pl->noise_offset[size_t(b) * M + n];
                if (len < T || off < 0 || off > len - T) {
                    snprintf(msg, sizeof msg, "clip %d noise %d: offset %d outside [0, %d]", b, n, off, len - T);
                    return fail(IRIS_ERR_INVALID, msg);
                }
                const int shift = off - s0;
                const int kT = nb.n_frames[nid];
                push(nb, nid, shift, std::max(0, -shift), std::min(T, kT - shift),
                     pl->noise_gain[size_t(b) * M + n], -1);
            }
        }
        c->h_seg_ptr[b + 1] = int32_t(c->h_segs.size());
        max_segs = std::max(max_segs, c->h_seg_ptr[b + 1] - c->h_seg_ptr[b]);
        if (!bg.spec && c->h_seg_ptr[b + 1] - c->h_seg_ptr[b] > fused_max_segments()) {
            snprintf(msg, sizeof msg, "clip %d mixes %d segments; the fused kernel takes at most %d", b,
                     c->h_seg_ptr[b + 1] - c->h_seg_ptr[b], fused_max_segments());
            return fail(IRIS_ERR_UNSUPPORTED, msg);
        }
        // mask draws (transforms.py:25-26)
        for (int i = 0; i < n_tm; ++i) {
            const int size = pl->time_masks[(size_t(b) * n_tm + i) * 2];
            const int off = pl->time_masks[(size_t(b) * n_tm + i) * 2 + 1];
            if (size < 0 || off < 0 || off + size > T) return fail(IRIS_ERR_INVALID, "time mask outside the clip");
        }
        for (int i = 0; i < n_fm; ++i) {
            const int size = pl->freq_masks[(size_t(b) * n_fm + i) * 2];
            const int off = pl->freq_masks[(size_t(b) * n_fm + i) * 2 + 1];
            if (size < 0 || off < 0 || off + size > kBins) return fail(IRIS_ERR_INVALID, "freq mask outside the spectrum");
        }
    }

    // ---- pack everything into one pinned blob, one H2D copy ----
    const int n_extra = (pl->chan_remap == IRIS_REMAP_MERGE_AUG) ? c_out - 2 : 0;
    size_t o = 0;
    const size_t o_segs = o; o = align_up(o + c->h_segs.size() * sizeof(Seg), 16);
    const size_t o_ptr = o;  o = align_up(o + size_t(B + 1) * 4, 16);
    const size_t o_nv = o;   o = align_up(o + size_t(B) * 4, 16);
    const size_t o_vid = o;  o = align_up(o + size_t(B) * std::max(V, 1) * 4, 16);
    const size_t o_vsh = o;  o = align_up(o + size_t(B) * std::max(V, 1) * 4, 16);
    const size_t o_vkt = o;  o = align_up(o + size_t(B) * std::max(V, 1) * 4, 16);
    const size_t o_tm = o;   o = align_up(o + size_t(B) * n_tm * 8, 16);
    const size_t o_fm = o;   o = align_up(o + size_t(B) * n_fm * 8, 16);
    const size_t o_mf = o;   o = align_up(o + size_t(B) * n_extra * 4, 16);
    const size_t o_msf = o;  o = align_up(o + size_t(B) * n_extra * 4, 16);
    const size_t total = o;
    const int slot = c->stage_next;
    c->stage_next = (slot + 1) % iris_ctx::kStageRing;
    if (c->h_stage[slot]) CU(cudaEventSynchronize(c->stage_free[slot]));   // the upload that used it has drained
    rc = ensure_stage(c, slot, total);
    if (rc) return rc;
    // The blob travels on the context's copy stream into a ring of device blobs, so that the
    // upload of batch i + 1 overlaps the kernels of batch i.  Slot reuse: blob_used[s] (recorded on
    // the caller's stream at the NEXT upload) marks the end of every kernel that read blob s.
    if (!c->copy) {
        CU(cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking));
        for (int i = 0; i < iris_ctx::kStageRing; ++i) {
            CU(cudaEventCreateWithFlags(&c->blob_ready[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&c->blob_used[i], cudaEventDisableTiming));
        }
    }
    const int prev = (slot + iris_ctx::kStageRing - 1) % iris_ctx::kStageRing;
    CU(cudaEventRecord(c->blob_used[prev], st));
    c->blob_used_valid[prev] = true;
    DevBuf& blob = c->plan_blobs[slot];
    if (c->blob_used_valid[slot]) {
        if (total > blob.cap) CU(cudaEventSynchronize(c->blob_used[slot]));   // about to free it
        else CU(cudaStreamWaitEvent(c->copy, c->blob_used[slot], 0));
    }
    CU(blob.reserve(total));
    char* h = static_cast<char*>(c->h_stage[slot]);
    memcpy(h + o_segs, c->h_segs.data(), c->h_segs.size() * sizeof(Seg));
    memcpy(h + o_ptr, c->h_seg_ptr.data(), size_t(B + 1) * 4);
    if (V > 0) {
        int32_t* nv = reinterpret_cast<int32_t*>(h + o_nv);
        for (int b = 0; b < B; ++b) nv[b] = (V == 1) ? 1 : pl->n_voices[b];
        memcpy(h + o_vid, pl->voice_id, size_t(B) * V * 4);
        memcpy(h + o_vsh, vshift.data(), size_t(B) * V * 4);
        memcpy(h + o_vkt, vkt.data(), size_t(B) * V * 4);
    }
    if (n_tm) memcpy(h + o_tm, pl->time_masks, size_t(B) * n_tm * 8);
    if (n_fm) memcpy(h + o_fm, pl->freq_masks, size_t(B) * n_fm * 8);
    if (n_extra) {
        memcpy(h + o_mf, pl->merge_factor, size_t(B) * n_extra * 4);
        float* sf = reinterpret_cast<float*>(h + o_msf);
        for (size_t i = 0; i < size_t(B) * n_extra; ++i) sf[i] = sqrtf(1.f - pl->merge_factor[i]);
    }
    CU(cudaMemcpyAsync(blob.p, h, total, cudaMemcpyHostToDevice, c->copy));
    CU(cudaEventRecord(c->stage_free[slot], c->copy));
    CU(cudaEventRecord(c->blob_ready[slot], c->copy));
    CU(cudaStreamWaitEvent(st, c->blob_ready[slot], 0));
    c->last_upload_bytes = total;
    char* d = blob.as<char>();
    c->d_segs = reinterpret_cast<Seg*>(d + o_segs);
    c->d_seg_ptr = reinterpret_cast<int32_t*>(d + o_ptr);
    c->d_n_voices = reinterpret_cast<int32_t*>(d + o_nv);
    c->d_voice_id = reinterpret_cast<int32_t*>(d + o_vid);
    c->d_voice_shift = reinterpret_cast<int32_t*>(d + o_vsh);
    c->d_voice_kt = reinterpret_cast<int32_t*>(d + o_vkt);
    c->d_tmask = n_tm ? reinterpret_cast<int32_t*>(d + o_tm) : nullptr;
    c->d_fmask = n_fm ? reinterpret_cast<int32_t*>(d + o_fm) : nullptr;
    c->d_merge_f = n_extra ? reinterpret_cast<float*>(d + o_mf) : nullptr;
    c->d_merge_sf = n_extra ? reinterpret_cast<float*>(d + o_msf) : nullptr;
    c->B = B; c->T = T; c->V = V; c->M = M; c->C = C;
    c->n_tmask = n_tm; c->n_fmask = n_fm;
    c->filter_k = pl->stft_filter > 0 ? pl->stft_filter : 0;
    c->remap = pl->chan_remap;
    c->c_out = c_out;
    c->max_segs = max_segs;
    c->spec_mode = bg.spec;
    c->has_plan = true;
    c->labels_done = false;
    c->tile_sig.valid = false;
    return IRIS_OK;
}

int iris_labels(iris_ctx* c, float* d_vtk, float* d_frame, uint8_t* d_keep, iris_stream stream) {
    if (!c) return fail(IRIS_ERR_INVALID, "NULL ctx");
    if (!c->has_plan) return fail(IRIS_ERR_STATE, "no plan uploaded");
    int rc = set_device(c);
    if (rc) return rc;
    return run_labels(c, d_vtk, d_frame, d_keep, static_cast<cudaStream_t>(stream), c->feat_hint);
}

int iris_features(iris_ctx* c, int mode, float* d_out, iris_stream stream) {
    return iris_features_select(c, mode, IRIS_SELECT_ALL, d_out, stream);
}

int iris_features_select(iris_ctx* c, int mode, int select, float* d_out, iris_stream stream) {
    if (!c || !d_out) return fail(IRIS_ERR_INVALID, "NULL argument");
    int out_type = OUT_F32;
    if (!split_feature_mode(mode, &mode, &out_type))
        return fail(IRIS_ERR_INVALID, "bad feature mode: at most one of IRIS_OUT_BF16 / IRIS_OUT_F16 above the mode");
    if (mode == IRIS_FEAT_SE && out_type != OUT_F32)
        return fail(IRIS_ERR_INVALID, "IRIS_FEAT_SE writes float32 blocks: no IRIS_OUT_* flag");
    if (reinterpret_cast<uintptr_t>(d_out) & 15)
        return fail(IRIS_ERR_INVALID, "the feature buffer must be 16-byte aligned (vector stores)");
    if (select < IRIS_SELECT_ALL || select > IRIS_SELECT_BG_NOISE) return fail(IRIS_ERR_INVALID, "bad segment selection");
    if (select != IRIS_SELECT_ALL && mode != IRIS_FEAT_COMPLEX)
        return fail(IRIS_ERR_INVALID, "only_voice / only_noise are complex spectrograms (pipeline.py:37-38)");
    if (!c->has_plan) return fail(IRIS_ERR_STATE, "no plan uploaded");
    if ((mode < IRIS_FEAT_COMPLEX || mode > IRIS_FEAT_LOGMEL_MINMAX) && mode != IRIS_FEAT_SE)
        return fail(IRIS_ERR_INVALID, "bad feature mode");
    if (mode == IRIS_FEAT_SE && (c->C != 2 || c->remap != IRIS_REMAP_NONE))
        return fail(IRIS_ERR_UNSUPPORTED, "IRIS_FEAT_SE takes 2-channel plans without a channel remap");
    int rc = set_device(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!c->labels_done) {   // accept flags of the voices are an input of the mix
        rc = run_labels(c, nullptr, nullptr, nullptr, st, select == IRIS_SELECT_ALL ? mode : -1);
        if (rc) return rc;
    }
    const bool mel = mel_mode(mode);
    if (mel && c->n_mel == 0) return fail(IRIS_ERR_STATE, "iris_set_mel not called");
    if (c->spec_mode) return spec_features(c, mode, select, d_out, st, out_type);
    if (mel && !c->mel_fusable)
        return fail(IRIS_ERR_UNSUPPORTED,
                    "a mel filter wider than 16 bins (or more than 64 taps over the 32-filter rounds): run "
                    "IRIS_FEAT_MAGPHASE + iris_op_mel instead of the fused mel epilogue");
    FusedParams p;
    rc = feature_params(c, mode, select, p);
    if (rc) return rc;
    p.out = d_out;
    c->feat_hint = select == IRIS_SELECT_ALL ? mode : -1;
    if (mel) {
        if (p.do_minmax) {   // per-clip (~min, max) bit patterns; k_logmel_post leaves them
                             // zeroed, so only a fresh allocation is cleared
            const void* before = c->minmax.p;
            CU(c->minmax.reserve(size_t(c->B) * 12));   // [B,2] min/max words + [B] k_logmel_post counters
            if (c->minmax.p != before) CU(cudaMemsetAsync(c->minmax.p, 0, c->minmax.cap, st));
            p.minmax = c->minmax.as<uint32_t>();
            if (out_type != OUT_F32) {   // k_fused writes fp32 mel + extrema to scratch, k_logmel_post converts
                rc = mel_scratch(c, &p.out);
                if (rc) return rc;
            }
        }
        rc = p.do_minmax ? run_logmel_minmax(c, p, d_out, st, out_type) : timed_fused(c, p, FM_MEL, st, out_type);
        if (rc) return rc;
    } else {
        rc = timed_fused(c, p, mode == IRIS_FEAT_SE ? FM_SE : mode, st, out_type);
    }
    if (rc) return rc;
    return IRIS_OK;
}

int iris_stft(iris_ctx* c, const float* wav, int n_chan, int64_t n, int normalize, float* d_out,
              iris_stream stream) {
    if (!c || !wav || !d_out) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (n_chan < 1 || n <= kNFft / 2) return fail(IRIS_ERR_INVALID, "need n_samples > 256");
    int rc = set_device(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t kT = 1 + n / kHop, plen = 256 * (kT + 1);
    if (n_chan > 32) return fail(IRIS_ERR_UNSUPPORTED, "more than 32 channels");
    const int n_pairs = (n_chan + 1) / 2;
    // Seg::pair_stride (floats between pair planes) is an int32_t; only a second pair plane uses it
    if (n_pairs > 1 && 2 * plen > INT32_MAX)
        return fail(IRIS_ERR_UNSUPPORTED, "iris_stft: 3 or more channels of more than 1073741311 samples "
                                          "(pair stride above 2^31 - 1)");
    CU(c->stft_pad.reserve((size_t(plen) * n_pairs * 2 + size_t(n) * n_chan) * 4));
    CU(c->stft_small.reserve(256));
    float* P = c->stft_pad.as<float>();
    float* raw = P + size_t(plen) * n_pairs * 2;
    CU(cudaMemcpyAsync(raw, wav, size_t(n) * n_chan * 4, cudaMemcpyDefault, st));
    struct Small { int64_t off[2]; int64_t poff[2]; Seg seg; int32_t ptr[2]; } h;
    h.off[0] = 0; h.off[1] = n; h.poff[0] = 0; h.poff[1] = plen;
    h.seg.base = P; h.seg.pair_stride = int32_t(2 * plen);
    h.seg.shift = 0; h.seg.t_lo = 0; h.seg.t_hi = int32_t(kT); h.seg.gain = 1.f;
    h.seg.keep_idx = -1;
    h.ptr[0] = 0; h.ptr[1] = 1;
    CU(cudaMemcpyAsync(c->stft_small.p, &h, sizeof h, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));   // h is on the stack
    Small* d = c->stft_small.as<Small>();
    CU(launch_bank_prepare(raw, d->off, d->poff, 1, n_chan, normalize, P, st));
    FusedParams p;
    fill_common(c, p);
    p.segs = &d->seg;
    p.seg_ptr = d->ptr;
    p.B = 1; p.T = int32_t(kT);
    set_geometry(c, p, n_chan, false);
    p.out = d_out;
    rc = run_fused(c, p, FM_COMPLEX, 1, st);
    c->tile_sig.valid = false;   // the one-segment list of this call is rewritten by the next one
    return rc;
}

int iris_metric_counts(iris_ctx* c, const float* y_true, const float* y_pred, int B, int T, int K,
                       float thr, int32_t* d_triples, uint64_t* d_tpfpfn, uint64_t* d_sums,
                       float* d_er, iris_stream stream) {
    if (!c || !y_true || !y_pred || !d_triples) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (B < 1 || T < 1 || K < 1) return fail(IRIS_ERR_INVALID, "bad shape");
    int rc = set_device(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CU(launch_metric_counts(y_true, y_pred, B, T, T, K, thr, d_triples,
                            reinterpret_cast<unsigned long long*>(d_tpfpfn),
                            reinterpret_cast<unsigned long long*>(d_sums), st));
    if (d_er) CU(launch_er_finalize(d_triples, B, d_er, st));
    return IRIS_OK;
}

int iris_er_counts_pooled(iris_ctx* c, const float* y_true, int T, const float* y_pred, int T_pred, int B,
                          int K, float thr, int32_t* d_triples, float* d_er, iris_stream stream) {
    if (!c || !y_true || !y_pred || !d_triples) return fail(IRIS_ERR_INVALID, "NULL argument");
    if (B < 1 || T < 1 || T_pred < 1 || K < 1) return fail(IRIS_ERR_INVALID, "bad shape");
    int rc = set_device(c);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CU(launch_metric_counts(y_true, y_pred, B, T, T_pred, K, thr, d_triples, nullptr, nullptr, st));
    if (d_er) CU(launch_er_finalize(d_triples, B, d_er, st));
    return IRIS_OK;
}

int iris_debug_claims(int64_t n_tiles, int grid, int chunk, int pair_merge, int64_t q, int32_t* schedule5,
                      int64_t* first, int32_t* len) {
    if (n_tiles < 0 || grid < 1 || chunk < 1 || !schedule5 || !first || !len)
        return fail(IRIS_ERR_INVALID, "iris_debug_claims: bad argument");
    fused_debug_schedule(n_tiles, grid, chunk, pair_merge, schedule5);
    int l = 0;
    *first = claim_range(schedule5[0], schedule5[1], schedule5[2], schedule5[3], schedule5[4], q, l);
    *len = l;
    return IRIS_OK;
}

int iris_profile_enable(iris_ctx* c, int enable) {
    if (!c) return fail(IRIS_ERR_INVALID, "NULL ctx");
    c->profile = enable != 0;
    return IRIS_OK;
}

int iris_profile_read(iris_ctx* c, double* total_ms, int32_t* n_launches, int reset) {
    if (!c) return fail(IRIS_ERR_INVALID, "NULL ctx");
    double tot = 0.0;
    for (size_t i = 0; i < c->prof_used; ++i) {
        CU(cudaEventSynchronize(c->prof_events[i].second));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, c->prof_events[i].first, c->prof_events[i].second));
        tot += ms;
    }
    if (total_ms) *total_ms = tot;
    if (n_launches) *n_launches = int32_t(c->prof_used);
    if (reset) c->prof_used = 0;
    return IRIS_OK;
}

int iris_plan_bytes(iris_ctx* c, int mode, const uint8_t* host_keep, int64_t* bytes_in,
                    int64_t* bytes_out) {
    return iris_plan_bytes_clips(c, mode, host_keep, 0, c ? c->B : 0, bytes_in, bytes_out);
}

int iris_profile_clips(iris_ctx* c) { return c ? c->prof_clips : 0; }

int iris_plan_bytes_clips(iris_ctx* c, int mode, const uint8_t* host_keep, int clip_lo, int clip_hi,
                          int64_t* bytes_in, int64_t* bytes_out) {
    if (!c || !c->has_plan) return fail(IRIS_ERR_STATE, "no plan uploaded");
    if (clip_lo < 0 || clip_hi > c->B || clip_lo > clip_hi) return fail(IRIS_ERR_INVALID, "bad clip range");
    int out_type = OUT_F32;
    if (!split_feature_mode(mode, &mode, &out_type))
        return fail(IRIS_ERR_INVALID, "bad feature mode: at most one of IRIS_OUT_BF16 / IRIS_OUT_F16 above the mode");
    if (mode == IRIS_FEAT_SE && out_type != OUT_F32)
        return fail(IRIS_ERR_INVALID, "IRIS_FEAT_SE writes float32 blocks: no IRIS_OUT_* flag");
    const int64_t out_elem = out_type == OUT_F32 ? 4 : 2;
    int64_t in = 0;
    for (size_t i = size_t(c->h_seg_ptr[clip_lo]); i < size_t(c->h_seg_ptr[clip_hi]); ++i) {
        const Seg& s = c->h_segs[i];
        if (s.keep_idx >= 0 && host_keep && !host_keep[s.keep_idx]) continue;
        // frames [t_lo, t_hi) read the samples of rows t_lo+shift .. t_hi+shift once,
        // never more than the source holds
        if (c->spec_mode) {   // [257, frames, 2C] cells of the frames the segment covers
            // the mel modes need only the bin rows that carry a non-zero mel weight
            const int rows = mel_mode(mode) ? c->mel_f_n : mode == IRIS_FEAT_SE ? kBins - 1 : kBins;
            in += int64_t(s.t_hi - s.t_lo) * rows * 2 * c->C * 4;
            continue;
        }
        const int64_t samples = std::min<int64_t>(int64_t(s.t_hi - s.t_lo + 1) * 256, c->h_seg_len[i]);
        in += samples * 4 * c->C;
    }
    int64_t out;
    if (mode == IRIS_FEAT_SE) out = int64_t(clip_hi - clip_lo) * (kBins - 1) * c->T * 2 * c->C * out_elem;   // C + C/2 + C/2
    else if (mel_mode(mode)) out = int64_t(clip_hi - clip_lo) * c->n_mel * c->T * c->c_out * out_elem;
    else out = int64_t(clip_hi - clip_lo) * kBins * c->T * spec_width(mode, c->remap, c->c_out) * out_elem;
    if (bytes_in) *bytes_in = in;
    if (bytes_out) *bytes_out = out;
    return IRIS_OK;
}

}  // extern "C"
