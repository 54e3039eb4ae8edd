// Frame-label construction and same-class overlap rejection of
// pipeline.merge_complex_specs (pipeline.py:41-84) + data_utils.to_frame_labels
// (data_utils.py:64-70), as an integer-exact kernel over precomputed per-frame
// activity flags (activity = reduce_max(voice, (f, 2C)) > 0, pipeline.py:55).
// One CTA per clip; voices are visited in order because acceptance of voice v depends
// on the labels of the voices accepted before it (pipeline.py:78-84).
#include <cstring>

#include "iris_common.cuh"
#include "iris_launch.h"
#include "iris_tiles.cuh"

namespace iris {

// Shared memory: the running frame labels L[T*K] (float) and the activity bytes of the
// clip's voices act[V][T], gathered up front so that the sequential per-voice passes run from
// shared memory (one global round trip per clip instead of two per voice).
// build_tiles: the CTA also writes the tile blocks of its clip (iris_tiles.cuh) for the k_fused
// launch behind it: the keep flags it has just decided are their only input that is not in the plan.
// SE: the tile blocks are those of an FM_SE launch (build_tile_block; its own instance, as the run-time
// choice spills this kernel)
template <bool SE>
__global__ void __launch_bounds__(1024) k_labels(const LabelParams p, const int build_tiles,
                                                 const __grid_constant__ FusedParams fp) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int b = blockIdx.x;
    // a feature kernel launched behind this one with programmatic stream serialization may start
    // its prologue; it waits for the whole grid before it reads a tile block
    cudaTriggerProgrammaticLaunchCompletion();
    const int TK = p.T * p.K;
    float* L = reinterpret_cast<float*>(s_raw);                       // [T*K]
    float* lab = L + TK;                                               // [V*K]
    uint8_t* act = reinterpret_cast<uint8_t*>(lab + p.V * p.K);       // [V][T]
    const int nv = p.n_voices[b];
    for (int i = threadIdx.x; i < TK; i += blockDim.x) L[i] = 0.f;
    // per-voice metadata first (ids / shifts / frame counts: one round trip), then
    // ONE flattened gather of all V x T activity bytes: the loads are independent, so they
    // pipeline instead of paying a memory round trip per voice
    __shared__ int s_id[64], s_shift[64], s_kT[64];
    // tile lists (build_tiles): the clip's segment range rides on the metadata round trip, its segments
    // and mask rectangles on the activity gather, the keep flags stay in shared memory -- the tile
    // threads at the end touch no global memory but their own blocks
    __shared__ int s_seg0, s_nseg;
    __shared__ Seg s_segs[kMaxStages + 8];
    __shared__ uint8_t s_kept[kMaxStages + 8];
    __shared__ uint8_t s_keepv[64];
    __shared__ int32_t s_tm[32], s_fm[32];
    if (build_tiles && threadIdx.x == 32) {
        s_seg0 = fp.seg_ptr[b];
        s_nseg = fp.seg_ptr[b + 1] - s_seg0;
    }
    for (int v = threadIdx.x; v < p.V; v += blockDim.x) {
        // one round trip: the frame count of the voice comes with the plan (0 behind n_voices)
        s_id[v] = p.voice_id[size_t(b) * p.V + v];
        s_shift[v] = p.voice_shift[size_t(b) * p.V + v];
        s_kT[v] = p.voice_kt[size_t(b) * p.V + v];
    }
    __syncthreads();
    {
        int v = 0, t = threadIdx.x;
        while (t >= p.T && v < p.V) { t -= p.T; ++v; }
#pragma unroll 4
        for (int i = threadIdx.x; i < p.V * p.T; i += blockDim.x) {
            const int k = t + s_shift[v];
            act[i] = (k >= 0 && k < s_kT[v]) ? p.activity[size_t(s_id[v]) * p.act_stride + k] : uint8_t(0);
            t += blockDim.x;
            while (t >= p.T && v + 1 < p.V) { t -= p.T; ++v; }
        }
    }
    for (int i = threadIdx.x; i < p.V * p.K; i += blockDim.x) {
        const int v = i / p.K;
        lab[i] = v < nv ? p.bank_labels[size_t(s_id[v]) * p.K + (i - v * p.K)] : 0.f;
    }
    const bool seg_cached = build_tiles && s_nseg <= kMaxStages + 8 && fp.n_tmask <= 16 && fp.n_fmask <= 16;
    if (seg_cached) {
        const int t = int(blockDim.x) - 1 - int(threadIdx.x);   // the last threads: the first ones carry the gather's tail
        if (t < s_nseg) s_segs[t] = fp.segs[s_seg0 + t];
        if (fp.tmask && t < 2 * fp.n_tmask) s_tm[t] = fp.tmask[size_t(b) * fp.n_tmask * 2 + t];
        if (fp.fmask && t < 2 * fp.n_fmask) s_fm[t] = fp.fmask[size_t(b) * fp.n_fmask * 2 + t];
    }
    __syncthreads();
    for (int v = 0; v < p.V; ++v) {
        float* lv = p.labels_vtk ? p.labels_vtk + (size_t(b) * p.V + v) * TK : nullptr;
        if (v >= nv) {   // uniform
            if (lv) for (int i = threadIdx.x; i < TK; i += blockDim.x) lv[i] = 0.f;
            if (threadIdx.x == 0) { p.keep[size_t(b) * p.V + v] = 0; s_keepv[v] = 0; }
            continue;
        }
        const uint8_t* av = act + v * p.T;
        const float* lb = lab + v * p.K;
        // no_overlap = max over (t, c) of (sum of accepted labels + candidate) < 2  (pipeline.py:78-79)
        //            = no element reaches 2: one block-wide OR instead of a max reduction.  Thread
        // x owns frames x, x + blockDim, ... for every voice, so L needs no barrier of its own.
        int hit = 0;
        for (int t = threadIdx.x; t < p.T; t += blockDim.x) {
            const float a = av[t] ? 1.f : 0.f;
            for (int c = 0; c < p.K; ++c) hit |= (L[t * p.K + c] + lb[c] * a >= 2.f);
        }
        const int keep_i = __syncthreads_or(hit) ? 0 : 1;
        if (threadIdx.x == 0) { p.keep[size_t(b) * p.V + v] = uint8_t(keep_i); s_keepv[v] = uint8_t(keep_i); }
        const float keep = keep_i ? 1.f : 0.f;
        for (int t = threadIdx.x; t < p.T; t += blockDim.x) {
            const float a = av[t] ? 1.f : 0.f;
            for (int c = 0; c < p.K; ++c) {
                const float cand = lb[c] * a * keep;              // l * no_overlap (pipeline.py:84)
                L[t * p.K + c] += cand;
                if (lv) lv[t * p.K + c] = cand;
            }
        }
    }
    __syncthreads();   // the final copy below walks L with another thread-to-element map
    float* out = p.frame_labels + size_t(b) * TK;
    for (int i = threadIdx.x; i < TK; i += blockDim.x) out[i] = L[i];
    if (build_tiles) {   // (the barrier above also orders thread 0's keep flags before these reads)
        const int per_clip = ((fp.T + fp.fr - 1) / fp.fr) * fp.n_pairs;
        if (seg_cached) {
            // keep_idx of a voice segment is b * V + v (iris_plan_upload): its flag is in shared memory
            if (int(threadIdx.x) < s_nseg) {
                const int ki = s_segs[threadIdx.x].keep_idx;
                s_kept[threadIdx.x] = ki < 0 ? 1 : s_keepv[ki - b * p.V];
            }
            __syncthreads();
        }
        for (int r = threadIdx.x; r < per_clip; r += blockDim.x)
            build_tile_block<SE>(fp, b * per_clip + r, per_clip, seg_cached ? s_segs : nullptr, seg_cached ? s_kept : nullptr,
                                 seg_cached ? s_tm : nullptr, seg_cached ? s_fm : nullptr);
    }
}

cudaError_t launch_labels(const LabelParams& p, cudaStream_t stream, const FusedParams* tiles) {
    if (p.B <= 0) return cudaSuccess;
    const size_t smem = (size_t(p.T) * p.K + size_t(p.V) * p.K) * 4 + size_t(p.V) * p.T;
    if (smem > 200 * 1024 || p.V > 64) return cudaErrorInvalidValue;
    const bool se = tiles && tiles->seg_select == 3;
    static bool attr_set[2] = {false, false};
    if (smem > 48 * 1024 && !attr_set[se]) {
        cudaError_t e = cudaFuncSetAttribute(se ? k_labels<true> : k_labels<false>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[se] = true;
    }
    // 1024 threads per clip: one frame per thread, so the sequential per-voice passes are a
    // handful of instructions per warp (256 threads measured 17 us, latency-bound)
    if (tiles && (tiles->keep != p.keep || tiles->B != p.B)) return cudaErrorInvalidValue;
    FusedParams none;
    if (!tiles) memset(&none, 0, sizeof none);
    // one wave of clips (two 1024-thread CTAs per SM): one frame per thread is fastest; larger batches run in
    // several waves and the kernel is latency-bound per CTA, so half-size CTAs (four per SM) finish sooner
    // (1024 clips: step 0.82 -> 0.81 ms; 256 clips: 226.3 vs 226.7 us)
    const int threads = p.B > 296 ? 512 : 1024;
    if (se) k_labels<true><<<p.B, threads, smem, stream>>>(p, 1, *tiles);
    else k_labels<false><<<p.B, threads, smem, stream>>>(p, tiles ? 1 : 0, tiles ? *tiles : none);
    return cudaGetLastError();
}

}  // namespace iris
