// Host-callable launchers of the libiris kernels (internal; the public surface is include/iris.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace iris {

struct FusedParams;

// build_tiles: k_tiles builds the tile blocks first; false: the kernel in front (k_labels) wrote them.
// out_type: OutType (iris_common.cuh) of p.out
cudaError_t launch_fused(const FusedParams& p, int mode, int num_sms, cudaStream_t stream, bool build_tiles,
                         int out_type);
size_t fused_smem_bytes(const FusedParams& p, int mode);
bool fused_reads_plane(const FusedParams& p, int mode);   // FusedParams::plane of a launch
void fused_debug_schedule(long long n_tiles, int grid, int chunk, int pair_merge, int32_t out[5]);
int fused_max_segments();      // mixing segments one clip may have
bool fused_stages_output(int mode, int remap, int fr);   // FusedParams::stage_out for a launch
int fused_max_mel_taps();      // sum over the 32-filter rounds of the longest filter
int fused_max_mel_filter();    // taps of the longest filter
int fused_pick_fr(int mel_taps);   // frames per tile (consumer warps per CTA)
size_t fused_tile_bytes(const FusedParams& p, int* stride_out);   // size of p.tile_blocks

// k_post.cu -- from the fp32 features at src into dst of OutType out_type.  src == dst: in place (OUT_F32
// only), nothing to do without do_minmax or do_log; src != dst: with neither flag it only converts.
// minmax: [B,2] extrema words of the clips at src; done: [B] zeroed counters (both may be null without do_minmax)
cudaError_t launch_logmel_post(const float* src, void* dst, int out_type, uint32_t* minmax, unsigned* done, int B,
                               size_t per_clip, int do_minmax, int do_log, cudaStream_t stream);

// k_bank.cu
cudaError_t launch_bank_prepare(const float* wav, const int64_t* d_offsets, const int64_t* d_pad_offsets,
                                int n_items, int n_chan, int normalize, float* padded,
                                cudaStream_t stream);

// k_labels.cu
struct LabelParams {
    int B, T, V, K;
    const int32_t* n_voices;     // [B]
    const int32_t* voice_id;     // [B,V]
    const int32_t* voice_shift;  // [B,V]  source frame k = t + shift
    const int32_t* voice_kt;     // [B,V]  frames of the voice (0 behind n_voices): n_frames[voice_id], resolved on the host
    const int32_t* n_frames;     // [n_items] true frame count of each voice
    const uint8_t* activity;     // [n_items, act_stride]
    int act_stride;
    const float* bank_labels;    // [n_items, K]
    float* labels_vtk;           // [B,V,T,K] or null
    float* frame_labels;         // [B,T,K]
    uint8_t* keep;               // [B,V]
};
// tiles != null: every CTA also builds the tile blocks of its clip for the k_fused launch that
// follows (tiles->keep must be p.keep, tiles->tile_blocks sized by fused_tile_bytes)
cudaError_t launch_labels(const LabelParams& p, cudaStream_t stream, const FusedParams* tiles = nullptr);

// k_metrics.cu
cudaError_t launch_metric_counts(const float* y_true, const float* y_pred, int B, int T, int Tp, int K,
                                 float threshold, int32_t* triples, unsigned long long* tpfpfn,
                                 unsigned long long* sums, cudaStream_t stream);
cudaError_t launch_er_finalize(const int32_t* triples, int B, float* er, cudaStream_t stream);

// k_ops.cu -- stand-alone stages (un-fused forms of the fused epilogue + label / metric helpers)
cudaError_t launch_axis_scale(const float* x, const float* m, float* out, size_t outer, size_t n_axis,
                              size_t inner, cudaStream_t st);
cudaError_t launch_axis_shift(const float* x, float* out, size_t outer, size_t n_axis, size_t inner,
                              int delta, cudaStream_t st);
cudaError_t launch_pointwise(int op, const float* x, float* out, size_t rows, int C, int width,
                             int n_log, float scalar, cudaStream_t st);
cudaError_t launch_chan_map(const float* x, float* out, size_t rows, int w_in, int w_out,
                            const int32_t* idx, const float* coef, size_t rows_per_sample,
                            cudaStream_t st);
cudaError_t launch_mel_project(const float* x, const float* W, const int32_t* lo, const int32_t* len,
                               float* out, int B, int F, int T, int C, int n_mel, cudaStream_t st);
cudaError_t launch_minmax(const float* x, float* out, uint32_t* mm, size_t S, size_t per_sample, int w,
                          int split, int variant, cudaStream_t st);
cudaError_t launch_sum_axis(const float* y, float* out, size_t outer, int V, size_t inner,
                            cudaStream_t st);
cudaError_t launch_avg_pool_time(const float* y, float* out, int B, int T, int K, int r, int out_len,
                                 int pad_left, int binarize, cudaStream_t st);
cudaError_t launch_cos_sim(const float* y_true, const float* y_pred, float* out, int B, int T, int K,
                           cudaStream_t st);

// data_utils.normalize (data_utils.py:32-34); acc: one double of scratch
cudaError_t launch_normalize(const float* x, float* out, size_t n, double* acc, cudaStream_t st);

cudaError_t launch_phase_vocoder(const float* x, float* out, int F, int T, int C, int T_out, const int32_t* i0,
                                 const int32_t* i1, const float* alpha, float adv_step, cudaStream_t st);
cudaError_t launch_sum_pool2(const float* y, float* out, int B, int T, int K, float scale, cudaStream_t st);
cudaError_t launch_density_labels(const float* y, float* out, size_t outer, int V, int TK, cudaStream_t st);

// k_resample.cu -- kaldi.resample_waveform (data_utils.py:20-21) of a list of items.  The device blob
// of a launch starts with its ResampleItem array; the filter tables follow.
struct ResampleItem {
    long long in_off, out_off;   // float offsets of the item's [n_chan, n_in] / [n_chan, n_out] blocks
    long long n_in, n_out;       // samples per channel
    long long table;             // byte offset in the blob of first[u_out] (int32), weights[u_out * W]; -1: copy
    long long cta0;              // first CTA of the item (it has ceil(n_out / chunk))
    int u_in, u_out, W, pad;
};
// smem_floats: the largest table of the launch that is staged in shared memory (0: none)
cudaError_t launch_resample(const float* wav, float* out, int n_chan, const char* d_blob, int n_items,
                            long long n_ctas, int chunk, int smem_floats, cudaStream_t st);

// k_istft.cu -- torch.istft of [B,257,T,2C] spectrograms into [B,C,L] (L >= 1); tw1: the ctx's warp FFT twiddles
cudaError_t launch_istft(const float* spec, float* out, int B, int T, int C, long long L, const float4* tw1,
                         cudaStream_t st);

// k_spec.cu -- spectrogram-format banks (the reference's pickled [257, t, 2C] lists)
cudaError_t launch_spec_activity(const float* specs, const int64_t* frame_off, int n_items, int F, int W,
                                 int max_frames, uint8_t* activity, cudaStream_t st);
cudaError_t launch_specmix(const FusedParams& p, int mode, const float* melW, const int32_t* mel_lo,
                           const int32_t* mel_len, cudaStream_t st, int out_type);   // out_type: OutType of p.out
size_t specmix_mel_smem(int C, int f_n);

// k_eval.cu -- evaluation-side chain of metrics.evaluate (metrics.py:59-87, 109-133, 176-214)
cudaError_t launch_eval_windows(const float* x, float* out, long long outer, long long T, long long inner,
                                int frame_len, int step, int n_win, cudaStream_t st);
cudaError_t launch_eval_merge(const float* preds, float* out, int n_win, int n_p, int K, int up, int step,
                              int L, cudaStream_t st);
cudaError_t launch_eval_smooth(const float* x, float* tmp, float* out, int L, int K, int k_avg, int k_max,
                               float thr, cudaStream_t st);
cudaError_t launch_eval_events(const float* y, int L, int K, int hop, int sr, int32_t* rows, int max_rows,
                               int32_t* n_rows, cudaStream_t st);
cudaError_t launch_get_er(const int32_t* gt, int m, const int32_t* pred, int pred_stride, int pred_time_col,
                          const int32_t* n_pred_ptr, int n_pred_max, int32_t* order_p, int32_t* order_g,
                          int32_t* out, cudaStream_t st);

}  // namespace iris
