// Spectrogram-bank path: the reference's own data format (utils.load_data, utils.py:88-94 --
// a pickled list of pre-computed complex spectrograms [257, t, 2C]; pipeline.py:113-175 mixes
// those).  Banks registered in this format are mixed in the SPECTROGRAM domain, exactly the
// arithmetic of pipeline.merge_complex_specs (pipeline.py:29-106):
//     out[f, t, :] = bg[f, t + o_b, :] + sum_v (g_v * voice_v[f, t + s_v, :]) * keep_v
//                                      + sum_n  g_n * noise_n[f, t + s_n, :]
// with the products and sums rounded separately in the reference's order (no FMA contraction),
// so the complex output is bit-identical to the CPU restatement.  The per-cell epilogue
// (masks, remap, stft_filter, mag / phase / log) is the one of the fused waveform kernel
// (iris_epilogue.cuh).  Pure streaming: every source cell is read once, every output cell
// written once; a warp covers 32 consecutive frames of one bin row (512 contiguous bytes per
// source for 2 channels).
#include "iris_common.cuh"
#include "iris_epilogue.cuh"
#include "iris_launch.h"

namespace iris {

// frame "active" iff any coefficient of the frame (any bin, re or im, any channel) is > 0
// (pipeline.py:55).  One thread per frame; consecutive threads read consecutive cells of a
// bin row.  items [n_items] spectrograms [F, t_i, W] packed back to back.
__global__ void k_spec_activity(const float* __restrict__ specs, const int64_t* __restrict__ frame_off,
                                int n_items, int F, int W, int max_frames, uint8_t* __restrict__ activity) {
    const int item = blockIdx.y;
    const int64_t f0 = frame_off[item];
    const int tI = int(frame_off[item + 1] - f0);
    const float* base = specs + size_t(f0) * F * W;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < tI; t += gridDim.x * blockDim.x) {
        float mx = 0.f;
        for (int f = 0; f < F; ++f) {
            const float* cell = base + (size_t(f) * tI + t) * W;
            for (int w = 0; w < W; ++w) mx = fmaxf(mx, cell[w]);
        }
        activity[size_t(item) * max_frames + t] = mx > 0.f ? 1 : 0;
    }
}

// Seg of a spectrogram bank: base = the item's [F, tI, 2C] array, pair_stride = tI.
//
// A CTA owns 32 consecutive frames of one clip (lane = frame) and walks all 257 bin rows, 8
// warps taking every 8th row: a warp's load of one source row is 32 cells = 512 contiguous
// bytes (2 channels).  The clip's segments that are kept and overlap the tile are compacted,
// in the reference's order, into shared memory once per CTA.
//   spectrogram modes: the cell goes through store_bin (masks, remap, filter, mag / phase).
//   FM_SE: the 'se' batch (include/iris.h, IRIS_FEAT_SE): besides the mix, the kept voices and background +
//   noises are summed into their own accumulators (the products and sums of the mix, so the three blocks are
//   bit-identical to three selected launches); real parts of bins 1..256, masks and filter on x only.
//   FM_MEL: |.| of the masked, filtered cell (every output channel of a remap) is parked in shared
//   memory [257][32][c_out]; after the walk the CTA projects its 32 frames on the mel filters (dense matrix, non-zero rows
//   [lo, lo + len) per filter; transforms.py:51-77), stores [n_mel][32 frames] rows of 128 /
//   256 contiguous bytes and reduces the per-clip extrema for the min-max pass (k_post.cu).
constexpr int kSpecTile = 32;      // frames per CTA
constexpr int kSpecWarps = 8;
constexpr int kSpecMaxSegs = 48;   // staged segments per tile; more fall back to the global list

// kMono: the spectrogram modes of a mono_chan plan (store_bin<.., true>).  Their minimum of 2 CTAs per SM keeps
// ptxas from its own choice of 64 registers with spills for the COMPLEX instance (0 = no minimum, as before).
template <int MODE, class OutT, bool kMono = false>
__global__ void __launch_bounds__(kSpecWarps * 32, kMono ? 2 : 0) k_specmix(const __grid_constant__ FusedParams p,
                                                            const float* __restrict__ melW,
                                                            const int32_t* __restrict__ mel_lo,
                                                            const int32_t* __restrict__ mel_len) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    __shared__ Seg s_segs[kSpecMaxSegs];
    __shared__ int s_n, s_overflow;
    const int b = blockIdx.y;
    const int t0 = blockIdx.x * kSpecTile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = t0 + lane;
    const bool live = t < p.T;
    const int C = p.C, W = 2 * C;
    const int Cm = p.c_out;   // FM_MEL: channels of the magnitudes (C, or c_out of a channel remap)
    const int g0 = p.seg_ptr[b], g1 = p.seg_ptr[b + 1];

    if (warp == 0) {   // ordered compaction of the segments this tile needs
        int n = 0;
        bool over = false;
        for (int base = g0; base < g1; base += 32) {
            const int s = base + lane;
            Seg sg;
            bool use = false;
            if (s < g1) {
                sg = p.segs[s];
                use = sg.t_lo < t0 + kSpecTile && sg.t_hi > t0 &&
                      !(sg.keep_idx >= 0 && p.keep[sg.keep_idx] == 0) &&
                      !((p.seg_select == 1 && sg.keep_idx < 0) || (p.seg_select == 2 && sg.keep_idx >= 0));
            }
            const unsigned bal = __ballot_sync(0xffffffffu, use);
            const int pos = n + __popc(bal & ((1u << lane) - 1u));
            if (use) {
                if (pos < kSpecMaxSegs) s_segs[pos] = sg;
                else over = true;
            }
            n += __popc(bal);
        }
        over = __any_sync(0xffffffffu, over);
        if (lane == 0) { s_n = n; s_overflow = over ? 1 : 0; }
    }
    __syncthreads();
    const bool staged = s_overflow == 0;
    const int n_seg = staged ? s_n : g1 - g0;

    // SpecAugment time mask of this frame (transforms.py:12-40)
    float mt = 1.f;
    if (p.tmask != nullptr && live) {
        const int32_t* tm = p.tmask + size_t(b) * p.n_tmask * 2;
        for (int i = 0; i < p.n_tmask; ++i)
            if (unsigned(t - tm[2 * i + 1]) < unsigned(tm[2 * i])) mt = 0.f;
    }
    // FM_MEL: only the bin rows that carry a non-zero mel weight are read at all
    // ([mel_f_lo, mel_f_lo + mel_f_n): bins 4..122 of 257 for the TF default matrix)
    float* mags = reinterpret_cast<float*>(sm_raw);   // [mel_f_n][32][Cm]
    const int f_begin = MODE == FM_MEL ? p.mel_f_lo : (MODE == FM_SE ? 1 : 0);
    const int f_end = MODE == FM_MEL ? p.mel_f_lo + p.mel_f_n : kBins;

    // U bin rows per warp iteration: their loads are issued together (the walk is latency-bound
    // otherwise: one 512-byte row per warp and segment in flight)
    constexpr int U = 4;
    for (int fb = f_begin + warp; fb < f_end; fb += kSpecWarps * U) {
        float m[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int f = fb + u * kSpecWarps;
            m[u] = mt;
            if (p.fmask != nullptr) {
                const int32_t* fm = p.fmask + size_t(b) * p.n_fmask * 2;
                for (int i = 0; i < p.n_fmask; ++i)
                    if (unsigned(f - fm[2 * i + 1]) < unsigned(fm[2 * i])) m[u] = 0.f;
            }
        }
        for (int pair = 0; pair < p.n_pairs; ++pair) {
            const bool has1 = 2 * pair + 1 < C;
            float r0[U], r1[U], i0[U], i1[U];
            float vr[U], nr[U];   // FM_SE: Re ch0 of the kept voices / of background + noises
#pragma unroll
            for (int u = 0; u < U; ++u) { r0[u] = 0.f; r1[u] = 0.f; i0[u] = 0.f; i1[u] = 0.f; vr[u] = 0.f; nr[u] = 0.f; }
            bool first = true, v_first = true, n_first = true;
            if (live) {
                for (int s = 0; s < n_seg; ++s) {
                    Seg sg;
                    if (staged) sg = s_segs[s];
                    else {
                        sg = p.segs[g0 + s];
                        if (sg.keep_idx >= 0 && p.keep[sg.keep_idx] == 0) continue;
                        if ((p.seg_select == 1 && sg.keep_idx < 0) || (p.seg_select == 2 && sg.keep_idx >= 0)) continue;
                    }
                    if (t < sg.t_lo || t >= sg.t_hi) continue;
                    const size_t row = size_t(sg.pair_stride) * W;
                    const float* cell0 = sg.base + size_t(fb) * row + size_t(t + sg.shift) * W;
                    float x0[U], x1[U], y0[U], y1[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        x0[u] = 0.f; x1[u] = 0.f; y0[u] = 0.f; y1[u] = 0.f;
                        if (fb + u * kSpecWarps < f_end) {
                            const float* cell = cell0 + size_t(u * kSpecWarps) * row;
                            if (C == 2) {
                                const float4 v = __ldg(reinterpret_cast<const float4*>(cell));
                                x0[u] = v.x; x1[u] = v.y; y0[u] = v.z; y1[u] = v.w;
                            } else {
                                x0[u] = __ldg(cell + 2 * pair);
                                y0[u] = __ldg(cell + C + 2 * pair);
                                if (has1) {
                                    x1[u] = __ldg(cell + 2 * pair + 1);
                                    y1[u] = __ldg(cell + C + 2 * pair + 1);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        if (first) {   // the background enters with gain 1 (pipeline.py:35)
                            r0[u] = __fmul_rn(sg.gain, x0[u]); r1[u] = __fmul_rn(sg.gain, x1[u]);
                            i0[u] = __fmul_rn(sg.gain, y0[u]); i1[u] = __fmul_rn(sg.gain, y1[u]);
                        } else {       // spec += gain * source (pipeline.py:81, 106): product, then sum
                            r0[u] = __fadd_rn(r0[u], __fmul_rn(sg.gain, x0[u]));
                            r1[u] = __fadd_rn(r1[u], __fmul_rn(sg.gain, x1[u]));
                            i0[u] = __fadd_rn(i0[u], __fmul_rn(sg.gain, y0[u]));
                            i1[u] = __fadd_rn(i1[u], __fmul_rn(sg.gain, y1[u]));
                        }
                    }
                    first = false;
                    if (MODE == FM_SE) {   // the same products, summed per subset in the same order
                        const bool voice = sg.keep_idx >= 0;
                        const bool sf = voice ? v_first : n_first;
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            const float g = __fmul_rn(sg.gain, x0[u]);
                            if (voice) vr[u] = sf ? g : __fadd_rn(vr[u], g);
                            else nr[u] = sf ? g : __fadd_rn(nr[u], g);
                        }
                        if (voice) v_first = false;
                        else n_first = false;
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int f = fb + u * kSpecWarps;
                if (f >= f_end) continue;
                if (MODE == FM_MEL) {
                    const float filt = (f >= 1 && f <= p.filter_k) ? 0.f : 1.f;   // data_utils.py:126-136
                    const float mm = m[u] * filt;
                    const float a0 = r0[u] * mm, b0 = i0[u] * mm, a1 = r1[u] * mm, b1 = i1[u] * mm;
                    float* o = mags + (size_t(f - f_begin) * kSpecTile + lane) * Cm + 2 * pair;
                    if (p.remap == REMAP_MONO_CHAN) {
                        // z_j = (re0 + re1) + i (re0 + im_j) (include/iris.h): the sums of the masked,
                        // filtered inputs (a bin the filter zeroes has |z_j| = 0 either way)
                        const float s = __fadd_rn(a0, a1), y0 = __fadd_rn(a0, b0), y1 = __fadd_rn(a0, b1);
                        o[0] = sqrt_approx(fmaf(s, s, y0 * y0));
                        o[1] = sqrt_approx(fmaf(s, s, y1 * y1));
                        continue;
                    }
                    o[0] = sqrt_approx(fmaf(a0, a0, b0 * b0));   // transforms.py:116
                    if (has1) o[1] = sqrt_approx(fmaf(a1, a1, b1 * b1));
                    // channel remap (C == 2, one pair): the other output channels from the masked, filtered
                    // inputs (zeros before the remap are zeros after it; the filter follows it in the
                    // reference).  Without a remap Cm == C and every channel is an input channel.
                    if (p.remap != REMAP_NONE) {
                        for (int c = 2; c < Cm; ++c) {
                            const float2 k = remap_coef(p, b, c);
                            const cpx z = remap_mix(p.remap, k.x, k.y, a0, a1, b0 + b1);
                            o[c] = sqrt_approx(fmaf(z.x, z.x, z.y * z.y));
                        }
                    }
                } else if (MODE == FM_SE) {
                    if (live) {
                        // x as store_bin forms it: masks, then the filter, by multiplication
                        float a0 = r0[u] * m[u], a1 = r1[u] * m[u];
                        if (f <= p.filter_k) { a0 *= 0.f; a1 *= 0.f; }   // data_utils.py:126-136 (f >= 1)
                        const size_t cells = size_t(p.B) * 256 * p.T;
                        const size_t c = (size_t(b) * 256 + (f - 1)) * p.T + t;
                        float* o = reinterpret_cast<float*>(p.out);
                        *reinterpret_cast<float2*>(o + 2 * c) = make_float2(a0, a1);
                        o[2 * cells + c] = vr[u];
                        o[3 * cells + c] = nr[u];
                    }
                } else if (live) {
                    store_bin<MODE, OutT, kMono>(p, b, f, t, pair, has1, r0[u], i0[u], r1[u], i1[u], m[u]);
                }
            }
        }
    }
    if (MODE != FM_MEL) return;
    __syncthreads();
    // mel[b, mi, t, c] = sum_f |X[b, f, t, c]| * W[f, mi]; lane = frame, warps take every 8th filter
    float mn = __int_as_float(0x7f800000), mx = 0.f;
    const bool lg = p.do_log && !p.do_minmax;
    for (int mi = warp; mi < p.n_mel; mi += kSpecWarps) {
        const int f0 = mel_lo[mi] - f_begin, f1 = f0 + mel_len[mi];
        for (int c = 0; c < Cm; ++c) {
            float acc = 0.f;
            for (int f = f0; f < f1; ++f)
                acc = fmaf(mags[(size_t(f) * kSpecTile + lane) * Cm + c], __ldg(melW + size_t(f + f_begin) * p.n_mel + mi), acc);
            if (live) {
                mn = fminf(mn, acc);
                mx = fmaxf(mx, acc);
                store_out1(reinterpret_cast<OutT*>(p.out) + ((size_t(b) * p.n_mel + mi) * p.T + t) * Cm + c,
                           lg ? __logf(acc + 1e-8f) : acc);
            }
        }
    }
    if (p.do_minmax) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        const bool go = lane == 0 && mn <= mx;
        red_max_u32_if(&p.minmax[2 * b], ~__float_as_uint(mn), go);
        red_max_u32_if(&p.minmax[2 * b + 1], __float_as_uint(mx), go);
    }
}

cudaError_t launch_spec_activity(const float* specs, const int64_t* frame_off, int n_items, int F, int W,
                                 int max_frames, uint8_t* activity, cudaStream_t st) {
    if (n_items <= 0 || max_frames <= 0) return cudaSuccess;
    dim3 grid(unsigned((max_frames + 127) / 128), unsigned(n_items));
    k_spec_activity<<<grid, 128, 0, st>>>(specs, frame_off, n_items, F, W, max_frames, activity);
    return cudaGetLastError();
}

size_t specmix_mel_smem(int C, int f_n) { return size_t(f_n) * kSpecTile * C * 4; }

// one k_specmix instance; FM_MEL: its dynamic shared memory attribute is set once per instance
template <int MODE, class OutT, bool kMono = false>
static cudaError_t launch_specmix_instance(const FusedParams& p, const float* melW, const int32_t* mel_lo,
                                           const int32_t* mel_len, cudaStream_t st) {
    size_t smem = 0;
    if constexpr (MODE == FM_MEL) {
        smem = specmix_mel_smem(p.c_out, p.mel_f_n);
        if (smem > 200 * 1024) return cudaErrorInvalidValue;
        static bool attr_set = false;
        if (!attr_set) {
            cudaError_t e = cudaFuncSetAttribute(k_specmix<MODE, OutT, kMono>,
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            if (e != cudaSuccess) return e;
            attr_set = true;
        }
    }
    const dim3 grid(unsigned((p.T + kSpecTile - 1) / kSpecTile), unsigned(p.B));
    k_specmix<MODE, OutT, kMono><<<grid, kSpecWarps * 32, smem, st>>>(p, melW, mel_lo, mel_len);
    return cudaGetLastError();
}

template <class OutT>
static cudaError_t launch_specmix_t(const FusedParams& p, int mode, const float* melW, const int32_t* mel_lo,
                                    const int32_t* mel_len, cudaStream_t st) {
    const bool mono = p.remap == REMAP_MONO_CHAN;   // the spectrogram modes of mono_chan: instances of their own
    if (mono && (p.C != 2 || p.c_out != 2)) return cudaErrorInvalidValue;
    switch (mode) {
        case FM_COMPLEX:
            return mono ? launch_specmix_instance<FM_COMPLEX, OutT, true>(p, nullptr, nullptr, nullptr, st)
                        : launch_specmix_instance<FM_COMPLEX, OutT>(p, nullptr, nullptr, nullptr, st);
        case FM_MAGPHASE:
            return mono ? launch_specmix_instance<FM_MAGPHASE, OutT, true>(p, nullptr, nullptr, nullptr, st)
                        : launch_specmix_instance<FM_MAGPHASE, OutT>(p, nullptr, nullptr, nullptr, st);
        case FM_LOGMAGPHASE:
            return mono ? launch_specmix_instance<FM_LOGMAGPHASE, OutT, true>(p, nullptr, nullptr, nullptr, st)
                        : launch_specmix_instance<FM_LOGMAGPHASE, OutT>(p, nullptr, nullptr, nullptr, st);
        case FM_MEL:
            if (p.remap != REMAP_NONE && !mono && (p.C != 2 || p.c_out < 3)) return cudaErrorInvalidValue;
            return launch_specmix_instance<FM_MEL, OutT>(p, melW, mel_lo, mel_len, st);
        default: return cudaErrorInvalidValue;
    }
}

// mode FM_MEL: p.out [B, n_mel, T, c_out], p.do_log / p.do_minmax / p.minmax as in the fused kernel;
// melW dense [257, n_mel] with the non-zero rows [lo, lo + len) of every filter.  out_type: OutType
// of p.out (the min-max mel features are fp32: k_logmel_post normalises them).
cudaError_t launch_specmix(const FusedParams& p, int mode, const float* melW, const int32_t* mel_lo,
                           const int32_t* mel_len, cudaStream_t st, int out_type) {
    if (p.B <= 0 || p.T <= 0) return cudaSuccess;
    if (p.B > 65535) return cudaErrorInvalidValue;
    if (out_type != OUT_F32 && p.do_minmax) return cudaErrorInvalidValue;
    if (mode == FM_SE) {   // fp32, 2 channels, no remap; every segment kept (the subsets are split per cell)
        if (out_type != OUT_F32 || p.C != 2 || p.remap != REMAP_NONE || p.seg_select != 0) return cudaErrorInvalidValue;
        return launch_specmix_instance<FM_SE, float>(p, nullptr, nullptr, nullptr, st);
    }
    switch (out_type) {
        case OUT_F32: return launch_specmix_t<float>(p, mode, melW, mel_lo, mel_len, st);
        case OUT_BF16: return launch_specmix_t<__nv_bfloat16>(p, mode, melW, mel_lo, mel_len, st);
        case OUT_F16: return launch_specmix_t<__half>(p, mode, melW, mel_lo, mel_len, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace iris
