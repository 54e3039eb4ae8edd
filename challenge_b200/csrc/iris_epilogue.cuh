// Per-bin epilogue shared by the fused waveform kernel (k_fused.cu) and the spectrogram-bank
// mix (k_spec.cu): masks, stft_filter, channel remaps, complex / mag-phase / log-mag-phase output.#pragma once
#include "iris_common.cuh"

namespace iris {

// Output channel c >= 2 of a channel remap of a 2-channel clip (data_utils.py:79-82, 100-117) from the
// real parts r0, r1 of the two input channels and the sum of their imaginary parts: stereo_mono
// X0 + X1; random_merge_aug (f re0 + sqrt(1 - f) re1, im0 + im1) with fa = f, sf = sqrt(1 - f) of the
// clip and channel.  Channels 0 and 1 are the inputs themselves.
__device__ __forceinline__ cpx remap_mix(int remap, float fa, float sf, float r0, float r1, float isum) {
    if (remap == REMAP_STEREO_MONO) return cpx{r0 + r1, isum};
    return cpx{fa * r0 + sf * r1, isum};
}
// (fa, sf) of output channel c >= 2 of clip b (random_merge_aug; unused by stereo_mono)
__device__ __forceinline__ float2 remap_coef(const FusedParams& p, int b, int c) {
    if (p.remap == REMAP_STEREO_MONO) return make_float2(1.f, 1.f);
    const size_t i = size_t(b) * (p.c_out - 2) + (c - 2);
    return make_float2(p.merge_f[i], p.merge_sf[i]);
}

// One (bin f, frame t, channel pair) of the output: (r0, i0) / (r1, i1) are the complex values of
// channels 2*pair and 2*pair + 1, m the product of the SpecAugment masks of this cell.  OutT: the
// element type of p.out (iris_common.cuh, store_out*).  kMono: the plan's remap is mono_chan, whose cells
// have a layout of their own (a run-time branch for it caps the spectrogram-mode k_specmix instances at 64
// registers, with spills).
template <int MODE, class OutT, bool kMono>
__device__ __forceinline__ void store_bin(const FusedParams& p, int b, int f, int t, int pair,
                                          bool has1, float r0, float i0, float r1, float i1,
                                          float m) {
    // masks are applied by multiplication (transforms.py:40) so zeros keep their sign
    r0 *= m; i0 *= m; r1 *= m; i1 *= m;
    const float filt = (f >= 1 && f <= p.filter_k) ? 0.f : 1.f;   // data_utils.py:126-136
    if constexpr (kMono) {
        // mono_chan (include/iris.h IRIS_REMAP_MONO_CHAN): the columns [re0 + re1, re0 + im0, re0 + im1] of
        // the masked inputs, then stft_filter (the reference's order and rounding: the complex spectrogram of
        // spectrogram banks is bit-identical); magnitude and phase of z_j = (re0 + re1) + i (re0 + im_j)
        float s = __fadd_rn(r0, r1), y0 = __fadd_rn(r0, i0), y1 = __fadd_rn(r0, i1);
        if (p.filter_k > 0) { s *= filt; y0 *= filt; y1 *= filt; }
        const size_t cell = (size_t(b) * kBins + f) * p.T + t;
        if (MODE == FM_COMPLEX) {
            OutT* o = reinterpret_cast<OutT*>(p.out) + cell * 3;
            store_out1(o, s);
            store_out1(o + 1, y0);
            store_out1(o + 2, y1);
        } else {
            float a0 = sqrt_approx(fmaf(s, s, y0 * y0));
            float a1 = sqrt_approx(fmaf(s, s, y1 * y1));
            if (MODE == FM_LOGMAGPHASE) {
                a0 = __logf(a0 + 1e-8f);
                a1 = __logf(a1 + 1e-8f);
            }
            store_out4(reinterpret_cast<OutT*>(p.out) + cell * 4, make_float4(a0, a1, fast_atan2f(y0, s), fast_atan2f(y1, s)));
        }
    } else if (p.remap == REMAP_NONE) {
        const int C = p.C;
        OutT* o = reinterpret_cast<OutT*>(p.out) + ((size_t(b) * kBins + f) * p.T + t) * size_t(2 * C);
        if (p.filter_k > 0) { r0 *= filt; i0 *= filt; r1 *= filt; i1 *= filt; }
        float a0 = r0, a1 = r1, b0 = i0, b1 = i1;   // first half / second half of the last dim
        if (MODE != FM_COMPLEX) {
            a0 = sqrt_approx(fmaf(r0, r0, i0 * i0));   // transforms.py:116
            b0 = fast_atan2f(i0, r0);                  // transforms.py:117
            a1 = sqrt_approx(fmaf(r1, r1, i1 * i1));
            b1 = fast_atan2f(i1, r1);
            if (MODE == FM_LOGMAGPHASE) {            // transforms.py:80-86
                a0 = __logf(a0 + 1e-8f);   // MUFU.LG2 * ln 2, as in the log-mel epilogue (|error| ~1e-6)
                a1 = __logf(a1 + 1e-8f);
            }
        }
        if (C == 2) {
            store_out4(o, make_float4(a0, a1, b0, b1));
        } else if (has1 && (C & 1) == 0) {
            store_out2(o + 2 * pair, a0, a1);
            store_out2(o + C + 2 * pair, b0, b1);
        } else {
            store_out1(o + 2 * pair, a0);
            store_out1(o + (C + 2 * pair), b0);
            if (has1) {
                store_out1(o + (2 * pair + 1), a1);
                store_out1(o + (C + 2 * pair + 1), b1);
            }
        }
    } else {
        // C == 2 input; c_out output channels (data_utils.py:79-82, 100-117)
        const int Co = p.c_out;
        OutT* o = reinterpret_cast<OutT*>(p.out) + ((size_t(b) * kBins + f) * p.T + t) * size_t(2 * Co);
        for (int c = 0; c < Co; ++c) {
            float re, im;
            if (c == 0) { re = r0; im = i0; }
            else if (c == 1) { re = r1; im = i1; }
            // (one branch per remap with the remap a constant: a single remap_mix(p.remap, remap_coef(..))
            // call moves the registers of the spectrogram-mode k_specmix instances and gives the half
            // ones a stack frame)
            else if (p.remap == REMAP_STEREO_MONO) {
                const cpx z = remap_mix(REMAP_STEREO_MONO, 1.f, 1.f, r0, r1, i0 + i1);
                re = z.x; im = z.y;
            } else {
                const float fa = p.merge_f[size_t(b) * (Co - 2) + (c - 2)];
                const float sf = p.merge_sf[size_t(b) * (Co - 2) + (c - 2)];
                const cpx z = remap_mix(REMAP_MERGE_AUG, fa, sf, r0, r1, i0 + i1);
                re = z.x; im = z.y;
            }
            if (p.filter_k > 0) { re *= filt; im *= filt; }
            float a = re, ph = im;
            if (MODE != FM_COMPLEX) {
                a = sqrt_approx(fmaf(re, re, im * im));
                ph = fast_atan2f(im, re);
                if (MODE == FM_LOGMAGPHASE) a = __logf(a + 1e-8f);
            }
            store_out1(o + c, a);
            store_out1(o + (Co + c), ph);
        }
    }
}

}  // namespace iris
