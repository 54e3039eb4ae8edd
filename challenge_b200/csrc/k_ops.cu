// Stand-alone stages of transforms.py / data_utils.py / metrics.py for callers that apply the
// reference's functions one at a time (the fused kernel in k_fused.cu is the hot path; these
// are the same stages un-fused, so that every public function of the drop-in modules runs on
// the GPU).  All of them stream fp32 tensors once: grid-stride loops, coalesced along the
// innermost axis, grids capped at a multiple of the SM count by the launchers.
#include "iris_common.cuh"
#include "iris_launch.h"

namespace iris {

namespace {
constexpr int kOpThreads = 256;
inline unsigned op_grid(size_t n, int per_thread = 1) {
    size_t blocks = (n + size_t(kOpThreads) * per_thread - 1) / (size_t(kOpThreads) * per_thread);
    const size_t cap = 148 * 16;
    return unsigned(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}
}  // namespace

// out[o, a, i] = x[o, a, i] * m[a]     transforms.mask (transforms.py:12-40, the product at :40),
// data_utils.stft_filter (data_utils.py:126-136); m is the 0/1 vector both build by concat.
__global__ void __launch_bounds__(kOpThreads) k_axis_scale(const float* __restrict__ x,
                                                           const float* __restrict__ m,
                                                           float* __restrict__ out, size_t total,
                                                           size_t n_axis, size_t inner) {
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < total;
         i += size_t(gridDim.x) * kOpThreads) {
        const size_t a = (i / inner) % n_axis;
        out[i] = x[i] * m[a];
    }
}

// transforms.random_shift (transforms.py:43-47): zero-pad `width` both sides along the axis,
// crop n_axis cells at `offset`  =>  out[o, a, i] = x[o, a + offset - width, i] or 0
__global__ void __launch_bounds__(kOpThreads) k_axis_shift(const float* __restrict__ x,
                                                           float* __restrict__ out, size_t total,
                                                           size_t n_axis, size_t inner, int delta) {
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < total;
         i += size_t(gridDim.x) * kOpThreads) {
        const long long a = (long long)((i / inner) % n_axis) + delta;
        out[i] = (a >= 0 && a < (long long)n_axis) ? x[i + (long long)delta * (long long)inner] : 0.f;
    }
}

// rows of [2C]: first C = real / magnitude, last C = imag / phase
//   OP 0: complex_to_magphase (transforms.py:111-123); an odd input width (3, C = 2) is mono_chan's
//         [real, imag0, imag1], the real column broadcast, into rows of 2C = 4
//   OP 1: magphase_to_complex (transforms.py:126-134)
//   OP 2: log_magphase        (transforms.py:80-86): log(x + 1e-8) on the first n_log columns
//   OP 3: log_on_mel          (data_utils.py:50-55):  log(x + 1e-8) everywhere
//   OP 4: multiply_label      (data_utils.py:120-123): x * scalar
template <int OP>
__global__ void __launch_bounds__(kOpThreads) k_pointwise(const float* __restrict__ x,
                                                          float* __restrict__ out, size_t rows,
                                                          int C, int width, int n_log, float scalar) {
    if (OP == 0 || OP == 1) {
        const size_t n = rows * size_t(C);
        for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < n;
             i += size_t(gridDim.x) * kOpThreads) {
            const size_t r = i / C, c = i - r * C;
            const float a = x[r * width + ((width & 1) ? 0 : c)], b = x[r * width + (width - C) + c];
            float u, v;
            if (OP == 0) {
                u = sqrtf(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)));   // sqrt(real**2 + img**2)
                v = atan2f(b, a);
            } else {
                u = a * cosf(b);
                v = a * sinf(b);
            }
            out[r * 2 * C + c] = u;
            out[r * 2 * C + C + c] = v;
        }
    } else {
        const size_t n = rows * size_t(width);
        for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < n;
             i += size_t(gridDim.x) * kOpThreads) {
            const float v = x[i];
            float o;
            if (OP == 2) o = (int(i % width) < n_log) ? logf(v + 1e-8f) : v;
            else if (OP == 3) o = logf(v + 1e-8f);
            else o = v * scalar;
            out[i] = o;
        }
    }
}

// Channel remaps of data_utils.py as out[r, j] = c0[j] * x[r, i0[j]] (+ c1[j] * x[r, i1[j]]):
// mono_chan (73-76), stereo_mono (79-82), random_merge_aug (100-117).  coef is per sample
// (`rows_per_sample` rows share one coefficient set); products and the sum are rounded
// separately, like the reference's mul / mul / add.
__global__ void __launch_bounds__(kOpThreads) k_chan_map(const float* __restrict__ x,
                                                         float* __restrict__ out, size_t rows,
                                                         int w_in, int w_out,
                                                         const int32_t* __restrict__ idx,   // [w_out,2]
                                                         const float* __restrict__ coef,    // [S,w_out,2]
                                                         size_t rows_per_sample) {
    const size_t n = rows * size_t(w_out);
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < n;
         i += size_t(gridDim.x) * kOpThreads) {
        const size_t r = i / w_out;
        const int j = int(i - r * w_out);
        const float* cf = coef + ((r / rows_per_sample) * w_out + j) * 2;
        const int i0 = idx[2 * j], i1 = idx[2 * j + 1];
        float v = __fmul_rn(cf[0], x[r * w_in + i0]);
        if (i1 >= 0) v = __fadd_rn(v, __fmul_rn(cf[1], x[r * w_in + i1]));
        out[i] = v;
    }
}

// transforms.magphase_to_mel (transforms.py:51-77): mel[b, m, t, c] = sum_f mag[b, f, t, c] *
// W[f, m] over the non-zero rows [lo[m], lo[m] + len[m]) of column m (W dense [F, n_mel]);
// x is [B, F, T, 2C] (magnitude = first C of the last axis), out [B, n_mel, T, C].
__global__ void __launch_bounds__(kOpThreads) k_mel_project(const float* __restrict__ x,
                                                            const float* __restrict__ W,
                                                            const int32_t* __restrict__ lo,
                                                            const int32_t* __restrict__ len,
                                                            float* __restrict__ out, int B, int F,
                                                            int T, int C, int n_mel) {
    const size_t TC = size_t(T) * C;
    const size_t n = size_t(B) * n_mel * TC;
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < n;
         i += size_t(gridDim.x) * kOpThreads) {
        const size_t tc = i % TC;
        const int m = int((i / TC) % n_mel);
        const size_t b = i / (TC * n_mel);
        const size_t t = tc / C, c = tc - t * C;
        const float* xp = x + ((b * F) * T + t) * size_t(2 * C) + c;
        float acc = 0.f;
        const int f0 = lo[m], f1 = f0 + len[m];
        for (int f = f0; f < f1; ++f)
            acc = fmaf(xp[size_t(f) * T * 2 * C], W[size_t(f) * n_mel + m], acc);
        out[i] = acc;
    }
}

// Per-sample extrema of group g of the last axis (width `w`, groups split at `split`):
// data_utils.minmax (data_utils.py:37-47; one group) and transforms.minmax_norm_magphase
// (transforms.py:89-107; magnitude half and phase half).  mm[s, g] = (min, max) as ordered
// uint32 keys reduced with atomicMin / atomicMax; mm is pre-filled with (0xffffffff, 0).
__device__ __forceinline__ uint32_t f2key(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
__global__ void __launch_bounds__(kOpThreads) k_minmax_reduce(const float* __restrict__ x,
                                                              uint32_t* __restrict__ mm,
                                                              size_t per_sample, int w, int split) {
    const size_t s = blockIdx.y;
    const float* xs = x + s * per_sample;
    uint32_t lo[2] = {0xffffffffu, 0xffffffffu}, hi[2] = {0u, 0u};
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < per_sample;
         i += size_t(gridDim.x) * kOpThreads) {
        const int g = int(i % w) >= split ? 1 : 0;
        const uint32_t k = f2key(xs[i]);
        lo[g] = min(lo[g], k);
        hi[g] = max(hi[g], k);
    }
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        for (int o = 16; o > 0; o >>= 1) {
            lo[g] = min(lo[g], __shfl_xor_sync(0xffffffffu, lo[g], o));
            hi[g] = max(hi[g], __shfl_xor_sync(0xffffffffu, hi[g], o));
        }
        if ((threadIdx.x & 31) == 0 && lo[g] <= hi[g]) {
            atomicMin(&mm[(s * 2 + g) * 2], lo[g]);
            atomicMax(&mm[(s * 2 + g) * 2 + 1], hi[g]);
        }
    }
}
// variant 0: safe_div(x - min, max - min) = (x - min) / max(max - min, 1e-8)   (utils.py:114-116)
// variant 1: (x - min) / (max - min + 1e-8)                                    (transforms.py:102-103)
__global__ void __launch_bounds__(kOpThreads) k_minmax_apply(const float* __restrict__ x,
                                                             const uint32_t* __restrict__ mm,
                                                             float* __restrict__ out,
                                                             size_t per_sample, int w, int split,
                                                             int variant) {
    const size_t s = blockIdx.y;
    float mn[2], den[2];
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        mn[g] = key2f(mm[(s * 2 + g) * 2]);
        const float d = key2f(mm[(s * 2 + g) * 2 + 1]) - mn[g];
        den[g] = variant == 0 ? fmaxf(d, 1e-8f) : d + 1e-8f;
    }
    const float* xs = x + s * per_sample;
    float* os = out + s * per_sample;
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < per_sample;
         i += size_t(gridDim.x) * kOpThreads) {
        const int g = int(i % w) >= split ? 1 : 0;
        os[i] = __fdiv_rn(xs[i] - mn[g], den[g]);
    }
}

// data_utils.to_frame_labels (data_utils.py:64-70): out[o, i] = sum_v y[o, v, i], v ascending
__global__ void __launch_bounds__(kOpThreads) k_sum_axis(const float* __restrict__ y,
                                                         float* __restrict__ out, size_t outer,
                                                         int V, size_t inner) {
    const size_t n = outer * inner;
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < n;
         i += size_t(gridDim.x) * kOpThreads) {
        const size_t o = i / inner, k = i - o * inner;
        float acc = 0.f;
        for (int v = 0; v < V; ++v) acc += y[(o * V + v) * inner + k];
        out[i] = acc;
    }
}

// Keras AveragePooling1D(r, r, 'same') over time on [B, T, K]: window i covers
// [i*r - pad_left, i*r - pad_left + r) clipped to [0, T), averaged over the valid cells.
//   binarize != 0: data_utils.label_downsample (data_utils.py:85-97): out = (avg >= 0.5)
//   binarize == 0: the smoothing of metrics.er_score (metrics.py:222-224): out = avg
__global__ void __launch_bounds__(kOpThreads) k_avg_pool_time(const float* __restrict__ y,
                                                              float* __restrict__ out, int B, int T,
                                                              int K, int r, int out_len,
                                                              int pad_left, int binarize) {
    const size_t n = size_t(B) * out_len * K;
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < n;
         i += size_t(gridDim.x) * kOpThreads) {
        const int k = int(i % K);
        const int w = int((i / K) % out_len);
        const size_t b = i / (size_t(K) * out_len);
        const int lo = max(w * r - pad_left, 0), hi = min(w * r - pad_left + r, T);
        float acc = 0.f;
        for (int t = lo; t < hi; ++t) acc += y[(b * T + t) * K + k];
        const float avg = __fdiv_rn(acc, float(hi - lo));
        out[i] = binarize ? (avg >= 0.5f ? 1.f : 0.f) : avg;
    }
}

// metrics.cos_sim (metrics.py:277-287): per sample, the negative cosine similarity along time
// of every class (keras: l2-normalise with rsqrt(max(sum sq, 1e-12))), averaged over the
// classes that occur in y_true.  One warp per sample.
__global__ void __launch_bounds__(kOpThreads) k_cos_sim(const float* __restrict__ y_true,
                                                        const float* __restrict__ y_pred,
                                                        float* __restrict__ out, int B, int T, int K) {
    const int warp = (blockIdx.x * kOpThreads + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= B) return;
    const float* a = y_true + size_t(warp) * T * K;
    const float* p = y_pred + size_t(warp) * T * K;
    float res = 0.f, n_cls = 0.f;
    float cs_k[8];
    float occ[8];
    for (int k = 0; k < K && k < 8; ++k) {
        float saa = 0.f, spp = 0.f, sap = 0.f, sa = 0.f;
        for (int t = lane; t < T; t += 32) {
            const float u = a[size_t(t) * K + k], v = p[size_t(t) * K + k];
            saa = fmaf(u, u, saa);
            spp = fmaf(v, v, spp);
            sap = fmaf(u, v, sap);
            sa += u;
        }
        for (int o = 16; o > 0; o >>= 1) {
            saa += __shfl_xor_sync(0xffffffffu, saa, o);
            spp += __shfl_xor_sync(0xffffffffu, spp, o);
            sap += __shfl_xor_sync(0xffffffffu, sap, o);
            sa += __shfl_xor_sync(0xffffffffu, sa, o);
        }
        cs_k[k] = -sap * rsqrtf(fmaxf(saa, 1e-12f)) * rsqrtf(fmaxf(spp, 1e-12f));
        occ[k] = sa > 0.f ? 1.f : 0.f;
        n_cls += occ[k];
    }
    const float den = fmaxf(n_cls, 1e-8f);   // safe_div (utils.py:114-116)
    for (int k = 0; k < K && k < 8; ++k) res += cs_k[k] * (occ[k] / den);
    if (lane == 0) out[warp] = res;
}

// ---- launchers ----
// trainer.preprocess_labels (trainer.py:86-94), one of its five stages:
// avg_pool1d(y, 2, strides=2, 'SAME') * 2 on [B, T, K] -> [B, ceil(T/2), K].  SAME pads on the
// right only (total pad <= 1) and TF averages over the valid cells, so a full pair gives
// (a + b) / 2 * 2 = a + b (the halving and doubling are exact) and a lone last cell a / 1 * 2.
// `scale` multiplies the result (the final `y *= multiplier`, 1 for the inner stages).
__global__ void __launch_bounds__(kOpThreads) k_sum_pool2(const float* __restrict__ y, float* __restrict__ out,
                                                          int B, int T, int K, float scale) {
    const int out_len = (T + 1) / 2;
    const size_t n = size_t(B) * out_len * K;
    for (size_t i = blockIdx.x * size_t(kOpThreads) + threadIdx.x; i < n;
         i += size_t(gridDim.x) * kOpThreads) {
        const int k = int(i % K);
        const int w = int((i / K) % out_len);
        const size_t b = i / (size_t(K) * out_len);
        const float a = y[(b * T + 2 * w) * K + k];
        float v;
        if (2 * w + 1 < T) v = __fmul_rn(__fmul_rn(__fadd_rn(a, y[(b * T + 2 * w + 1) * K + k]), 0.5f), 2.f);
        else v = __fmul_rn(a, 2.f);
        out[i] = scale == 1.f ? v : __fmul_rn(v, scale);
    }
}

// trainer.to_density_labels (trainer.py:97-104): y [outer, V, T, K] -> [outer, T, K]:
// every voice divided by max(its total over (T, K), 1e-8), then summed over the voices in
// ascending order.  One CTA per `outer`; the totals are reduced in a fixed tree (labels are
// 0/1, so any order gives the same integer).
__global__ void __launch_bounds__(256) k_density_labels(const float* __restrict__ y, float* __restrict__ out,
                                                        int V, int TK) {
    __shared__ float red[256];
    __shared__ float den[64];
    const float* yo = y + size_t(blockIdx.x) * V * TK;
    for (int v = 0; v < V; ++v) {
        float s = 0.f;
        for (int i = threadIdx.x; i < TK; i += 256) s += yo[size_t(v) * TK + i];
        red[threadIdx.x] = s;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) den[v] = fmaxf(red[0], 1e-8f);
        __syncthreads();
    }
    for (int i = threadIdx.x; i < TK; i += 256) {
        float acc = 0.f;
        for (int v = 0; v < V; ++v) acc = __fadd_rn(acc, __fdiv_rn(yo[size_t(v) * TK + i], den[v]));
        out[size_t(blockIdx.x) * TK + i] = acc;
    }
}

// transforms.phase_vocoder (transforms.py:137-195): time-stretch of a complex spectrogram
// x [F, T, 2C] -> out [F, T_out, 2C].  Output step j interpolates the magnitudes of frames
// i0[j], i1[j] (a zero frame past the end) with weight alpha[j] and advances the phase by the
// wrapped phase difference of the two frames; the phase is a running sum over the steps
// (tf.cumsum), so one thread walks one (bin, channel) row.  i0 / i1 / alpha are the host's
// tf.range(0, T, rate) arithmetic.
__global__ void __launch_bounds__(128) k_phase_vocoder(const float* __restrict__ x, float* __restrict__ out,
                                                       int F, int T, int C, int T_out,
                                                       const int32_t* __restrict__ i0,
                                                       const int32_t* __restrict__ i1,
                                                       const float* __restrict__ alpha, float adv_step) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= F * C) return;
    const int f = row / C, c = row - f * C;
    const float* xf = x + size_t(f) * T * 2 * C;
    float* of = out + size_t(f) * T_out * 2 * C;
    const float adv = __fmul_rn(adv_step, float(f));          // tf.linspace: start + step * i
    const float two_pi = 6.28318530717958647692f;
    auto re_at = [&](int t) { return t < T ? xf[size_t(t) * 2 * C + c] : 0.f; };
    auto im_at = [&](int t) { return t < T ? xf[size_t(t) * 2 * C + C + c] : 0.f; };
    float acc = 0.f;
    float next = atan2f(im_at(0), re_at(0));                   // phase_0: angle of the first frame
    for (int j = 0; j < T_out; ++j) {
        acc = __fadd_rn(acc, next);                            // cumsum([phase_0, phase[:-1]])
        const int a = i0[j], b = i1[j];
        const float r0 = re_at(a), m0 = im_at(a), r1 = re_at(b), m1 = im_at(b);
        const float n0 = sqrtf(__fadd_rn(__fmul_rn(r0, r0), __fmul_rn(m0, m0)));
        const float n1 = sqrtf(__fadd_rn(__fmul_rn(r1, r1), __fmul_rn(m1, m1)));
        float ph = __fadd_rn(__fadd_rn(atan2f(m1, r1), -atan2f(m0, r0)), -adv);
        ph = __fadd_rn(ph, -__fmul_rn(two_pi, rintf(__fdiv_rn(ph, two_pi))));
        next = __fadd_rn(ph, adv);
        const float al = alpha[j];
        const float mag = __fadd_rn(__fmul_rn(al, n1), __fmul_rn(__fadd_rn(1.f, -al), n0));
        float sn, cs;
        sincosf(acc, &sn, &cs);
        of[size_t(j) * 2 * C + c] = __fmul_rn(mag, cs);
        of[size_t(j) * 2 * C + C + c] = __fmul_rn(mag, sn);
    }
}

cudaError_t launch_axis_scale(const float* x, const float* m, float* out, size_t outer, size_t n_axis,
                              size_t inner, cudaStream_t st) {
    const size_t total = outer * n_axis * inner;
    if (total == 0) return cudaSuccess;
    k_axis_scale<<<op_grid(total, 4), kOpThreads, 0, st>>>(x, m, out, total, n_axis, inner);
    return cudaGetLastError();
}
cudaError_t launch_axis_shift(const float* x, float* out, size_t outer, size_t n_axis, size_t inner,
                              int delta, cudaStream_t st) {
    const size_t total = outer * n_axis * inner;
    if (total == 0) return cudaSuccess;
    k_axis_shift<<<op_grid(total, 4), kOpThreads, 0, st>>>(x, out, total, n_axis, inner, delta);
    return cudaGetLastError();
}
cudaError_t launch_pointwise(int op, const float* x, float* out, size_t rows, int C, int width,
                             int n_log, float scalar, cudaStream_t st) {
    if (rows == 0 || width == 0) return cudaSuccess;
    const unsigned g = op_grid(rows * size_t(width), 4);
    switch (op) {
        case 0: k_pointwise<0><<<g, kOpThreads, 0, st>>>(x, out, rows, C, width, n_log, scalar); break;
        case 1: k_pointwise<1><<<g, kOpThreads, 0, st>>>(x, out, rows, C, width, n_log, scalar); break;
        case 2: k_pointwise<2><<<g, kOpThreads, 0, st>>>(x, out, rows, C, width, n_log, scalar); break;
        case 3: k_pointwise<3><<<g, kOpThreads, 0, st>>>(x, out, rows, C, width, n_log, scalar); break;
        case 4: k_pointwise<4><<<g, kOpThreads, 0, st>>>(x, out, rows, C, width, n_log, scalar); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
cudaError_t launch_chan_map(const float* x, float* out, size_t rows, int w_in, int w_out,
                            const int32_t* idx, const float* coef, size_t rows_per_sample,
                            cudaStream_t st) {
    if (rows == 0) return cudaSuccess;
    k_chan_map<<<op_grid(rows * size_t(w_out), 4), kOpThreads, 0, st>>>(x, out, rows, w_in, w_out, idx,
                                                                        coef, rows_per_sample);
    return cudaGetLastError();
}
cudaError_t launch_mel_project(const float* x, const float* W, const int32_t* lo, const int32_t* len,
                               float* out, int B, int F, int T, int C, int n_mel, cudaStream_t st) {
    const size_t n = size_t(B) * n_mel * T * C;
    if (n == 0) return cudaSuccess;
    k_mel_project<<<op_grid(n, 2), kOpThreads, 0, st>>>(x, W, lo, len, out, B, F, T, C, n_mel);
    return cudaGetLastError();
}
cudaError_t launch_minmax(const float* x, float* out, uint32_t* mm, size_t S, size_t per_sample, int w,
                          int split, int variant, cudaStream_t st) {
    if (S == 0 || per_sample == 0) return cudaSuccess;
    for (size_t s0 = 0; s0 < S; s0 += 32768) {
        const size_t ns = S - s0 < 32768 ? S - s0 : 32768;
        unsigned gx = unsigned((per_sample + kOpThreads * 8 - 1) / (kOpThreads * 8));
        gx = gx < 1 ? 1 : (gx > 64 ? 64 : gx);
        dim3 grid(gx, unsigned(ns));
        k_minmax_reduce<<<grid, kOpThreads, 0, st>>>(x + s0 * per_sample, mm + s0 * 4, per_sample, w, split);
        k_minmax_apply<<<grid, kOpThreads, 0, st>>>(x + s0 * per_sample, mm + s0 * 4,
                                                    out + s0 * per_sample, per_sample, w, split, variant);
    }
    return cudaGetLastError();
}
cudaError_t launch_sum_axis(const float* y, float* out, size_t outer, int V, size_t inner,
                            cudaStream_t st) {
    if (outer * inner == 0) return cudaSuccess;
    k_sum_axis<<<op_grid(outer * inner), kOpThreads, 0, st>>>(y, out, outer, V, inner);
    return cudaGetLastError();
}
cudaError_t launch_avg_pool_time(const float* y, float* out, int B, int T, int K, int r, int out_len,
                                 int pad_left, int binarize, cudaStream_t st) {
    const size_t n = size_t(B) * out_len * K;
    if (n == 0) return cudaSuccess;
    k_avg_pool_time<<<op_grid(n), kOpThreads, 0, st>>>(y, out, B, T, K, r, out_len, pad_left, binarize);
    return cudaGetLastError();
}
cudaError_t launch_cos_sim(const float* y_true, const float* y_pred, float* out, int B, int T, int K,
                           cudaStream_t st) {
    if (B <= 0) return cudaSuccess;
    if (K > 8) return cudaErrorInvalidValue;
    k_cos_sim<<<(B * 32 + kOpThreads - 1) / kOpThreads, kOpThreads, 0, st>>>(y_true, y_pred, out, B, T, K);
    return cudaGetLastError();
}

cudaError_t launch_phase_vocoder(const float* x, float* out, int F, int T, int C, int T_out, const int32_t* i0,
                                 const int32_t* i1, const float* alpha, float adv_step, cudaStream_t st) {
    if (F * C == 0 || T_out == 0) return cudaSuccess;
    k_phase_vocoder<<<(F * C + 127) / 128, 128, 0, st>>>(x, out, F, T, C, T_out, i0, i1, alpha, adv_step);
    return cudaGetLastError();
}
cudaError_t launch_sum_pool2(const float* y, float* out, int B, int T, int K, float scale, cudaStream_t st) {
    const size_t n = size_t(B) * ((T + 1) / 2) * K;
    if (n == 0) return cudaSuccess;
    k_sum_pool2<<<op_grid(n), kOpThreads, 0, st>>>(y, out, B, T, K, scale);
    return cudaGetLastError();
}
cudaError_t launch_density_labels(const float* y, float* out, size_t outer, int V, int TK, cudaStream_t st) {
    if (outer == 0 || TK == 0) return cudaSuccess;
    if (V > 64 || outer > 0x7fffffff) return cudaErrorInvalidValue;
    k_density_labels<<<unsigned(outer), 256, 0, st>>>(y, out, V, TK);
    return cudaGetLastError();
}

// ---- data_utils.normalize (data_utils.py:32-34): x / (10 * sqrt(mean(x^2))) over the whole clip ----
// Same arithmetic as the bank registration (k_bank.cu): squares summed in fp64, mean and
// sqrt(.) * 10 in fp32 like torch, then a division per sample.
__global__ void __launch_bounds__(256) k_sumsq(const float* __restrict__ x, size_t n, double* __restrict__ acc) {
    double a = 0.0;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const float v = x[i];
        a += double(v) * double(v);
    }
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    __shared__ double part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += part[w];
        atomicAdd(acc, t);
    }
}
__global__ void __launch_bounds__(256) k_rms_scale(const float* __restrict__ x, float* __restrict__ out, size_t n,
                                                   double* __restrict__ acc) {
    const float rms = sqrtf(float(*acc / double(n))) * 10.f;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x)
        out[i] = x[i] / rms;
}
cudaError_t launch_normalize(const float* x, float* out, size_t n, double* acc, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(acc, 0, sizeof(double), st);
    if (e != cudaSuccess) return e;
    const unsigned grid = unsigned(n / 1024 < 1 ? 1 : (n / 1024 > 592 ? 592 : n / 1024));
    k_sumsq<<<grid, 256, 0, st>>>(x, n, acc);
    k_rms_scale<<<grid, 256, 0, st>>>(x, out, n, acc);
    return cudaGetLastError();
}

}  // namespace iris
