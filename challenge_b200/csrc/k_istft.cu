// Inverse STFT: torch.istft(n_fft=512, hop_length=256, window=hann_window(512) (periodic), center=True,
// normalized=False, onesided=True, length=L) of each channel of spectrograms in the layout of
// data_utils.load_wav, [B, 257, T, 2C] (real parts of the C channels, then their imaginary parts), written
// as [B, C, L] float32.
//
// Output sample s = 256 h + r (hop h, r < 256) is sample r + 256 of frame h plus sample r of frame h + 1,
// each times the window, over the window-square envelope w[r]^2 + w[r + 256]^2 (>= 0.5, static_assert
// below).  Past the last frame's centre (h = T - 1) only frame h covers s, and from s = 256 T on nothing
// does: zeros, as torch pads a longer `length`.
//
// A CTA owns kHops consecutive hops of one (item, channel pair) and computes the kHops + 1 frames they
// need, one per warp (the last frame is the halo the next tile computes again), so every output sample
// is summed by one thread in a fixed order: no atomics, bit-identical from run to run.
//  1. The CTA copies the bins of its frames into shared memory; 8 threads read 8 consecutive frames of
//     one bin row (128 contiguous bytes for 2 channels).
//  2. Each warp rebuilds z = X_a + i X_b over all 512 points from the Hermitian halves of the pair's two
//     channels (imaginary parts of bins 0 and 256 dropped, as a C2R transform drops them) and inverts it
//     with the forward warp FFT of fftwarp.cuh: IFFT(z) = conj(FFT(conj(z))) / 512, whose real part is
//     channel a and imaginary part channel b.  The 1 / 512 rides on the overlap-add weights.
//  3. After a CTA barrier each thread forms its samples of every hop from the two frames in shared
//     memory and stores them, consecutive threads on consecutive samples.
// Shared memory: one 4368-byte buffer per warp, holding in turn its frame's 257 bins, the FFT exchange
// rows and the 512 output samples.
#include "fftwarp.cuh"
#include "iris_common.cuh"
#include "iris_launch.h"

namespace iris {

constexpr int kIstftWarps = 8;
constexpr int kHops = kIstftWarps - 1;                // output hops per CTA
constexpr int kIstftBuf = kXwBytes + 16;             // 16 B past the exchange rows: the 8 warps' bin
                                                     // rows start 4 banks apart (conflict-free staging)
static_assert(kBins * 16 <= kIstftBuf && kNFft * 8 <= kIstftBuf, "per-warp buffer too small");

// overlap-add weights: lo[r] = w[r] / (512 env[r]) for sample r of frame h + 1, hi[r] = w[r + 256] /
// (512 env[r]) for sample r + 256 of frame h, tail[r] = 1 / (512 w[r + 256]) where frame h is alone
// (torch's (x w) / w^2), with env[r] = w[r]^2 + w[r + 256]^2 and w the periodic Hann window
struct OlaWeights {
    float lo[256], hi[256], tail[256];
};
constexpr double hann512(int n) { return 0.5 - 0.5 * cx_cos2pi(n, 512); }
constexpr OlaWeights make_ola_weights() {
    OlaWeights t{};
    for (int r = 0; r < 256; ++r) {
        const double wl = hann512(r), wh = hann512(r + 256), env = wl * wl + wh * wh;
        t.lo[r] = float(wl / (512.0 * env));
        t.hi[r] = float(wh / (512.0 * env));
        t.tail[r] = float(1.0 / (512.0 * wh));
    }
    return t;
}
constexpr double min_hann_envelope() {
    double m = 1.0;
    for (int r = 0; r < 256; ++r) {
        const double e = hann512(r) * hann512(r) + hann512(r + 256) * hann512(r + 256);
        m = e < m ? e : m;
    }
    return m;
}
// torch.istft rejects an envelope below 1e-11 (NOLA); at 50 % overlap the periodic Hann one is at least 1/2
static_assert(min_hann_envelope() >= 0.5 - 1e-12, "periodic Hann at hop 256 must satisfy NOLA");
// the tail divides by w[r + 256] >= w[511] = sin^2(pi / 512) > 0
static_assert(hann512(511) > 3e-5, "tail weights must stay finite");

__device__ const OlaWeights kOla = make_ola_weights();

// kC: 2 and 1 read the pair's cell as one float4 / float2 (a 2- or 1-channel spectrogram), 0 reads any C
template <int kC>
__global__ void __launch_bounds__(kIstftWarps * 32) k_istft(const float* __restrict__ spec, float* __restrict__ out,
                                                            int T, int C, long long L, int n_hops,
                                                            const float4* __restrict__ tw1) {
    __shared__ __align__(16) unsigned char sm[kIstftWarps * kIstftBuf];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int h0 = blockIdx.x * kHops, pair = blockIdx.y, b = blockIdx.z;
    const int ca = 2 * pair;
    const bool has_b = ca + 1 < C;
    // frame h0 + j is read by hop h0 + j and by hop h0 + j - 1
    auto needed = [&](int j) { return h0 + j < T && h0 + j <= n_hops; };

    // ---- 1. bins of frames h0 .. h0 + kHops: buffer j holds {re_a, re_b, im_a, im_b} of bin f at 16 f ----
    const float* item = spec + size_t(b) * kBins * T * 2 * C;
    for (int e = tid; e < kBins * kIstftWarps; e += kIstftWarps * 32) {
        const int f = e >> 3, j = e & 7;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (needed(j)) {
            const float* cell = item + (size_t(f) * T + h0 + j) * 2 * C;
            if (kC == 2) {
                v = __ldg(reinterpret_cast<const float4*>(cell));
            } else if (kC == 1) {
                const float2 x = __ldg(reinterpret_cast<const float2*>(cell));
                v = make_float4(x.x, 0.f, x.y, 0.f);
            } else {
                v.x = __ldg(cell + ca);
                v.z = __ldg(cell + C + ca);
                if (has_b) {
                    v.y = __ldg(cell + ca + 1);
                    v.w = __ldg(cell + C + ca + 1);
                }
            }
        }
        *reinterpret_cast<float4*>(sm + j * kIstftBuf + f * 16) = v;
    }
    __syncthreads();

    // ---- 2. one frame per warp ----
    unsigned char* buf = sm + warp * kIstftBuf;
    if (needed(warp)) {   // warp-uniform
        const float4* bins = reinterpret_cast<const float4*>(buf);
        // register i of the lane holds point k = lane + 32 i of conj(z)
        cpx v[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int k = lane + 32 * i;
            const bool mirror = k > 256;                    // z[k] = conj(X_a[512 - k]) + i conj(X_b[512 - k])
            float4 x = bins[mirror ? 512 - k : k];
            if (k == 0 || k == 256) { x.z = 0.f; x.w = 0.f; }
            v[i] = mirror ? cpx{x.x + x.w, x.z - x.y} : cpx{x.x - x.w, -(x.z + x.y)};
        }
        __syncwarp();   // every lane has its bins: the buffer becomes the exchange rows
        const int k1 = warp_k1(lane), par = warp_par(lane);
        {
            const float4 q0 = __ldg(tw1 + lane), q1 = __ldg(tw1 + 32 + lane), q2 = __ldg(tw1 + 64 + lane),
                         q4 = __ldg(tw1 + 128 + lane);
            warp_pass1(v, cpx{q0.z, q0.w}, cpx{q1.x, q1.y}, cpx{q2.x, q2.y}, cpx{q4.x, q4.y});
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) *reinterpret_cast<float2*>(buf + xw_write_off(k, lane)) = make_float2(v[k].x, v[k].y);
        __syncwarp();
        const unsigned char* row = buf + xw_read_off(k1, 0);
        const float sgn = par ? -1.f : 1.f;
        cpx u[16];
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const float4 a = *reinterpret_cast<const float4*>(row + 16 * m);
            const float4 c = *reinterpret_cast<const float4*>(row + 16 * (m + 8));
            constexpr_for_pair(m, [&](float c0, float s0, float c1, float s1) {
                u[2 * m] = warp_dif(cpx{a.x, a.y}, cpx{c.x, c.y}, sgn, par != 0, c0, s0);
                u[2 * m + 1] = warp_dif(cpx{a.z, a.w}, cpx{c.z, c.w}, sgn, par != 0, c1, s1);
            });
        }
        Fft<16>::run(u);
        __syncwarp();   // the exchange rows are read: the buffer becomes the frame
        // register jj holds FFT(conj z)[n] = 512 conj(x[n]) for n = k1 + 16 par + 32 jj: (x_a, x_b) * 512
        float2* frame = reinterpret_cast<float2*>(buf);
        const int n0 = k1 + 16 * par;
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) frame[n0 + 32 * jj] = make_float2(u[jj].x, -u[jj].y);
    }
    __syncthreads();

    // ---- 3. overlap-add: thread tid owns sample r = tid of every hop of the tile ----
    const int r = tid;
    const float wlo = kOla.lo[r], whi = kOla.hi[r], wtail = kOla.tail[r];
    float* oa = out + (size_t(b) * C + ca) * size_t(L);
    float* ob = oa + size_t(L);
    for (int q = 0; q < kHops; ++q) {
        const int h = h0 + q;
        const long long s = 256ll * h + r;
        if (h >= n_hops || s >= L) break;
        float2 y = make_float2(0.f, 0.f);
        if (h < T) {
            const float2 xh = reinterpret_cast<const float2*>(sm + q * kIstftBuf)[256 + r];
            if (h + 1 < T) {   // frame h, then frame h + 1
                const float2 xn = reinterpret_cast<const float2*>(sm + (q + 1) * kIstftBuf)[r];
                y = make_float2(fmaf(xh.x, whi, xn.x * wlo), fmaf(xh.y, whi, xn.y * wlo));
            } else {
                y = make_float2(xh.x * wtail, xh.y * wtail);
            }
        }
        oa[s] = y.x;
        if (has_b) ob[s] = y.y;
    }
}

cudaError_t launch_istft(const float* spec, float* out, int B, int T, int C, long long L, const float4* tw1,
                         cudaStream_t st) {
    const int n_hops = int((L + 255) / 256);
    dim3 grid(unsigned((n_hops + kHops - 1) / kHops), unsigned((C + 1) / 2), unsigned(B));
    const int threads = kIstftWarps * 32;
    if (C == 2) k_istft<2><<<grid, threads, 0, st>>>(spec, out, T, C, L, n_hops, tw1);
    else if (C == 1) k_istft<1><<<grid, threads, 0, st>>>(spec, out, T, C, L, n_hops, tw1);
    else k_istft<0><<<grid, threads, 0, st>>>(spec, out, T, C, L, n_hops, tw1);
    return cudaGetLastError();
}

}  // namespace iris
