// torchaudio.compliance.kaldi.resample_waveform (data_utils.py:20-21; Kaldi's LinearResample): a
// polyphase windowed-sinc FIR.  With U_in = orig / gcd and U_out = new / gcd,
//   out[c, u * U_out + i] = sum_j w[i][j] * wav[c, first[i] + u * U_in + j]      (zero outside)
// One launch resamples a list of items (one waveform for iris_resample, a whole bank for
// iris_bank_register_audio), each with the table of its own rate pair.  A CTA computes `chunk`
// consecutive outputs of one item, every channel, so the U_out x W weight table it stages in shared
// memory (when it fits) is loaded once per chunk * n_chan outputs; items whose table does not fit read
// it through the cache.  One thread per output sample and channel at a time: consecutive threads read
// overlapping, nearly contiguous input windows (L1 / L2 hits).  Items already at the target rate
// (table < 0) are copied.
#include "iris_common.cuh"
#include "iris_launch.h"

namespace iris {

__global__ void __launch_bounds__(256) k_resample(const float* __restrict__ wav, float* __restrict__ out,
                                                  int n_chan, const char* __restrict__ blob, int n_items,
                                                  int chunk, int smem_floats) {
    extern __shared__ float s_w[];
    const ResampleItem* items = reinterpret_cast<const ResampleItem*>(blob);
    int lo = 0, hi = n_items - 1;          // the item of this CTA: the last one with cta0 <= blockIdx.x
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (items[mid].cta0 <= (long long)blockIdx.x) lo = mid;
        else hi = mid - 1;
    }
    const ResampleItem it = items[lo];
    const long long n0 = ((long long)blockIdx.x - it.cta0) * chunk;
    const long long n1 = n0 + chunk < it.n_out ? n0 + chunk : it.n_out;
    const float* x = wav + it.in_off;
    float* y = out + it.out_off;
    if (it.table < 0) {
        for (int c = 0; c < n_chan; ++c)
            for (long long n = n0 + threadIdx.x; n < n1; n += blockDim.x)
                y[size_t(c) * it.n_out + n] = x[size_t(c) * it.n_in + n];
        return;
    }
    const int32_t* first = reinterpret_cast<const int32_t*>(blob + it.table);
    const float* wt = reinterpret_cast<const float*>(first + it.u_out);
    const int W = it.W;
    if (it.u_out * W <= smem_floats) {
        for (int i = threadIdx.x; i < it.u_out * W; i += blockDim.x) s_w[i] = wt[i];
        __syncthreads();
        wt = s_w;
    }
    for (long long n = n0 + threadIdx.x; n < n1; n += blockDim.x) {
        const long long u = n / it.u_out;
        const int i = int(n - u * it.u_out);
        const long long k0 = (long long)first[i] + u * it.u_in;
        const float* w = wt + size_t(i) * W;
        for (int c = 0; c < n_chan; ++c) {
            const float* xc = x + size_t(c) * it.n_in;
            float acc = 0.f;
            for (int j = 0; j < W; ++j) {
                const long long k = k0 + j;
                if (k >= 0 && k < it.n_in) acc = fmaf(w[j], xc[k], acc);
            }
            y[size_t(c) * it.n_out + n] = acc;
        }
    }
}

cudaError_t launch_resample(const float* wav, float* out, int n_chan, const char* d_blob, int n_items,
                            long long n_ctas, int chunk, int smem_floats, cudaStream_t st) {
    if (n_ctas <= 0) return cudaSuccess;
    const size_t smem = size_t(smem_floats) * sizeof(float);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_resample, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess) return e;
    }
    k_resample<<<unsigned(n_ctas), 256, smem, st>>>(wav, out, n_chan, d_blob, n_items, chunk, smem_floats);
    return cudaGetLastError();
}

}  // namespace iris
