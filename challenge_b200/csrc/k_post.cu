// Second pass of the log-mel features: per-clip min-max normalisation
// (data_utils.minmax, data_utils.py:37-47 with utils.safe_div, utils.py:114-116)
// followed by log(x + 1e-8) (data_utils.log_on_mel, data_utils.py:50-55), in place, right
// after k_fused (what is left of the batch in L2 is read from there: at 256 clips ~5 of the 102 MB, the
// rest comes back from HBM, measured in place).  The per-clip min/max were reduced
// by k_fused (atomicMax on (~bits(min), bits(max))); this kernel leaves that scratch zeroed
// for the next launch.
//   y = log((x - min) / max(max - min, 1e-8) + 1e-8)
// is evaluated as log2((x - min) * inv + 1e-8) * ln2 with inv = 1 / max(max - min, 1e-8):
// FADD, FFMA, MUFU.LG2, FMUL per element.
// With bfloat16 / float16 features (IRIS_OUT_BF16 / IRIS_OUT_F16) k_fused writes the fp32 mel into a
// context scratch and k_logmel_post<bf16 / f16> reads it from there and stores the converted result; the
// many-channel spectrogram-bank path also uses it as a conversion-only pass (neither min-max nor log).

#include "iris_common.cuh"
#include "iris_launch.h"

namespace iris {

constexpr int kPostThreads = 256;
constexpr int kPostChunks = 8;   // CTAs per clip

__device__ __forceinline__ float post_one(float x, float mn, float inv, float eps, int do_log) {
    x = fmaf(x - mn, inv, eps);   // x - mn first: exact near the clip minimum, where log amplifies
    return do_log ? __logf(x) : x;
}

// OutT = float with src == dst: in place.  Otherwise from the fp32 features at src (k_fused's scratch)
// into dst, with one rounding to OutT at the store.  src and dst may alias (no __restrict__): each
// element is loaded and stored by the same thread in the same iteration.  The minimum of 8 CTAs per SM holds
// every instance at 32 registers: left to itself ptxas gives the fp32 one 38 (its two pointers), 6 CTAs per SM,
// measured 1.4 % slower in place at configs[1] on B200 (profiles/r13_launch_templates.txt).
template <class OutT>
__global__ void __launch_bounds__(kPostThreads, 2048 / kPostThreads)
    k_logmel_post(const float* src, OutT* dst, uint32_t* __restrict__ minmax, size_t per_clip, int do_minmax,
                  int do_log, unsigned* done) {
    const int b = blockIdx.y;
    cudaGridDependencySynchronize();   // launched behind k_fused with programmatic stream serialization
    float inv = 1.f, mn = 0.f;
    const float eps = do_log ? 1e-8f : 0.f;
    if (do_minmax) {
        mn = __uint_as_float(~__ldcg(&minmax[2 * b]));
        const float mx = __uint_as_float(__ldcg(&minmax[2 * b + 1]));
        inv = 1.f / fmaxf(mx - mn, 1e-8f);
    }
    const float* base = src + size_t(b) * per_clip;
    OutT* out = dst + size_t(b) * per_clip;
    const size_t chunk = (per_clip + kPostChunks - 1) / kPostChunks;
    if ((per_clip & 3) == 0 && (chunk & 3) == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0 &&
        (reinterpret_cast<uintptr_t>(out) & (4 * sizeof(OutT) - 1)) == 0) {
        const float4* v = reinterpret_cast<const float4*>(base);
        const size_t lo = size_t(blockIdx.x) * (chunk >> 2);
        const size_t hi = min(lo + (chunk >> 2), per_clip >> 2);
        for (size_t i = lo + threadIdx.x; i < hi; i += 4 * kPostThreads) {
            float4 a[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i + u * kPostThreads < hi) a[u] = __ldcg(v + i + u * kPostThreads);
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i + u * kPostThreads < hi) {
                    a[u].x = post_one(a[u].x, mn, inv, eps, do_log);
                    a[u].y = post_one(a[u].y, mn, inv, eps, do_log);
                    a[u].z = post_one(a[u].z, mn, inv, eps, do_log);
                    a[u].w = post_one(a[u].w, mn, inv, eps, do_log);
                    store_out4(out + 4 * (i + u * kPostThreads), a[u]);
                }
        }
    } else {
        const size_t lo = size_t(blockIdx.x) * chunk, hi = min(lo + chunk, per_clip);
        for (size_t i = lo + threadIdx.x; i < hi; i += kPostThreads)
            store_out1(out + i, post_one(base[i], mn, inv, eps, do_log));
    }
    if (do_minmax) {   // the last chunk of the clip re-zeroes the scratch
        __syncthreads();
        if (threadIdx.x == 0) {
            if (atomicAdd(&done[b], 1u) == gridDim.x - 1) {
                minmax[2 * b] = 0u;
                minmax[2 * b + 1] = 0u;
                done[b] = 0u;
            }
        }
    }
}

cudaError_t launch_logmel_post(const float* src, void* dst, int out_type, uint32_t* minmax, unsigned* done, int B,
                               size_t per_clip, int do_minmax, int do_log, cudaStream_t stream) {
    const bool in_place = src == dst;
    if (B <= 0 || per_clip == 0 || (in_place && !do_minmax && !do_log)) return cudaSuccess;
    if (out_type != OUT_F32 && out_type != OUT_BF16 && out_type != OUT_F16) return cudaErrorInvalidValue;
    // in place, a half-width element i would land on float i / 2, which another thread may not have read yet
    if (in_place && out_type != OUT_F32) return cudaErrorInvalidValue;
    for (int b0 = 0; b0 < B; b0 += 65535) {
        int nb = B - b0 < 65535 ? B - b0 : 65535;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(kPostChunks, nb);
        cfg.blockDim = dim3(kPostThreads);
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        const float* s = src + size_t(b0) * per_clip;
        const size_t o = size_t(b0) * per_clip;
        uint32_t* mm = minmax ? minmax + 2 * size_t(b0) : static_cast<uint32_t*>(nullptr);
        unsigned* dn = done ? done + b0 : static_cast<unsigned*>(nullptr);
        cudaError_t e;
        if (out_type == OUT_BF16)
            e = cudaLaunchKernelEx(&cfg, k_logmel_post<__nv_bfloat16>, s, static_cast<__nv_bfloat16*>(dst) + o, mm,
                                   per_clip, do_minmax, do_log, dn);
        else if (out_type == OUT_F16)
            e = cudaLaunchKernelEx(&cfg, k_logmel_post<__half>, s, static_cast<__half*>(dst) + o, mm, per_clip,
                                   do_minmax, do_log, dn);
        else
            e = cudaLaunchKernelEx(&cfg, k_logmel_post<float>, s, static_cast<float*>(dst) + o, mm, per_clip,
                                   do_minmax, do_log, dn);
        if (e != cudaSuccess) return e;
    }
    return cudaGetLastError();
}

}  // namespace iris
