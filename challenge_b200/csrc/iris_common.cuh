// Shared device-side definitions for libiris (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "fftcore.cuh"

namespace iris {

constexpr int kNFft = 512;
constexpr int kHop = 256;
constexpr int kBins = 257;

// One mixing segment of one output clip: source frames k = t + shift of the padded,
// pair-interleaved waveform P (k_bank.cu; row h of a pair plane = P[256h .. 256h+256) as
// float2) contribute gain * frame_k to output frames t in [t_lo, t_hi).
struct Seg {
    const float* base;    // pair plane 0 of P
    int32_t pair_stride;  // floats between pair planes (= 2 * 256 * (kT + 1))
    int32_t shift;        // k = t + shift
    int32_t t_lo, t_hi;   // valid output frames
    float gain;
    int32_t keep_idx;     // index into keep[] (voice accept flags) or -1
};
static_assert(sizeof(Seg) == 32, "Seg layout");

enum FusedMode : int {
    FM_COMPLEX = 0,
    FM_MAGPHASE = 1,
    FM_LOGMAGPHASE = 2,
    FM_MEL = 3,
    FM_ACTIVITY = 4,
    FM_SE = 5,   // IRIS_FEAT_SE: x, only_voice, only_noise of the 'se' model (include/iris.h)
    FM_PLANE = 6,   // bank registration: bins 0..127 of every frame into the bank's STFT bin plane
};

enum ChanRemap : int { REMAP_NONE = 0, REMAP_STEREO_MONO = 1, REMAP_MERGE_AUG = 2, REMAP_MONO_CHAN = 3 };

// element type of the feature output (IRIS_OUT_BF16 / IRIS_OUT_F16 of include/iris.h)
enum OutType : int { OUT_F32 = 0, OUT_BF16 = 1, OUT_F16 = 2 };

// ---- feature stores: the one place that knows the output format ----
// All arithmetic is fp32; a half-width output converts at the store with round-to-nearest-even
// (bit for bit what torch's .to(bfloat16 / float16) does to the fp32 result, fp16 overflow -> +-inf).
// 1, 2 or 4 consecutive elements; 2 and 4 need 2- / 4-element alignment (8 / 16 bytes for float).
template <class T> __device__ __forceinline__ T out_cvt(float a);
template <> __device__ __forceinline__ float out_cvt<float>(float a) { return a; }
template <> __device__ __forceinline__ __nv_bfloat16 out_cvt<__nv_bfloat16>(float a) { return __float2bfloat16_rn(a); }
template <> __device__ __forceinline__ __half out_cvt<__half>(float a) { return __float2half_rn(a); }
// two values as one 32-bit word, a in the low half (the lower address)
template <class T> __device__ __forceinline__ uint32_t out_pack2(float a, float b);
template <> __device__ __forceinline__ uint32_t out_pack2<__nv_bfloat16>(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
template <> __device__ __forceinline__ uint32_t out_pack2<__half>(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
template <class T>
__device__ __forceinline__ void store_out1(T* o, float a) { *o = out_cvt<T>(a); }
template <class T>
__device__ __forceinline__ void store_out2(T* o, float a, float b) {
    if constexpr (sizeof(T) == 4) *reinterpret_cast<float2*>(o) = make_float2(a, b);
    else *reinterpret_cast<uint32_t*>(o) = out_pack2<T>(a, b);
}
template <class T>
__device__ __forceinline__ void store_out4(T* o, float4 v) {
    if constexpr (sizeof(T) == 4) *reinterpret_cast<float4*>(o) = v;
    else *reinterpret_cast<uint2*>(o) = make_uint2(out_pack2<T>(v.x, v.y), out_pack2<T>(v.z, v.w));
}

struct FusedParams {
    const Seg* segs;
    const int32_t* seg_ptr;  // [B+1]
    const uint8_t* keep;     // voice accept flags, may be null
    int32_t B, T, C;         // clips, frames per clip, input channels
    int32_t n_pairs;         // ceil(C/2): a tile is `fr` frames of one (clip, channel pair)
    int32_t fr;              // frames per tile = consumer warps per CTA
    int32_t c_out;           // output channels (C unless remapped; 2 pseudo-channels for mono_chan)
    // SpecAugment rectangles (size, offset) per clip; null => none
    const int32_t* tmask;
    int32_t n_tmask;
    const int32_t* fmask;
    int32_t n_fmask;
    int32_t filter_k;  // stft_filter: zero bins 1..k
    int32_t fm_bits;   // k_tiles writes the zeroed bins 0..127 of a tile as a bitmap instead of the
                       // (size, offset) list (mel epilogues that read bins below 128 only)
    int32_t remap;
    const float* merge_f;   // [B, c_out-2] factor
    const float* merge_sf;  // [B, c_out-2] sqrt(1-factor)
    // per-tile stage lists (k_tiles -> k_fused)
    unsigned char* tile_blocks;  // [n_tiles] blocks of tile_stride bytes
    int32_t tile_stride;
    int32_t max_segs;            // most mixing segments any clip has
    int32_t chunk;               // consecutive tiles per work claim
    int32_t n_big, n_mid;        // claim schedule (launch_fused): n_big claims of `chunk` tiles, n_mid of
    int32_t chunk_mid, chunk_tail;   // `chunk_mid`, the rest `chunk_tail`
    int32_t seg_select;          // 0: every segment; 1: voices only; 2: background + noises only
                                 // (only_voice / only_noise of pipeline.py:37-38, 82-83, 104-108);
                                 // 3 (FM_SE): channel pair q of a tile is bank pair 0 restricted as by q + 1
    uint32_t* sched;             // [2] next chunk, CTAs finished; zero between launches
    // outputs
    float* out;             // layout depends on mode
    int32_t stage_out;      // spectrogram modes: store through the shared-memory staging area
    int32_t pair_merge;     // stage_out with C == 4: the two channel pairs of a tile are stored together
    uint8_t* activity;      // FM_ACTIVITY: [B, T]
    // FM_MEL epilogue variants: log(x + 1e-8) and per-clip min-max before the log
    int32_t do_log, do_minmax;
    uint32_t* minmax;       // [B,2] atomicMax of (~bits(min), bits(max)); zeroed by k_tiles
    // mel projection: filters are handled in rounds of 32 (m = lane + 32 r); every filter of
    // round r reads mel_L[r] consecutive magnitudes starting at bin mel_f_lo + mel_info[m]
    // (shorter filters are zero-padded), weights at mel_w[(row0(r) + i) * 32 + lane]
    int32_t n_mel;
    int32_t mel_f_lo;       // lowest bin with a non-zero weight
    int32_t mel_f_n;        // number of bins in [f_lo, f_hi]
    int32_t mel_taps;       // sum of mel_L
    int32_t mel_L[4];
    const uint32_t* mel_info;  // [n_mel] first tap, relative to mel_f_lo
    const float* mel_w;        // [mel_taps][32]
    // 2-channel mel from the STFT bin planes of the banks (Bank::plane, k_fused EPI_PLANE): a stage whose
    // source row s lies in bank k's waveform [pl_wave[k], pl_wave[k] + pl_floats[k]) is read from the
    // plane row s + pl_delta[k], with the full gain (the plane holds X, not the packed two-channel FFT)
    int32_t plane;
    const float* pl_wave[3];
    int64_t pl_floats[3];
    int64_t pl_delta[3];    // FM_PLANE (the pass that builds a plane): pl_delta[0] is its own bank's
    // tables (fftwarp.cuh)
    const float4* tw1;      // [8][32] {W512^(n2*2q), W512^(n2*(2q+1))}
    const float4* ts;       // [8][2]  {t(2m), t(2m+1)}, t(i) = par ? W32^i : 1
    const float* hann;      // [512] periodic Hann
};

// ---- PTX helpers: mbarrier + bulk async copy (TMA 1-D) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// Blocking wait: try_wait with a suspend-time hint parks the warp in hardware until the phase
// completes (or ~10 ms pass), so a waiting warp issues next to nothing.  __nanosleep-based
// back-off measured ~15 ns per poll on B200 (170 wasted instructions per frame); this form is
// what CUTLASS' ClusterBarrier::wait uses.
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "IRIS_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra IRIS_DONE_%=;\n\t"
        "bra IRIS_WAIT_%=;\n\t"
        "IRIS_DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity), "r"(0x989680u)
        : "memory");
}
// arrive from the lanes where `pred` holds, as ONE predicated instruction (an `if` around
// mbar_arrive splits the warp until the next reconvergence point)
__device__ __forceinline__ void mbar_arrive_if(uint64_t* bar, bool pred) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %1, 0;\n\t"
        "@p mbarrier.arrive.shared::cta.b64 _, [%0];\n\t}" ::"r"(smem_u32(bar)),
        "r"(uint32_t(pred))
        : "memory");
}
// fire-and-forget atomic max (no return value: nothing to wait for)
__device__ __forceinline__ void red_max_u32_if(uint32_t* addr, uint32_t v, bool pred) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %2, 0;\n\t"
        "@p red.global.max.u32 [%0], %1;\n\t}" ::"l"(addr),
        "r"(v), "r"(uint32_t(pred))
        : "memory");
}
// L2 cache policies: the streamed bank rows are marked evict-first, the mel rows that the
// second pass (k_logmel_post) re-reads right after the kernel evict-last, so the 102 MB of
// features survive in the 126 MB L2 next to the input stream
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// global -> shared bulk copy under an L2 cache policy, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                              uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void st_f2_hint(float* addr, float a, float b, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(addr), "f"(a), "f"(b), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ float sqrt_approx(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// atan2 for the phase features (transforms.py:117): octant reduction + the degree-17 odd
// polynomial of Abramowitz & Stegun 4.4.49 (|error| <= 3.1e-7 rad over the plane, measured
// against float64), IEEE signed-zero / axis cases included: atan2(+-0, -x) = +-pi,
// atan2(+-0, +-0) = +-0 or +-pi by the sign bit of x.  ~22 instructions vs ~45 for atan2f.
__device__ __forceinline__ float fast_atan2f(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float hi = fmaxf(ax, ay), lo = fminf(ax, ay);
    const float a = hi > 0.f ? __fdividef(lo, hi) : 0.f;
    const float s = a * a;
    float r = 0.0028662257f;
    r = fmaf(r, s, -0.0161657367f);
    r = fmaf(r, s, 0.0429096138f);
    r = fmaf(r, s, -0.0752896400f);
    r = fmaf(r, s, 0.1065626393f);
    r = fmaf(r, s, -0.1420889944f);
    r = fmaf(r, s, 0.1999355085f);
    r = fmaf(r, s, -0.3333314528f);
    r = fmaf(r, s, 1.0f);
    r *= a;
    if (ay > ax) r = 1.57079632679489662f - r;
    if (__float_as_uint(x) >> 31) r = 3.14159265358979324f - r;
    return copysignf(r, y);
}
// Two atan2 for cells whose magnitude m = sqrt(x^2 + y^2) is already there (the mag/phase epilogue of
// k_fused): half-angle form.  With d = m + |x|, t = y / d lies in [-1, 1] for every (x, y), so the
// octant reduction (two abs, max, min, compare, two fix-ups per value) disappears:
//     atan2(y, x) = 2 atan(t)                      x >= +0
//                 = copysign(pi, y) - 2 atan(t)    x <= -0
// Same degree-17 polynomial (coefficients doubled: exact), |error| <= ~7e-7 rad.  Signed zeros as
// IEEE atan2: y = +-0 gives t = +-0, hence +-0 or +-pi by the sign bit of x; x = y = 0 has d clamped
// to a tiny positive number so that t stays +-0.  23 instructions for two values instead of 32.
__device__ __forceinline__ void fast_atan2f_mag_x2(float y0, float x0, float m0, float y1, float x1, float m1,
                                                   float& r0, float& r1) {
    // (|y| in the max keeps |t| <= 1 when m underflowed to 0 for denormal-range inputs; one FMNMX3)
    const float d0 = fmaxf(fmaxf(m0 + fabsf(x0), fabsf(y0)), 1e-30f), d1 = fmaxf(fmaxf(m1 + fabsf(x1), fabsf(y1)), 1e-30f);
    const cpx t{__fdividef(y0, d0), __fdividef(y1, d1)};
    const cpx s = cmul2(t, t);
    cpx r{2.f * 0.0028662257f, 2.f * 0.0028662257f};
    r = cfma2(r, s, cpx{2.f * -0.0161657367f, 2.f * -0.0161657367f});
    r = cfma2(r, s, cpx{2.f * 0.0429096138f, 2.f * 0.0429096138f});
    r = cfma2(r, s, cpx{2.f * -0.0752896400f, 2.f * -0.0752896400f});
    r = cfma2(r, s, cpx{2.f * 0.1065626393f, 2.f * 0.1065626393f});
    r = cfma2(r, s, cpx{2.f * -0.1420889944f, 2.f * -0.1420889944f});
    r = cfma2(r, s, cpx{2.f * 0.1999355085f, 2.f * 0.1999355085f});
    r = cfma2(r, s, cpx{2.f * -0.3333314528f, 2.f * -0.3333314528f});
    r = cfma2(r, s, cpx{2.f, 2.f});
    r = cmul2(r, t);
    r0 = (__float_as_uint(x0) >> 31) ? copysignf(3.14159265358979324f, y0) - r.x : r.x;
    r1 = (__float_as_uint(x1) >> 31) ? copysignf(3.14159265358979324f, y1) - r.y : r.y;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace iris
