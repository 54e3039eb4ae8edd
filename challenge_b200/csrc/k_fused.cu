// Fused hot path: gather + time-domain mix of the gained source frames, window,
// 512-point FFT per frame (two real channels packed into one complex transform, ONE WARP per
// frame, 16 points per lane), then the epilogue (SpecAugment masks, channel remap,
// stft_filter, complex / mag-phase / log-mag-phase output, or magnitude -> sparse mel ->
// per-clip min-max), writing each feature once.
//
// Replaces, for one output clip, the chain
//   data_utils.load_wav (STFT, data_utils.py:9-29)  ->  pipeline.merge_complex_specs
//   (pipeline.py:6-110)  ->  data_utils.augment (58-61)  ->  stereo_mono /
//   random_merge_aug / stft_filter (79-136)  ->  transforms.complex_to_magphase
//   (transforms.py:111-123)  ->  magphase_to_mel (51-77)  ->  data_utils.minmax (37-47)
//   ->  data_utils.log_on_mel (50-55)
// using linearity of the STFT: sum_k g_k STFT(src_k)[frame] = FFT(w * sum_k g_k frame_k).
//
// Structure.  A tile is FR consecutive output frames of one (clip, channel pair); a CTA has
// FR consumer warps (warp j owns frame j of the tile) and one producer warp.
//  * For every tile a TileBlock lists the mixing segments that are kept and overlap it (stage
//    descriptors + the tile's mask bits; iris_tiles.cuh).  The blocks are written by the label
//    kernel (k_labels, which decides the keep flags) or, without a label pass in front, by k_tiles.
//  * Tiles are claimed in chunks of consecutive tiles that shrink towards the end of the launch
//    (fused_schedule): the first claim of a CTA is its block index, the later ones come from a global
//    counter.  The producer warp copies the TileBlock of each tile into a shared-memory descriptor
//    ring and fetches every stage -- (j_cnt + 1) contiguous 2 KB rows of the pair-interleaved bank, or
//    j_cnt rows of the bank's STFT bin plane for the 2-channel mel launches that read it (EPI_PLANE) --
//    with ONE cp.async.bulk (TMA 1-D) into a ring of 3 (mel) or 2 (spectrogram modes) stage buffers:
//    full[slot] completes when the bytes have landed, empty[slot] when all FR consumer warps have
//    read the slot.
//  * Consumer warps never synchronise with each other: each waits on full[slot], accumulates
//    gain * frame into its 16 complex registers per lane, releases the slot, and after the
//    last stage runs the warp FFT (fftwarp.cuh: 16-point FFT in registers, twiddle, one
//    exchange through its private 4.25 KB of shared memory, radix-2 DIF + 16-point FFT) and
//    the epilogue.  Rows shared by adjacent frames are read from the same slot, so every
//    source row enters the SM once per tile.
//  * LOGMEL_MINMAX: the warps of a CTA combine the extrema of a run of tiles of one clip in shared
//    memory and the last one sends them to global atomics; k_logmel_post (k_post.cu) normalises and
//    logs the batch right after (in place, or from an fp32 scratch into bfloat16 / float16 features).
#include <cstdlib>
#include <cstring>

#include "fftwarp.cuh"
#include "iris_common.cuh"
#include "iris_epilogue.cuh"
#include "iris_launch.h"
#include "iris_tiles.cuh"

namespace iris {

constexpr int kRing = 8;         // TileBlock ring entries (> stage buffers + 1, see the producer)
constexpr int kMaxFR = 16;       // consumer warps per CTA (sets the register budget)
constexpr int kMaxRegs = 96;     // no spills; 2 CTAs x 9 warps (FR = 8) or 17 warps (FR = 16) per SM fit the register file
constexpr int kMaxMel = 128;
constexpr int kMaxTaps = 64;     // sum over the 32-filter rounds of the longest filter
constexpr int kMaxFilter = 16;   // taps of the longest mel filter the fused epilogue takes

// ---- shared memory map (bytes) ----
constexpr int OFF_FULL = 0;                                  // uint64 full[<= 3]
constexpr int OFF_EMPTY = 32;                                // uint64 empty[<= 3]
constexpr int OFF_RING = 64;
constexpr int OFF_TW1 = OFF_RING + kRing * kTileBlockBytes;  // float4 [2][32]: {w, w^2}, {w^4, w^8}, w = W512^lane
constexpr int OFF_MSTART = OFF_TW1 + 2 * 32 * 16;            // uint32 [kMaxMel]
constexpr int OFF_MW = OFF_MSTART + kMaxMel * 4;             // float [mel_taps][32]
static_assert(OFF_TW1 % 16 == 0 && OFF_MW % 16 == 0, "table alignment");

// float [256]: first half of the periodic Hann window (w[n + 256] = 1 - w[n])
__host__ __device__ inline uint32_t off_hann(int mel_taps) {
    return (uint32_t(OFF_MW) + uint32_t(mel_taps) * 128u + 127u) & ~127u;
}
__host__ __device__ inline uint32_t off_xch(int mel_taps) { return off_hann(mel_taps) + 1024u; }
__host__ __device__ inline uint32_t off_slots(int mel_taps, int fr) {
    return off_xch(mel_taps) + uint32_t(fr) * uint32_t(kXwBytes);   // kXwBytes % 128 == 0
}
__host__ __device__ inline uint32_t slot_bytes(int fr) { return uint32_t(fr + 1) * 2048u; }
// stage buffers per CTA: the modes that write whole spectrograms trade one stage buffer for
// the store staging area below
constexpr int kMelSlots = 3;
__host__ __device__ constexpr int slots_of(int mode) {
    return (mode == FM_MEL || mode == FM_ACTIVITY || mode == FM_PLANE) ? kMelSlots : 2;
}
// staging of a tile's [257 bins][FR frames] x 16 B output pieces (16-byte columns XOR-swizzled
// by the bin so that both the per-frame writes and the per-bin reads are conflict-free)
__host__ __device__ inline uint32_t stage_bytes(int fr) { return uint32_t(kBins) * uint32_t(fr) * 16u; }
__host__ __device__ inline uint32_t smem_total(int mel_taps, int fr, int mode, bool staged) {
    return off_slots(mel_taps, fr) + slots_of(mode) * slot_bytes(fr) + (staged ? stage_bytes(fr) : 0u);
}
// spectrogram modes without a channel remap (16 B per (bin, frame, pair)) store through the
// staging area; 8 frames per tile give 128-byte rows
__host__ __device__ inline bool stages_output(int mode, int remap, int fr) {
    return mode != FM_MEL && mode != FM_ACTIVITY && mode != FM_PLANE && remap == REMAP_NONE && fr == 8;
}

// ---- pre-kernel: one thread per tile builds its TileBlock (launches without a k_labels pass in
// front, or whose tile layout differs from the one k_labels was asked to build) ----
__global__ void __launch_bounds__(128) k_tiles(const FusedParams p) {
    const int tile = blockIdx.x * blockDim.x + threadIdx.x;
    // programmatic dependent launch: k_fused may start its prologue (barriers, zero fill of the stage
    // buffers) now; it waits for this grid before it touches a tile block
    cudaTriggerProgrammaticLaunchCompletion();
    const int per_clip = ((p.T + p.fr - 1) / p.fr) * p.n_pairs;
    if (tile >= p.B * per_clip) return;
    if (tile < p.B && p.minmax != nullptr) {   // per-clip extrema scratch of the launch that follows
        p.minmax[2 * tile] = 0u;
        p.minmax[2 * tile + 1] = 0u;
    }
    if (p.seg_select == 3) build_tile_block<true>(p, tile, per_clip);
    else build_tile_block(p, tile, per_clip);
}

// one (bin, frame, channel pair) of the spectrogram modes without a channel remap:
// {first-half ch0, ch1, second-half ch0, ch1} = (re, re, im, im) or (|.|, |.|, phase, phase)
template <int MODE>
__device__ __forceinline__ float4 make_piece(const FusedParams& p, int f, float r0, float i0, float r1,
                                             float i1, float m) {
    // masks are applied by multiplication (transforms.py:40) so zeros keep their sign
    r0 *= m; i0 *= m; r1 *= m; i1 *= m;
    if (p.filter_k > 0) {                                          // data_utils.py:126-136
        const float filt = (f >= 1 && f <= p.filter_k) ? 0.f : 1.f;
        r0 *= filt; i0 *= filt; r1 *= filt; i1 *= filt;
    }
    float a0 = r0, a1 = r1, b0 = i0, b1 = i1;
    // (a short cut for masked cells -- |.| = +0, atan2(+-0, +-0) from the sign bits -- was measured on
    // B200: 4-ch MAGPHASE 678.7 -> 685.0 us; the branch costs more than the polynomial it skips)
    if (MODE != FM_COMPLEX) {
        a0 = sqrt_approx(fmaf(r0, r0, i0 * i0));   // transforms.py:116
        a1 = sqrt_approx(fmaf(r1, r1, i1 * i1));
        fast_atan2f_mag_x2(i0, r0, a0, i1, r1, a1, b0, b1);    // transforms.py:117, from the magnitudes above
        if (MODE == FM_LOGMAGPHASE) {            // transforms.py:80-86
            a0 = __logf(a0 + 1e-8f);   // MUFU.LG2 * ln 2, as in the log-mel epilogue (|error| ~1e-6)
            a1 = __logf(a1 + 1e-8f);
        }
    }
    return make_float4(a0, a1, b0, b1);
}
template <class OutT>
__device__ __forceinline__ void store_piece(const FusedParams& p, int b, int f, int t, int pair, bool has1,
                                            float4 v) {
    const int C = p.C;
    OutT* o = reinterpret_cast<OutT*>(p.out) + ((size_t(b) * kBins + f) * p.T + t) * size_t(2 * C);
    if (C == 2) {
        store_out4(o, v);
    } else if (has1 && (C & 1) == 0) {
        store_out2(o + 2 * pair, v.x, v.y);
        store_out2(o + C + 2 * pair, v.z, v.w);
    } else {
        store_out1(o + 2 * pair, v.x);
        store_out1(o + (C + 2 * pair), v.z);
        if (has1) {
            store_out1(o + (2 * pair + 1), v.y);
            store_out1(o + (C + 2 * pair + 1), v.w);
        }
    }
}

// NJ: output registers per lane the epilogue needs: 4 = bins below 128 only (mel matrices
// whose support ends below bin 128), 8 = all 257 bins.
// EPI: 0 = every epilogue switch is read from FusedParams at run time; otherwise the 2-channel mel
// epilogues of a matrix with the default shape -- filters of at most 2 / 4 / 6 bins in the three
// rounds of 32, which is tf.signal.linear_to_mel_weight_matrix(80, 257, 16000), transforms.py:55 --
// with their switches fixed at compile time (EPI_C2 | EPI_MINMAX or EPI_LOG or neither): no
// per-round flag branches, no odd-channel selects, C folded into the address arithmetic, the
// projection loops unrolled to their 12 taps.  Measured: plain mel 202 -> 190 us.  (Those instances now exist
// with EPI_PLANE only: the 2-channel launches with bins below 128 read the bin planes.)
// EPI_REMAP: the mel epilogue of a channel remap (stereo_mono / random_merge_aug: 2 input channels, c_out
// output channels), switches read at run time like EPI == 0.
// EPI_MONO, alone or on top of the 2-channel variants above: mono_chan (include/iris.h IRIS_REMAP_MONO_CHAN)
// keeps two channels, so it is the 2-channel epilogue with (re0 + re1, re0 + im_j) formed before |.|.
// EPI_PLANE (NJ = 4, 2 channels, no remap or mono_chan): no FFT.  A stage is j_cnt rows of the sources' STFT
// bin planes (Bank::plane: bins 0..127 of one frame per 2 KB row, {re0, re1, im0, im1} per bin); lane l mixes
// bins l + 32 q in registers, product then sum as pipeline.merge_complex_specs rounds, and the magnitudes go to
// the same projection, extrema, log and store code as the FFT path.  With EPI_C2 the fixed-shape instance,
// without it the generic one (IRIS_NO_FIXED_EPI); both do the same arithmetic in the same order.
// OutT: element type of p.out (float, __nv_bfloat16, __half).  The half instances have no min-max
// epilogue: the min-max log-mel features are normalised by k_logmel_post, which converts.
// MODE FM_PLANE (NJ = 4) is the registration pass that writes a bank's plane from its waveform.
constexpr int EPI_MINMAX = 1, EPI_LOG = 2, EPI_C2 = 4, EPI_REMAP = 8, EPI_MONO = 16, EPI_PLANE = 32;
constexpr int kFixFR = 8;   // frames per tile of the fixed mel variants
__host__ __device__ constexpr int fixed_mel_L(int r) { return r == 0 ? 2 : (r == 1 ? 4 : (r == 2 ? 6 : 0)); }
template <int MODE, int NJ, int EPI, class OutT>
__global__ void __maxnreg__(kMaxRegs) k_fused(const __grid_constant__ FusedParams p) {
    extern __shared__ __align__(128) unsigned char sm[];
    // per-clip extrema of the CTA: {~bits(min), bits(max), warps arrived, -} per run of tiles of one
    // clip; the consumer warps are never more than S <= 3 tiles apart, 8 entries never collide
    __shared__ uint32_t s_mm[8][4];
    constexpr bool kMel = (MODE == FM_MEL);
    constexpr bool kFix = (EPI & EPI_C2) != 0;   // switches below are compile-time constants
    constexpr bool kRemap = (EPI == EPI_REMAP);
    constexpr bool kPlane = (EPI & EPI_PLANE) != 0;
    static_assert(!kPlane || (kMel && NJ == 4), "the plane epilogue is the 2-channel mel epilogue of bins below 128");
    static_assert(!kFix || kMel, "fixed epilogues exist for the mel modes only");
    static_assert(!kRemap || kMel, "the remap epilogue is a mel epilogue");
    constexpr bool kMono = (EPI & EPI_MONO) != 0;
    static_assert(!kMono || kMel, "the mono_chan epilogue is a mel epilogue");
    constexpr bool kF32 = sizeof(OutT) == 4;
    static_assert(kF32 || (MODE != FM_ACTIVITY && !(EPI & EPI_MINMAX)), "activity flags and the min-max epilogue are fp32 only");
    constexpr int S = slots_of(MODE);      // stage buffers
    const bool do_minmax = !kF32 ? false : kFix ? bool(EPI & EPI_MINMAX) : (p.do_minmax != 0);
    const bool do_lg = kFix ? bool(EPI & EPI_LOG) : (p.do_log && !p.do_minmax);
    const int C = kFix ? 2 : p.C;
    const int Cm = kRemap ? p.c_out : C;   // channels of the mel output
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    // fixed variants: 8 frames per tile and the 12 taps of the default mel shape, so that the
    // shared-memory map folds into immediates
    const int FR = kFix ? kFixFR : p.fr;
    const int mel_taps = kFix ? (fixed_mel_L(0) + fixed_mel_L(1) + fixed_mel_L(2)) : p.mel_taps;
    uint64_t* full = reinterpret_cast<uint64_t*>(sm + OFF_FULL);
    uint64_t* empty = reinterpret_cast<uint64_t*>(sm + OFF_EMPTY);
    const int n_tiles = p.B * ((p.T + FR - 1) / FR) * p.n_pairs;   // of the whole batch
    const uint32_t slotB = slot_bytes(FR);
    unsigned char* slots = sm + off_slots(mel_taps, FR);

    // ---- work claims of the producer warp (see there) ----
    const int chunks16 = p.tile_stride >> 4;
    const int CH = p.chunk, CM = p.chunk_mid, CT = p.chunk_tail;
    const long long n_big = p.n_big, n_mid = p.n_mid;
    auto claim_range = [&](long long q, int& len) -> long long {
        return iris::claim_range(CH, CM, CT, n_big, n_mid, q, len);
    };
    auto load_block = [&](int tile) -> int4 {
        const unsigned char* blk = p.tile_blocks + size_t(tile) * p.tile_stride;
        return lane < chunks16 ? __ldg(reinterpret_cast<const int4*>(blk) + lane) : make_int4(0, 0, 0, 0);
    };
    // the block of the CTA's first tile is requested before the setup below, not after it
    int len = 0;
    long long first = 0;
    int4 c_first = make_int4(0, 0, 0, 0);
    if (warp == FR) {
        cudaGridDependencySynchronize();   // the tile blocks come from the kernel in front (k_labels / k_tiles)
        first = claim_range(blockIdx.x, len);
        if (first < n_tiles) c_first = load_block(int(first));
    }

    // ---- one-time setup: barriers, finite data in the stage buffers (the tables are loaded by the
    // consumer warps while the producer warp is already fetching the first tile) ----
    {
        // rows of a slot outside a stage's frame range are read (and multiplied by 0) by the
        // frames the stage does not cover: they must hold finite numbers
        float4* z = reinterpret_cast<float4*>(slots);
        for (uint32_t i = tid; i < S * slotB / 16; i += blockDim.x) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tid < 32) s_mm[tid >> 2][tid & 3] = 0u;
        if (tid == 0) {
            for (int s = 0; s < S; ++s) {
                mbar_init(&full[s], 1);
                mbar_init(&empty[s], uint32_t(FR));
            }
            fence_mbar_init();
        }
        fence_proxy_async();   // the zero fill (generic proxy) precedes the bulk copies (async proxy)
        __syncthreads();
    }
    // everything above overlapped k_tiles (programmatic dependent launch); its tile blocks and the
    // zeroed extrema scratch are visible from here on
    cudaGridDependencySynchronize();

    if (warp == FR) {
        // =========================== producer warp ===========================
        // The producer is at most S stages ahead of the slowest consumer and every tile
        // has at least one stage, so when it writes ring entry i the slowest consumer is
        // still in tile >= i - S - 1: kRing > S + 1 entries never collide.
        uint32_t slot = 0, phase = 0;
        const uint64_t pol_stream = l2_policy_evict_first();
        // Work claims (launch_fused sets the schedule): claim q covers p.chunk consecutive tiles for
        // q < n_big, then p.chunk_mid tiles for n_mid claims, then p.chunk_tail tiles -- the chunks
        // shrink towards the end of the launch so that the CTAs finish within about one tile of each
        // other (whole chunks to the end left the slower CTA of an SM up to two chunks, ~20 us, behind).
        // The first claim of a CTA is its block index, the later ones come from a global counter and
        // are issued when the LAST tile of the current claim starts: a CTA never owns more than one
        // chunk.  Consecutive tiles of a clip mostly stay on one SM (per-clip state changes rarely,
        // the row shared by two tiles is re-read one tile later).
        int i = 0;
        if (first < n_tiles) {
            int tile = int(first);
            int last = int(min((long long)n_tiles, first + len));
            int4 c = c_first;
            while (true) {
                unsigned char* ent = sm + OFF_RING + (i & (kRing - 1)) * kTileBlockBytes;
                if (lane < chunks16) *reinterpret_cast<int4*>(ent + 16 * lane) = c;
                __syncwarp();
                const int n = __shfl_sync(0xffffffffu, c.x, 0);
                const TileBlock* tb = reinterpret_cast<const TileBlock*>(ent);
                // look ahead: the block of the next tile of this claim is fetched while the stages of
                // this one are issued; at the last tile of a claim the next claim goes out instead
                const bool more = tile + 1 < last;
                unsigned nxt = 0;
                int4 c2 = make_int4(0, 0, 0, 0);
                if (more) c2 = load_block(tile + 1);
                else if (lane == 0) nxt = atomicAdd(&p.sched[0], 1u);
                for (int s = 0; s < n; ++s) {
                    // the whole warp waits (one instruction per poll either way) so that it stays
                    // converged
                    mbar_wait_parked(&empty[slot], phase ^ 1u);
                    if (lane == 0) {
                        const StageDesc d = tb->d[s];
                        if (d.j_cnt == 0) {
                            mbar_arrive(&full[slot]);
                        } else {
                            // frames j_lo .. j_lo + j_cnt - 1: their plane rows, or the j_cnt + 1 waveform
                            // rows they span
                            const uint32_t bytes = (uint32_t(d.j_cnt) + (kPlane ? 0u : 1u)) * 2048u;
                            mbar_arrive_expect_tx(&full[slot], bytes);
                            bulk_g2s_hint(slots + slot * slotB + uint32_t(d.j_lo) * 2048u, d.src, bytes, &full[slot], pol_stream);
                        }
                    }
                    if (++slot == S) { slot = 0; phase ^= 1u; }
                }
                ++i;
                if (more) {
                    ++tile;
                    c = c2;
                } else {
                    const long long q = (long long)__shfl_sync(0xffffffffu, nxt, 0) + gridDim.x;
                    first = claim_range(q, len);
                    if (first >= n_tiles) break;
                    tile = int(first);
                    last = int(min((long long)n_tiles, first + len));
                    c = load_block(tile);
                }
            }
        }
        // no work left to claim: a kernel launched behind this one with programmatic stream
        // serialization (k_logmel_post) may be scheduled; it still waits for the whole grid
        cudaTriggerProgrammaticLaunchCompletion();
        // end marker: a TileBlock with n == 0 behind one more (empty) stage
        {
            unsigned char* ent = sm + OFF_RING + (i & (kRing - 1)) * kTileBlockBytes;
            if (lane == 0) *reinterpret_cast<int4*>(ent) = make_int4(0, 0, 0, 0);
            __syncwarp();
            mbar_wait_parked(&empty[slot], phase ^ 1u);
            if (lane == 0) {
                mbar_arrive(&full[slot]);
                // the last CTA to get here resets the work counter for the next launch
                if (atomicAdd(&p.sched[1], 1u) == gridDim.x - 1) {
                    p.sched[0] = 0u;
                    p.sched[1] = 0u;
                }
            }
        }
    } else {
        // =========================== consumer warps ===========================
        {
            // base powers of the inter-pass twiddle (fftwarp.cuh): p.tw1[q][n2] = {w^(2q), w^(2q+1)}
            float4* s_tw1 = reinterpret_cast<float4*>(sm + OFF_TW1);
            if (tid < 32) {
                const float4 q0 = p.tw1[tid], q1 = p.tw1[32 + tid], q2 = p.tw1[64 + tid], q4 = p.tw1[128 + tid];
                s_tw1[tid] = make_float4(q0.z, q0.w, q1.x, q1.y);
                s_tw1[32 + tid] = make_float4(q2.x, q2.y, q4.x, q4.y);
            }
            if (kMel) {
                uint32_t* s_ms = reinterpret_cast<uint32_t*>(sm + OFF_MSTART);
                for (int i = tid; i < kMaxMel; i += FR * 32) s_ms[i] = p.mel_info[i];   // [4 rounds][32 lanes]
                float* s_mw = reinterpret_cast<float*>(sm + OFF_MW);
                for (int i = tid; i < mel_taps * 32; i += FR * 32) s_mw[i] = p.mel_w[i];
            }
            float* s_hann = reinterpret_cast<float*>(sm + off_hann(mel_taps));
            for (int i = tid; i < 256; i += FR * 32) s_hann[i] = p.hann[i];
            named_bar_sync(2, FR * 32);   // consumer warps only
        }
        const int j = warp;                        // tile-relative frame of this warp
        const int k1 = warp_k1(lane), par = warp_par(lane);
        const float sgn = par ? -1.f : 1.f;
        const int partner = warp_partner(lane);
        const bool l0 = (lane == 0);
        // Hann[n], n = lane + 32 q, read from shared memory every frame (8 conflict-free LDS.32): held in
        // 8 registers per lane it pushed the spectrogram instances into spills -- 2-ch COMPLEX 302 ->
        // 287 us, 4-ch mel 377 -> 363 us with the table in shared memory, the 2-ch mel instances unchanged
        const float* w8 = reinterpret_cast<const float*>(sm + off_hann(mel_taps)) + lane;
        unsigned char* xch = sm + off_xch(mel_taps) + warp * kXwBytes;
        const float4* s_tw1 = reinterpret_cast<const float4*>(sm + OFF_TW1) + lane;
        const unsigned char* my_rows = slots + j * 2048 + lane * 8;
        // running per-clip extrema of this lane (flushed when the clip changes)
        float mn = __int_as_float(0x7f800000), mx = 0.f;
        int mm_clip = -1;
        uint32_t mm_run = 0;   // runs of tiles of one clip this warp has flushed (the same sequence in every warp)
        // The extrema of a run are combined in shared memory; the last of the FR warps to arrive sends
        // the CTA's pair to the global scratch.  (One red.global pair per WARP and clip change --
        // 81 k per 256-clip launch on 512 addresses -- measured 4 us of the kernel.)
        auto flush_minmax = [&]() {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            }
            if (lane == 0) {
                uint32_t* sl = s_mm[mm_run & 7];
                if (mn <= mx) {
                    atomicMax(&sl[0], ~__float_as_uint(mn));
                    atomicMax(&sl[1], __float_as_uint(mx));
                }
                __threadfence_block();
                if (atomicAdd(&sl[2], 1u) == uint32_t(FR) - 1u) {
                    __threadfence_block();
                    const uint32_t a = *reinterpret_cast<volatile uint32_t*>(&sl[0]);
                    const uint32_t c = *reinterpret_cast<volatile uint32_t*>(&sl[1]);
                    *reinterpret_cast<volatile uint32_t*>(&sl[0]) = 0u;
                    *reinterpret_cast<volatile uint32_t*>(&sl[1]) = 0u;
                    *reinterpret_cast<volatile uint32_t*>(&sl[2]) = 0u;
                    red_max_u32_if(&p.minmax[2 * mm_clip], a, (a | c) != 0u);
                    red_max_u32_if(&p.minmax[2 * mm_clip + 1], c, (a | c) != 0u);
                }
            }
            __syncwarp();
            ++mm_run;
            mn = __int_as_float(0x7f800000);
            mx = 0.f;
        };

        uint32_t slot = 0, phase = 0;
        const uint64_t pol_keep = l2_policy_evict_last();
        // mel rows are re-read by k_logmel_post: ask L2 to keep them (a 256-clip batch does not fit
        // anyway, but the hint measures 4-8 us better than plain stores)
        const bool keep_l2 = kMel && do_minmax;
        OutT* clip_out = reinterpret_cast<OutT*>(p.out);   // out[b, 0, 0, 0] of the current clip (mel modes)
        uint32_t zbits = 0;
        int zb_clip = -1;
        const size_t clip_elems = size_t(p.n_mel) * p.T * Cm;
        for (int i = 0;; ++i) {
            const TileBlock* tb = reinterpret_cast<const TileBlock*>(sm + OFF_RING + (i & (kRing - 1)) * kTileBlockBytes);
            int4 hdr;
            float4 z[4];   // EPI_PLANE: the mixed {re0, re1, im0, im1} of bins lane + 32 q
            cpx v[16];
            if constexpr (kPlane) {
                // ---- mix of the stored bins: z = sum over the stages of gain * X, product then sum ----
                mbar_wait_parked(&full[slot], phase);   // also publishes the TileBlock of this tile
                hdr = *reinterpret_cast<const int4*>(tb);
                if (hdr.x == 0) break;                  // end marker
                // a time-masked frame and one behind the clip's end are not read (they still release
                // every slot of the tile)
                const bool live = int(hdr.z & 0xffffff) + j < p.T && !((uint32_t(hdr.w) >> j) & 1u);
#pragma unroll
                for (int q = 0; q < 4; ++q) z[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int e = 0; e < hdr.x; ++e) {
                    if (e > 0) mbar_wait_parked(&full[slot], phase);
                    const uint2 dd = *reinterpret_cast<const uint2*>(&tb->d[e].j_lo);   // j_lo | j_cnt << 16, gain
                    if (live && unsigned(j - int(dd.x & 0xffffu)) < (dd.x >> 16)) {
                        const float g = __uint_as_float(dd.y);
                        const float4* src = reinterpret_cast<const float4*>(slots + slot * slotB + j * 2048) + lane;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float4 x = src[32 * q];
                            z[q].x = __fadd_rn(z[q].x, __fmul_rn(g, x.x));
                            z[q].y = __fadd_rn(z[q].y, __fmul_rn(g, x.y));
                            z[q].z = __fadd_rn(z[q].z, __fmul_rn(g, x.z));
                            z[q].w = __fadd_rn(z[q].w, __fmul_rn(g, x.w));
                        }
                    }
                    __syncwarp();
                    mbar_arrive_if(&empty[slot], l0);
                    if (++slot == S) { slot = 0; phase ^= 1u; }
                }
            } else {
            // ---- gather + mix: v = sum over the stages of this tile of gain * frame ----
            mbar_wait_parked(&full[slot], phase);           // also publishes the TileBlock of this tile
            // the rows of the first stage are requested before the tile header is looked at (the end
            // marker's rows are stale but finite): the header's load-to-use latency hides behind them
            {
                const float2* src = reinterpret_cast<const float2*>(my_rows + slot * slotB);
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const float2 x = src[32 * q];
                    v[q] = cpx{x.x, x.y};
                }
            }
            hdr = *reinterpret_cast<const int4*>(tb);
            const int n_st = hdr.x;
            if (n_st == 0) break;                    // end marker
            // (skipping the row reads of time-masked frames -- ~11 % of the frames -- was measured on
            // B200: +2..5 % kernel time; the extra branch costs registers (93 -> 96 + a spill) and the
            // kernel is bound by issue latency at 4.4 warps per scheduler, not by shared-memory wavefronts)
            {
                const uint2 dd = *reinterpret_cast<const uint2*>(&tb->d[0].j_lo);   // j_lo | j_cnt << 16, gain
                const bool active = unsigned(j - int(dd.x & 0xffffu)) < (dd.x >> 16);
                const float g0 = active ? __uint_as_float(dd.y) : 0.f;
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = cscale(v[q], g0);
                __syncwarp();
                mbar_arrive_if(&empty[slot], l0);
                if (++slot == S) { slot = 0; phase ^= 1u; }
            }
            for (int e = 1; e < n_st; ++e) {
                mbar_wait_parked(&full[slot], phase);
                const uint2 dd = *reinterpret_cast<const uint2*>(&tb->d[e].j_lo);
                const bool active = unsigned(j - int(dd.x & 0xffffu)) < (dd.x >> 16);
                if (active) {
                    const float gn = __uint_as_float(dd.y);
                    const float2* src = reinterpret_cast<const float2*>(my_rows + slot * slotB);
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const float2 x = src[32 * q];
                        v[q] = caxpy(gn, cpx{x.x, x.y}, v[q]);
                    }
                }
                __syncwarp();
                mbar_arrive_if(&empty[slot], l0);
                if (++slot == S) { slot = 0; phase ^= 1u; }
            }
            }

            const int b = hdr.y;
            const int pair = kFix ? 0 : (hdr.z >> 24);
            const int t = (hdr.z & 0xffffff) + j;
            const bool in_range = t < p.T;
            const bool has1 = kFix ? true : (2 * pair + 1 < C);
            // SpecAugment time mask of this frame (transforms.py:12-40), precomputed per tile
            const float mt = ((uint32_t(hdr.w) >> j) & 1u) ? 0.f : 1.f;
            // a fully time-masked frame has zero magnitude everywhere: no FFT needed for mel
            const bool do_fft = in_range && !(kMel && mt == 0.f);

            // per-lane bitmap of the bins zeroed by the frequency masks (transforms.py:12-40)
            // and stft_filter (data_utils.py:126-136): bit jj -> bin k1 + 16 (2 jj + par),
            // bit 8 -> bin 256.  Recomputed when the clip changes.
            if (b != zb_clip) {
                zb_clip = b;
                if (kMel) clip_out = reinterpret_cast<OutT*>(p.out) + size_t(b) * clip_elems;
                zbits = 0;
                const int4 fmv = *reinterpret_cast<const int4*>(tb->fm);
                if (kPlane) {
                    // the same bitmap; the lane holds bin lane + 32 q, bit `lane` of word q
                    zbits = ((uint32_t(fmv.x) >> lane) & 1u) | (((uint32_t(fmv.y) >> lane) & 1u) << 1) |
                            (((uint32_t(fmv.z) >> lane) & 1u) << 2) | (((uint32_t(fmv.w) >> lane) & 1u) << 3);
                } else if (kMel && NJ == 4) {
                    // k_tiles left a bitmap of the zeroed bins 0..127 (p.fm_bits): bin
                    // k1 + 16 par + 32 jj is bit k1 + 16 par of word jj
                    const int sh = k1 + 16 * par;
                    zbits = ((uint32_t(fmv.x) >> sh) & 1u) | (((uint32_t(fmv.y) >> sh) & 1u) << 1) |
                            (((uint32_t(fmv.z) >> sh) & 1u) << 2) | (((uint32_t(fmv.w) >> sh) & 1u) << 3);
                } else {
                const int fmw[4] = {fmv.x, fmv.y, fmv.z, fmv.w};   // size | offset << 16
#pragma unroll
                for (int q = 0; q <= 4; ++q) {
                    if (q < 4 && q >= p.n_fmask) continue;
                    if (q == 4 && !kMel) continue;   // store_bin filters after the channel remap
                    const int size = q < 4 ? (fmw[q] & 0xffff) : p.filter_k;
                    const int off = q < 4 ? (fmw[q] >> 16) : 1;
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj)
                        if (unsigned(k1 + 16 * (2 * jj + par) - off) < unsigned(size)) zbits |= 1u << jj;
                    if (NJ == 8 && unsigned(256 - off) < unsigned(size)) zbits |= 1u << 8;
                }
                }
            }

            cpx u[16];
            if (!kPlane && do_fft) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float wq = w8[32 * q];
                    v[q] = cscale(v[q], wq);
                    v[q + 8] = caxpy(-wq, v[q + 8], v[q + 8]);
                }
                {
                    const float4 wa = s_tw1[0], wb = s_tw1[32];
                    warp_pass1(v, cpx{wa.x, wa.y}, cpx{wa.z, wa.w}, cpx{wb.x, wb.y}, cpx{wb.z, wb.w});
                }
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    *reinterpret_cast<float2*>(xch + xw_write_off(k, lane)) = make_float2(v[k].x, v[k].y);
                __syncwarp();
                const unsigned char* row = xch + xw_read_off(k1, 0);
                // DIF twiddles t(i) = par ? W32^i : 1 selected from compile-time constants (a
                // table in shared memory would cost 32 wavefronts per frame for 256 bytes)
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
                __syncwarp();   // every lane is done with the exchange rows (reused for |X| below)
            }

            // ---- epilogue ----
            // register jj holds bin f = k1 + 16 (2 jj + par); its mirror 512 - f is register
            // 15 - jj of the partner lane (lane 0: its own register (16 - jj) & 15)
            auto mirror = [&](int jj) -> cpx {
                const cpx mine = l0 ? u[(16 - jj) & 15] : u[15 - jj];
                return cpx{__shfl_sync(0xffffffffu, mine.x, partner), __shfl_sync(0xffffffffu, mine.y, partner)};
            };
            if (kRemap) {
                // ---- mel of a channel remap: output pair q = channels (2q, 2q + 1) of c_out.  Pair 0 is the
                // two input channels; the others are per-bin linear combinations of them (remap_mix), so a
                // mask or stft_filter zero of a bin zeroes every output channel of it.  Each round of 32
                // filters is stored as soon as it is summed (no accumulators held across the rounds).
                //   NJ = 4: the magnitudes of kG = 4 pairs at a time are parked in the exchange rows (128
                //   float2 per pair, indexed by the bin), from (re ch0, re ch1, im ch0 + im ch1) of the
                //   lane's 4 bins kept in registers.
                //   NJ = 8: those 27 registers spill the FFT; the exchange rows hold (re ch0, re ch1, im ch0,
                //   im ch1) of all 257 bins instead (4112 B) and the projection forms the magnitudes of a
                //   pair from them tap by tap.
                if (do_minmax && b != mm_clip) {
                    if (mm_clip >= 0) flush_minmax();
                    mm_clip = b;
                }
                constexpr int kS = 128;
                constexpr int kG = NJ == 4 ? 4 : 1;
                static_assert(4 * 128 * 8 <= kXwBytes && kBins * 16 <= kXwBytes, "exchange rows too small");
                float2* mg = reinterpret_cast<float2*>(xch);
                float4* xv = reinterpret_cast<float4*>(xch);
                const uint32_t* ms = reinterpret_cast<const uint32_t*>(sm + OFF_MSTART) + lane;
                const int n_op = (Cm + 1) >> 1;
                float xr0[4], xr1[4], xis[4];   // NJ = 4: re ch0, re ch1, im ch0 + im ch1 of the lane's bins
                if (do_fft) {   // warp-uniform
                    auto split = [&](int i, int f, cpx zf, cpx zm) {
                        const cpx re = cadd(zf, zm);
                        const cpx im = cadd(cpx{zf.y, -zf.x}, cpx{-zm.y, zm.x});
                        const bool z = (zbits >> i) & 1u;
                        if constexpr (NJ == 4) {
                            const cpx sq = cfma2(im, im, cmul2(re, re));
                            mg[f] = make_float2(z ? 0.f : sqrt_approx(sq.x), z ? 0.f : sqrt_approx(sq.y));
                            xr0[i] = z ? 0.f : re.x;
                            xr1[i] = z ? 0.f : re.y;
                            xis[i] = z ? 0.f : im.x + im.y;
                        } else {
                            xv[f] = z ? make_float4(0.f, 0.f, 0.f, 0.f) : make_float4(re.x, re.y, im.x, im.y);
                        }
                    };
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) split(jj, k1 + 16 * (2 * jj + par), u[jj], mirror(jj));
                    if (NJ == 8) {
                        const cpx z8 = u[8];
                        if (l0) split(8, 256, z8, z8);
                    }
                }
                for (int g0 = 0; g0 < n_op; g0 += kG) {
                    if (NJ == 4 && do_fft) {
                        if (g0 > 0) __syncwarp();   // the previous group is projected
                        for (int k = (g0 == 0 ? 1 : 0); k < kG && g0 + k < n_op; ++k) {
                            const int ca = 2 * (g0 + k), cb = ca + 1;
                            const float2 ka = remap_coef(p, b, ca), kb = cb < Cm ? remap_coef(p, b, cb) : ka;
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const cpx za = remap_mix(p.remap, ka.x, ka.y, xr0[i], xr1[i], xis[i]);
                                const cpx zb = remap_mix(p.remap, kb.x, kb.y, xr0[i], xr1[i], xis[i]);
                                mg[k * kS + k1 + 16 * (2 * i + par)] =
                                    make_float2(sqrt_approx(fmaf(za.x, za.x, za.y * za.y)),
                                                sqrt_approx(fmaf(zb.x, zb.x, zb.y * zb.y)));
                            }
                        }
                    }
                    if (do_fft) __syncwarp();
                    for (int k = 0; k < kG && g0 + k < n_op; ++k) {
                        const int c = 2 * (g0 + k);
                        const bool has_b = c + 1 < Cm;
                        // NJ = 8: |.| of channels c, c + 1 of bin f from the parked split values
                        const float2 ka = c >= 2 ? remap_coef(p, b, c) : make_float2(0.f, 0.f);
                        const float2 kb = c >= 2 && has_b ? remap_coef(p, b, c + 1) : ka;
                        auto tap = [&](int f) -> float2 {
                            if constexpr (NJ == 4) {
                                return mg[k * kS + f];
                            } else {
                                const float4 v = xv[f];
                                if (c == 0)
                                    return make_float2(sqrt_approx(fmaf(v.x, v.x, v.z * v.z)),
                                                       sqrt_approx(fmaf(v.y, v.y, v.w * v.w)));
                                const cpx za = remap_mix(p.remap, ka.x, ka.y, v.x, v.y, v.z + v.w);
                                const cpx zb = remap_mix(p.remap, kb.x, kb.y, v.x, v.y, v.z + v.w);
                                return make_float2(sqrt_approx(fmaf(za.x, za.x, za.y * za.y)),
                                                   sqrt_approx(fmaf(zb.x, zb.x, zb.y * zb.y)));
                            }
                        };
                        // sparse projection as in the 2-channel epilogue below, then out[b, m, t, c .. c + 1]
                        const float* wr = reinterpret_cast<const float*>(sm + OFF_MW) + lane;
                        OutT* o_t = clip_out + t * Cm + c;
                        const uint32_t row_elems = uint32_t(p.T) * uint32_t(Cm);
#pragma unroll
                        for (int r = 0; r < 4; ++r) {
                            const int L = p.mel_L[r];   // uniform
                            if (L == 0) break;
                            cpx sacc{0.f, 0.f};
                            if (do_fft) {
                                const int f0 = p.mel_f_lo + int(ms[32 * r] & 0xffffu);
#pragma unroll
                                for (int q = 0; q < kMaxFilter; q += 2) {
                                    if (q >= L) break;
                                    const float2 x0 = tap(f0 + q), x1 = tap(f0 + q + 1);
                                    sacc = caxpy(wr[32 * q], cpx{x0.x, x0.y}, sacc);
                                    sacc = caxpy(wr[32 * q + 32], cpx{x1.x, x1.y}, sacc);
                                }
                            }
                            wr += 32 * L;
                            const uint32_t mrow = ms[32 * r] >> 16;
                            if (in_range && mrow != 0xffffu) {
                                OutT* o = o_t + mrow * row_elems;
                                float a0 = sacc.x, a1 = sacc.y;
                                if (do_minmax) {
                                    mn = fminf(mn, has_b ? fminf(a0, a1) : a0);
                                    mx = fmaxf(mx, has_b ? fmaxf(a0, a1) : a0);
                                }
                                if (do_lg) {
                                    a0 = __logf(a0 + 1e-8f);
                                    a1 = __logf(a1 + 1e-8f);
                                }
                                // (plain stores: the evict-last hint of the 2-channel epilogue costs
                                // registers this epilogue does not have)
                                if ((Cm & 1) == 0) {
                                    store_out2(o, a0, a1);
                                } else {
                                    store_out1(o, a0);
                                    if (has_b) store_out1(o + 1, a1);
                                }
                            }
                        }
                    }
                }
            } else if (kMel) {
                if (do_minmax && b != mm_clip) {
                    if (mm_clip >= 0) flush_minmax();
                    mm_clip = b;
                }
                // (|ch0|, |ch1|) of every bin the lane holds, indexed by the bin itself (at most 257 x 8 B
                // of the warp's 4352-byte exchange rows): no range checks on the way in
                float2* mg = reinterpret_cast<float2*>(xch);
                const int f_lo = p.mel_f_lo;
                float acc0[4], acc1[4];   // mel filter of slot (round r, lane): iris_set_mel's assignment
                const uint32_t* ms = reinterpret_cast<const uint32_t*>(sm + OFF_MSTART) + lane;
#pragma unroll
                for (int r = 0; r < 4; ++r) { acc0[r] = 0.f; acc1[r] = 0.f; }
                if (do_fft) {   // warp-uniform
                    auto emit = [&](int f, int bit, cpx zf, cpx zm) {
                        // (re ch0, re ch1) and (im ch0, im ch1) of the split, as packed pairs
                        cpx re = cadd(zf, zm);
                        cpx im = cadd(cpx{zf.y, -zf.x}, cpx{-zm.y, zm.x});
                        if constexpr (kMono) {   // z_j = (re0 + re1) + i (re0 + im_j); a masked bin is 0 either way
                            const float s = re.x + re.y;
                            im = cpx{re.x + im.x, re.x + im.y};
                            re = cpx{s, s};
                        }
                        const cpx sq = cfma2(im, im, cmul2(re, re));
                        float m0 = sqrt_approx(sq.x);
                        float m1 = sqrt_approx(sq.y);
                        if ((zbits >> bit) & 1u) { m0 = 0.f; m1 = 0.f; }   // |x| * 0 == +0
                        mg[f] = make_float2(m0, m1);
                    };
                    if constexpr (kPlane) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            cpx re{z[q].x, z[q].y}, im{z[q].z, z[q].w};
                            if constexpr (kMono) {
                                const float s = re.x + re.y;
                                im = cpx{re.x + im.x, re.x + im.y};
                                re = cpx{s, s};
                            }
                            const cpx sq = cfma2(im, im, cmul2(re, re));
                            float m0 = sqrt_approx(sq.x);
                            float m1 = sqrt_approx(sq.y);
                            if ((zbits >> q) & 1u) { m0 = 0.f; m1 = 0.f; }
                            mg[lane + 32 * q] = make_float2(m0, m1);
                        }
                    } else {
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) emit(k1 + 16 * (2 * jj + par), jj, u[jj], mirror(jj));
                    if (NJ == 8) {
                        const cpx z8 = u[8];
                        if (l0) emit(256, 8, z8, z8);
                    }
                    }
                    __syncwarp();
                    // sparse mel projection (transforms.py:51-77): the filter of slot (r, lane) reads
                    // mel_L[r] taps starting at its first bin (low half of the slot's info word);
                    // shorter filters are zero-padded, so the trip count is uniform across the warp
                    const float* wr = reinterpret_cast<const float*>(sm + OFF_MW) + lane;
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const int L = kFix ? fixed_mel_L(r) : p.mel_L[r];   // 0 for r >= ceil(n_mel / 32); uniform
                        if (L == 0) break;
                        const float2* a = mg + f_lo + (ms[32 * r] & 0xffffu);
                        cpx sacc{0.f, 0.f};   // (ch0, ch1)
#pragma unroll
                        for (int q = 0; q < kMaxFilter; q += 2) {   // L is even (iris_set_mel pads)
                            if (q >= L) break;                        // uniform
                            const float2 x0 = a[q], x1 = a[q + 1];
                            const float w0 = wr[32 * q], w1 = wr[32 * q + 32];
                            sacc = caxpy(w0, cpx{x0.x, x0.y}, sacc);
                            sacc = caxpy(w1, cpx{x1.x, x1.y}, sacc);
                        }
                        acc0[r] = sacc.x;
                        acc1[r] = sacc.y;
                        wr += 32 * L;
                    }
                    // (the mags are consumed before the next frame's exchange writes: the
                    // __syncwarp() of the next tile's first mixing stage lies in between)
                }
                // ---- every lane stores its own mel values: out[b, m, t, 2*pair .. +1] ----
                if (in_range) {
                    OutT* o_t = clip_out + t * C + 2 * pair;
                    const uint32_t row_elems = uint32_t(p.T) * uint32_t(C);
                    const bool lg = do_lg;
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        if (kFix ? (fixed_mel_L(r) == 0) : (p.mel_L[r] == 0)) break;   // uniform: no work behind the last round
                        const uint32_t mrow = ms[32 * r] >> 16;   // mel row of this slot; 0xffff: idle lane
                        if (mrow != 0xffffu) {
                            OutT* o = o_t + mrow * row_elems;
                            float a0 = acc0[r], a1 = acc1[r];
                            if (do_minmax) {
                                mn = fminf(mn, has1 ? fminf(a0, a1) : a0);
                                mx = fmaxf(mx, has1 ? fmaxf(a0, a1) : a0);
                            }
                            if (lg) {
                                a0 = __logf(a0 + 1e-8f);
                                a1 = __logf(a1 + 1e-8f);
                            }
                            if ((C & 1) == 0) {
                                // (mono_chan with NJ = 8: plain stores, the hint's registers spill)
                                if constexpr (kF32 && !(kMono && NJ == 8)) {
                                    if (keep_l2) st_f2_hint(o, a0, a1, pol_keep);
                                    else store_out2(o, a0, a1);
                                } else {
                                    store_out2(o, a0, a1);
                                }
                            } else {
                                store_out1(o, a0);
                                if (has1) store_out1(o + 1, a1);
                            }
                        }
                    }
                }
            } else if (MODE == FM_PLANE) {
                // bins 0..127 of frame t of item b into row t of its plane (pl_delta[0] floats behind its
                // waveform): with the stage gain 1/2 the split values are X itself.  One segment per item
                // (bank_fill); frames past the item's end keep the zeros the plane was cleared to.
                const Seg sg = p.segs[p.seg_ptr[b]];
                if (do_fft && t < sg.t_hi) {
                    float4* row = reinterpret_cast<float4*>(const_cast<float*>(sg.base) + p.pl_delta[0] + size_t(t) * 512);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const cpx zf = u[jj], zm = mirror(jj);
                        row[k1 + 16 * (2 * jj + par)] = make_float4(zf.x + zm.x, zf.y + zm.y, zf.y - zm.y, zm.x - zf.x);
                    }
                }
            } else if (MODE == FM_ACTIVITY) {
                // frame "active" iff any STFT coefficient (any bin, re or im, any channel) > 0
                // (pipeline.py:55)
                float mxv = 0.f;
                if (do_fft) {
                    auto emit = [&](cpx zf, cpx zm) {
                        mxv = fmaxf(mxv, fmaxf(fmaxf(zf.x + zm.x, zf.y - zm.y),
                                               fmaxf(zf.y + zm.y, zm.x - zf.x)));
                    };
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) emit(u[jj], mirror(jj));
                    if (l0) emit(u[8], u[8]);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mxv = fmaxf(mxv, __shfl_xor_sync(0xffffffffu, mxv, o));
                if (in_range && l0 && mxv > 0.f) p.activity[size_t(b) * p.T + t] = 1;
            } else if (MODE == FM_SE) {
                // ---- the 'se' batch (include/iris.h, IRIS_FEAT_SE): the tile's channel pair 0 is the mix of the
                // kept voices, pair 1 background + noises (build_tile_block, seg_select 3); consecutive tiles of
                // this CTA, as in the 4-channel combined store below.  Pair 0 parks (Re V0, Re V1) in the staging
                // area, pair 1 parks (Re N0, Re N1, mask) in its exchange rows; the store phase of pair 1 writes,
                // for bins 1..256, x = (V + N) * mask * filter, only_voice = Re V0, only_noise = Re N0.  Every
                // in-range frame runs the FFT: the masks zero x only.
                float4* stg = reinterpret_cast<float4*>(slots + S * slotB);
                float4* park = pair == 1 ? reinterpret_cast<float4*>(xch) : stg;
                if (do_fft) {
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) {
                        const int f = k1 + 16 * (2 * jj + par);
                        const cpx zf = u[jj], zm = mirror(jj);
                        park[pair == 1 ? (f ^ j) : f * FR + (j ^ (f & 7))] =
                            make_float4(zf.x + zm.x, zf.y + zm.y, ((zbits >> jj) & 1u) ? 0.f : mt, 0.f);
                    }
                    if (l0) {
                        const cpx zf = u[8];
                        park[pair == 1 ? (256 ^ j) : 256 * FR + j] =
                            make_float4(zf.x + zf.x, zf.y + zf.y, ((zbits >> 8) & 1u) ? 0.f : mt, 0.f);
                    }
                }
                if (pair == 1) {   // warp-uniform (tile header)
                    named_bar_sync(1, FR * 32);
                    const int jt = lane & 7;
                    const int tt = (hdr.z & 0xffffff) + jt;
                    if (tt < p.T) {
                        const size_t cells = size_t(p.B) * 256 * p.T;   // (bin, frame) cells of one block channel
                        float* ov = p.out + 2 * cells;
                        float* on = ov + cells;
                        const unsigned char* x1 = sm + off_xch(mel_taps) + jt * kXwBytes;
                        for (int f = warp * 4 + (lane >> 3); f < kBins; f += FR * 4) {
                            if (f == 0) continue;
                            const float4 v = stg[f * FR + (jt ^ (f & 7))];
                            const float4 n = *reinterpret_cast<const float4*>(x1 + ((f ^ jt) << 4));
                            float a0 = (v.x + n.x) * n.z, a1 = (v.y + n.y) * n.z;   // masks by multiplication
                            if (f <= p.filter_k) { a0 *= 0.f; a1 *= 0.f; }          // data_utils.py:126-136
                            const size_t c = (size_t(b) * 256 + (f - 1)) * p.T + tt;
                            *reinterpret_cast<float2*>(p.out + 2 * c) = make_float2(a0, a1);
                            ov[c] = v.x;
                            on[c] = n.x;
                        }
                    }
                    named_bar_sync(1, FR * 32);   // staging + exchange rows are read before they are reused
                }
            } else if (p.stage_out) {
                // ---- spectrogram modes: every warp parks the 257 x 16 B pieces of its frame in
                // the staging area, then the 8 warps store bin rows of 8 frames = 128 B each ----
                float4* stg = reinterpret_cast<float4*>(slots + S * slotB);
                // 4-channel clips (p.pair_merge): the two channel pairs of a (clip, time) range are
                // consecutive tiles of one CTA.  Pair 0 only parks its pieces in the staging area;
                // pair 1 parks its own in the warp's (now idle) exchange rows -- bin f of frame j at
                // 16-byte position f ^ j, so that the 8 frames of a bin fall into 8 distinct bank
                // groups -- and the store phase writes whole 32-byte cells [re0..re3 | im0..im3]:
                // 8 frames = 256 contiguous bytes per bin instead of four 8-byte pieces per cell
                // written by two different tiles.
                const bool merge = p.pair_merge != 0;
                float4* park = (merge && pair == 1) ? reinterpret_cast<float4*>(xch) : stg;
                if (do_fft) {
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) {
                        const int f = k1 + 16 * (2 * jj + par);
                        const cpx zf = u[jj], zm = mirror(jj);
                        const int pos = (merge && pair == 1) ? (f ^ j) : f * FR + (j ^ (f & 7));
                        park[pos] =
                            make_piece<MODE>(p, f, zf.x + zm.x, zf.y - zm.y, zf.y + zm.y, zm.x - zf.x,
                                             ((zbits >> jj) & 1u) ? 0.f : mt);
                    }
                    if (l0) {
                        const cpx zf = u[8];
                        const int pos = (merge && pair == 1) ? (256 ^ j) : 256 * FR + j;
                        park[pos] = make_piece<MODE>(p, 256, zf.x + zf.x, zf.y - zf.y, zf.y + zf.y,
                                                     zf.x - zf.x, ((zbits >> 8) & 1u) ? 0.f : mt);
                    }
                }
                if (merge) {
                    if (pair == 1) {   // warp-uniform (tile header)
                        named_bar_sync(1, FR * 32);
                        const int jt = lane & 7, half = (lane >> 3) & 1;
                        const int tt = (hdr.z & 0xffffff) + jt;
                        if (tt < p.T) {
                            const unsigned char* x1 = sm + off_xch(mel_taps) + jt * kXwBytes + half * 8;
                            const unsigned char* x0 = reinterpret_cast<const unsigned char*>(stg) + half * 8;
                            OutT* o = reinterpret_cast<OutT*>(p.out) + (size_t(b) * kBins * p.T + tt) * 8 + half * 4;
                            for (int f = warp * 2 + (lane >> 4); f < kBins; f += FR * 2) {
                                const float2 a = *reinterpret_cast<const float2*>(x0 + (f * FR + (jt ^ (f & 7))) * 16);
                                const float2 c = *reinterpret_cast<const float2*>(x1 + ((f ^ jt) << 4));
                                store_out4(o + size_t(f) * p.T * 8, make_float4(a.x, a.y, c.x, c.y));
                            }
                        }
                        named_bar_sync(1, FR * 32);   // staging + exchange rows are read before they are reused
                    }
                    continue;
                }
                named_bar_sync(1, FR * 32);
                {
                    const int jt = lane & 7;                       // frame of the tile
                    const int tt = (hdr.z & 0xffffff) + jt;
                    if (tt < p.T) {
                        for (int f = warp * 4 + (lane >> 3); f < kBins; f += FR * 4)
                            store_piece<OutT>(p, b, f, tt, pair, has1, stg[f * FR + (jt ^ (f & 7))]);
                    }
                }
                named_bar_sync(1, FR * 32);   // the pieces are read before the next tile overwrites them
            } else if (do_fft) {
                // channel remaps: stft_filter is applied by store_bin (it follows the remap)
                const bool mono = p.remap == REMAP_MONO_CHAN;
                auto store = [&](int f, float r0, float i0, float r1, float i1, float m) {
                    if (mono) store_bin<MODE, OutT, true>(p, b, f, t, pair, has1, r0, i0, r1, i1, m);
                    else store_bin<MODE, OutT, false>(p, b, f, t, pair, has1, r0, i0, r1, i1, m);
                };
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const int f = k1 + 16 * (2 * jj + par);
                    const cpx zf = u[jj], zm = mirror(jj);
                    store(f, zf.x + zm.x, zf.y - zm.y, zf.y + zm.y, zm.x - zf.x, ((zbits >> jj) & 1u) ? 0.f : mt);
                }
                if (l0) {
                    const cpx zf = u[8];
                    store(256, zf.x + zf.x, zf.y - zf.y, zf.y + zf.y, zf.x - zf.x, ((zbits >> 8) & 1u) ? 0.f : mt);
                }
            }
        }
        if (kMel && do_minmax && mm_clip >= 0) flush_minmax();
    }
}

size_t fused_smem_bytes(const FusedParams& p, int mode) { return smem_total(p.mel_taps, p.fr, mode, p.stage_out != 0); }
int fused_max_segments() { return kMaxStages; }
bool fused_stages_output(int mode, int remap, int fr) { return stages_output(mode, remap, fr); }
int fused_max_mel_taps() { return kMaxTaps; }
int fused_max_mel_filter() { return kMaxFilter; }

// Frames per tile = consumer warps per CTA.  FR = 8 (two CTAs of 8 + 1 warps per SM: the
// consumer warps spread evenly over the 4 schedulers and two independent CTAs hide each
// other's load waits) measured fastest on B200: cfg2 mel 216 us vs 228 us for FR = 16 x 1 CTA
// and 271 us for FR = 20 at 80 registers (spills).
int fused_pick_fr(int mel_taps) {
    int want = kFixFR;
    while (want > 1 && smem_total(mel_taps, want, FM_MEL, false) > 227u * 1024u - 256u) --want;
    return want;
}

size_t fused_tile_bytes(const FusedParams& p, int* stride_out) {
    const int FR = p.fr;
    const long long n_tiles = (long long)p.B * p.n_pairs * ((p.T + FR - 1) / FR);
    int ms = p.max_segs < 1 ? 1 : p.max_segs;
    const int stride = 32 + 16 * ms;
    if (stride_out) *stride_out = stride;
    return size_t(n_tiles) * size_t(stride);
}

// Claim schedule of a launch (see the producer warp): whole chunks first, then half chunks for the
// last kTailMid tiles per CTA, single tiles (tile pairs of a 4-channel clip) for the last kTailOne.
// Measured on B200 (profiles/r02_trace_*.txt): with whole chunks to the end the CTAs of a 256-clip
// launch finish 22 us apart (the slower of the two CTAs of an SM needs ~13 us for a chunk of 4 and
// used to own a second one).
constexpr int kTailOne = 2, kTailMid = 6;
static void fused_schedule(FusedParams& p, long long n_tiles, int grid) {
    const int unit = p.pair_merge ? 2 : 1;   // both channel pairs of a (clip, time) range in one claim
    p.chunk_tail = unit;
    p.chunk_mid = (p.chunk / 2) / unit * unit;
    if (p.chunk_mid < unit) p.chunk_mid = unit;
    if (p.chunk <= unit) {   // nothing to shrink
        p.chunk_mid = p.chunk_tail = p.chunk;
        p.n_big = 0x7fffffff;
        p.n_mid = 0;
        return;
    }
    const long long tail_one = (long long)grid * kTailOne, tail_mid = (long long)grid * kTailMid;
    const long long rem = n_tiles > tail_one ? n_tiles - tail_one : 0;
    const long long mid = rem < tail_mid ? rem : tail_mid;
    p.n_big = int32_t((rem - mid) / p.chunk);
    p.n_mid = int32_t((rem - (long long)p.n_big * p.chunk) / p.chunk_mid);
}

// the schedule a launch of n_tiles tiles on `grid` CTAs would get: {chunk, chunk_mid, chunk_tail, n_big, n_mid}
void fused_debug_schedule(long long n_tiles, int grid, int chunk, int pair_merge, int32_t out[5]) {
    FusedParams p;
    memset(&p, 0, sizeof p);
    p.chunk = chunk;
    p.pair_merge = pair_merge;
    if (p.pair_merge && (p.chunk & 1)) ++p.chunk;
    fused_schedule(p, n_tiles, grid);
    out[0] = p.chunk; out[1] = p.chunk_mid; out[2] = p.chunk_tail; out[3] = p.n_big; out[4] = p.n_mid;
}

// The one rule for which launches read the banks' STFT bin planes instead of transforming the waveform: the
// mel modes of 2-channel waveform banks (the caller has filled pl_wave / pl_floats / pl_delta: every
// 2-channel waveform bank has a plane) whose channels stay two (no remap, or mono_chan) and whose mel support
// ends below bin 128 -- the bins a plane row holds.  prepare_fused sets p.plane from it, so that the tile
// blocks (k_tiles, k_labels) point into the planes.
bool fused_reads_plane(const FusedParams& p, int mode) {
    return mode == FM_MEL && p.C == 2 && (p.remap == REMAP_NONE || p.remap == REMAP_MONO_CHAN) &&
           p.mel_f_lo + p.mel_f_n <= 128 && p.seg_select == 0 && p.pl_wave[0] != nullptr;
}

// Persistent grid: as many CTAs as are resident at once, asked of the occupancy calculator once per kernel
// instance and device.  The register cap decides between 1 and 2 CTAs per SM: measured on B200, 96 registers
// give 2 x 9 warps, 104 and 112 only one CTA (576 x 112 = 64512 < 65536, but registers are granted per warp in
// larger units) -- 4-ch COMPLEX 570 -> 730 us, mel 200 -> 265 us.
template <int MODE, int NJ, int EPI, class OutT>
static cudaError_t launch_instance(FusedParams p, long long n_tiles, size_t smem, int num_sms, cudaStream_t stream) {
    const auto kernel = k_fused<MODE, NJ, EPI, OutT>;
    const int threads = (p.fr + 1) * 32;
    int dev = 0;
    cudaGetDevice(&dev);
    static int attr_dev = -1;   // function attributes are per device
    static int per_sm = 1;
    static size_t per_sm_smem = 0;
    if (attr_dev != dev) {
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - int(fa.sharedSizeBytes));
        if (e != cudaSuccess) return e;
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        attr_dev = dev;
        per_sm_smem = 0;
    }
    if (per_sm_smem != smem) {
        int nb = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem);
        if (e != cudaSuccess) return e;
        per_sm = nb < 1 ? 1 : nb;
        per_sm_smem = smem;
    }
    const long long max_ctas = (long long)num_sms * per_sm;
    const int grid = int(n_tiles < max_ctas ? n_tiles : max_ctas);
    fused_schedule(p, n_tiles, grid);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(unsigned(grid));
    cfg.blockDim = dim3(unsigned(threads));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, p);
}

// the instance of p.out's OutType
template <int MODE, int NJ, int EPI>
static cudaError_t launch_out(int out_type, const FusedParams& p, long long n_tiles, size_t smem, int num_sms,
                              cudaStream_t stream) {
    if (out_type == OUT_BF16) return launch_instance<MODE, NJ, EPI, __nv_bfloat16>(p, n_tiles, smem, num_sms, stream);
    if (out_type == OUT_F16) return launch_instance<MODE, NJ, EPI, __half>(p, n_tiles, smem, num_sms, stream);
    return launch_instance<MODE, NJ, EPI, float>(p, n_tiles, smem, num_sms, stream);
}

// a launch that reads the bin planes: EPI_PLANE | X, X = 0 or EPI_MONO for mono_chan; fixed: the default mel shape
template <int X>
static cudaError_t launch_plane(bool fixed, int out_type, const FusedParams& p, long long n_tiles, size_t smem,
                                int num_sms, cudaStream_t stream) {
    constexpr int kEpi = EPI_PLANE | X;
    if (!fixed) return launch_out<FM_MEL, 4, kEpi>(out_type, p, n_tiles, smem, num_sms, stream);
    if (p.do_minmax)
        return launch_instance<FM_MEL, 4, kEpi | EPI_C2 | EPI_MINMAX, float>(p, n_tiles, smem, num_sms, stream);
    if (p.do_log) return launch_out<FM_MEL, 4, kEpi | EPI_C2 | EPI_LOG>(out_type, p, n_tiles, smem, num_sms, stream);
    return launch_out<FM_MEL, 4, kEpi | EPI_C2>(out_type, p, n_tiles, smem, num_sms, stream);
}

// p.tile_blocks (fused_tile_bytes) is provided by the caller; build_tiles: k_tiles builds them first
// (otherwise the kernel in front -- k_labels -- has built them and triggers early).  out_type: OutType
// of p.out; FM_ACTIVITY and the min-max epilogue write fp32 only.
cudaError_t launch_fused(const FusedParams& p, int mode, int num_sms, cudaStream_t stream, bool build_tiles,
                         int out_type) {
    const int FR = p.fr;
    if (FR < 1 || FR > kMaxFR) return cudaErrorInvalidValue;
    const int tpc = (p.T + FR - 1) / FR;
    const long long n_tiles = (long long)p.B * p.n_pairs * tpc;
    if (n_tiles <= 0) return cudaSuccess;
    if (n_tiles > 0x7fffffffLL || p.max_segs > kMaxStages || p.n_pairs > 127) return cudaErrorInvalidValue;
    if (mode == FM_MEL && (long long)p.n_mel * p.T * p.c_out > 0x7fffffffLL) return cudaErrorInvalidValue;   // 32-bit row offsets inside a clip
    if (mode == FM_MEL && p.remap != REMAP_NONE &&
        (p.C != 2 || (p.remap == REMAP_MONO_CHAN ? p.c_out != 2 : p.c_out < 3)))
        return cudaErrorInvalidValue;
    const size_t smem = fused_smem_bytes(p, mode);
    if (smem > 227 * 1024 - 256) return cudaErrorInvalidValue;   // (128 B of static shared memory: s_mm)
    if (out_type != OUT_F32 && ((out_type != OUT_BF16 && out_type != OUT_F16) || mode == FM_ACTIVITY || p.do_minmax))
        return cudaErrorInvalidValue;
    if (build_tiles) k_tiles<<<unsigned((n_tiles + 127) / 128), 128, 0, stream>>>(p);
    // k_fused is a programmatic dependent launch behind k_tiles / k_labels: its prologue overlaps
    // their tail
    cudaError_t e;
    switch (mode) {
        case FM_COMPLEX: e = launch_out<FM_COMPLEX, 8, 0>(out_type, p, n_tiles, smem, num_sms, stream); break;
        case FM_MAGPHASE: e = launch_out<FM_MAGPHASE, 8, 0>(out_type, p, n_tiles, smem, num_sms, stream); break;
        case FM_LOGMAGPHASE: e = launch_out<FM_LOGMAGPHASE, 8, 0>(out_type, p, n_tiles, smem, num_sms, stream); break;
        case FM_MEL: {
            // p.plane (fused_reads_plane): 2 channels, no remap or mono_chan, support below bin 128 -- the mix of
            // the banks' stored bins, fixed-shape or generic instance.  Otherwise the FFT path: NJ = 8 for a
            // support reaching bin 128, NJ = 4 for C != 2 and the stereo_mono / random_merge_aug remaps.
            if (p.plane != (fused_reads_plane(p, mode) ? 1 : 0)) return cudaErrorInvalidValue;
            const bool nj8 = p.mel_f_lo + p.mel_f_n > 128;
            if (p.plane) {
                const bool fixed = p.mel_L[0] == fixed_mel_L(0) && p.mel_L[1] == fixed_mel_L(1) &&
                                   p.mel_L[2] == fixed_mel_L(2) && p.mel_L[3] == fixed_mel_L(3) && FR == kFixFR &&
                                   p.mel_taps == 12 && !getenv("IRIS_NO_FIXED_EPI");
                if (p.remap == REMAP_MONO_CHAN)
                    e = launch_plane<EPI_MONO>(fixed, out_type, p, n_tiles, smem, num_sms, stream);
                else
                    e = launch_plane<0>(fixed, out_type, p, n_tiles, smem, num_sms, stream);
            } else if (p.remap == REMAP_MONO_CHAN) {
                if (!nj8) return cudaErrorInvalidValue;   // bins below 128 only: the plane path
                e = launch_out<FM_MEL, 8, EPI_MONO>(out_type, p, n_tiles, smem, num_sms, stream);
            } else if (p.remap != REMAP_NONE) {
                if (nj8) e = launch_out<FM_MEL, 8, EPI_REMAP>(out_type, p, n_tiles, smem, num_sms, stream);
                else e = launch_out<FM_MEL, 4, EPI_REMAP>(out_type, p, n_tiles, smem, num_sms, stream);
            } else if (nj8) {
                e = launch_out<FM_MEL, 8, 0>(out_type, p, n_tiles, smem, num_sms, stream);
            } else {
                if (p.C == 2) return cudaErrorInvalidValue;   // the plane path
                e = launch_out<FM_MEL, 4, 0>(out_type, p, n_tiles, smem, num_sms, stream);
            }
            break;
        }
        case FM_ACTIVITY: e = launch_instance<FM_ACTIVITY, 8, 0, float>(p, n_tiles, smem, num_sms, stream); break;
        case FM_PLANE: e = launch_instance<FM_PLANE, 4, 0, float>(p, n_tiles, smem, num_sms, stream); break;
        case FM_SE:   // both virtual pairs of a (clip, time) range in one CTA: the combined store
            if (out_type != OUT_F32 || !p.pair_merge || p.seg_select != 3) return cudaErrorInvalidValue;
            e = launch_instance<FM_SE, 8, 0, float>(p, n_tiles, smem, num_sms, stream);
            break;
        default: return cudaErrorInvalidValue;
    }
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

}  // namespace iris
