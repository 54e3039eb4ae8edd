// Per-tile stage lists of the fused kernel (k_fused.cu): a tile is `fr` consecutive output frames of
// one (clip, channel pair); its TileBlock lists the mixing segments that are kept and overlap it
// plus the tile's mask bits.  Built by k_tiles (k_fused.cu) or, when a label pass runs in front of the
// feature launch anyway, by the CTA of k_labels that has just decided the clip's keep flags
// (k_labels.cu) -- one kernel launch less on the critical path of a step.
#pragma once
#include "iris_common.cuh"

namespace iris {

#ifndef IRIS_MAX_STAGES
#define IRIS_MAX_STAGES 24
#endif
constexpr int kMaxStages = IRIS_MAX_STAGES;   // mixing segments of one clip (upper bound on stages per tile; the ring copy takes <= 30)

struct StageDesc {
    const float* src;      // first row of the stage in the pair plane of the source
    uint16_t j_lo, j_cnt;  // tile-relative frames [j_lo, j_lo + j_cnt); j_cnt == 0: empty stage
    float gain;            // 0.5 * gain (the 1/2 of the two-channel split)
};
static_assert(sizeof(StageDesc) == 16, "StageDesc layout");

struct TileBlock {
    int32_t n;             // stages (>= 1)
    int32_t b;             // clip
    int32_t t0_pair;       // first frame | pair << 24
    uint32_t tmask_bits;   // bit j: frame t0 + j is time-masked (transforms.py:12-40)
    int16_t fm[8];         // (size, offset) x 4 frequency masks of the clip
    StageDesc d[kMaxStages];
};
static_assert(sizeof(TileBlock) == 32 + 16 * kMaxStages, "TileBlock layout");
constexpr int kTileBlockBytes = int(sizeof(TileBlock));


// Work claims of the persistent feature kernel (k_fused.cu, fused_schedule): claim q covers `chunk`
// consecutive tiles for q < n_big, `chunk_mid` tiles for the next n_mid claims, `chunk_tail` tiles after
// that; returns the first tile (>= the tile count: no work left) and the length in `len`.  Shared by the
// producer warp and the host-side check of the schedule (iris_debug_claims).
__host__ __device__ inline long long claim_range(int chunk, int chunk_mid, int chunk_tail, long long n_big,
                                                 long long n_mid, long long q, int& len) {
    if (q < n_big) { len = chunk; return q * chunk; }
    q -= n_big;
    if (q < n_mid) { len = chunk_mid; return n_big * chunk + q * chunk_mid; }
    len = chunk_tail;
    return n_big * chunk + n_mid * chunk_mid + (q - n_mid) * chunk_tail;
}

// tile = (clip * tiles_per_clip + time_tile) * n_pairs + pair, per_clip = tiles_per_clip * n_pairs
// seg_cache / keep_cache / tm_cache / fm_cache: the clip's segments, their keep flags (1 = kept or not a
// voice) and its mask rectangles staged in shared memory by the caller (k_labels), or null: read them
// from the plan.
// SE: the layout of FM_SE (p.seg_select == 3), two virtual channel pairs over bank pair 0: pair 0 takes the
// kept voices, pair 1 background + noises.  (A compile-time variant: a run-time select spills k_labels.)
template <bool SE = false>
__device__ __forceinline__ void build_tile_block(const FusedParams& p, int tile, int per_clip,
                                                 const Seg* seg_cache = nullptr, const uint8_t* keep_cache = nullptr,
                                                 const int32_t* tm_cache = nullptr, const int32_t* fm_cache = nullptr) {
    const int FR = p.fr;
    // tile order: clip, then time, then channel pair -- the pairs of one (clip, time) range are
    // consecutive tiles (same work chunk), so the partial sectors they write to the same
    // out[b, f, t, :] rows merge in L2 within microseconds
    const int b = tile / per_clip;
    const int r = tile - b * per_clip;
    const int pair = r % p.n_pairs;
    const int t0 = (r / p.n_pairs) * FR;
    const int t_end = min(t0 + FR, p.T);
    unsigned char* blk = p.tile_blocks + size_t(tile) * p.tile_stride;
    StageDesc* d = reinterpret_cast<StageDesc*>(blk + 32);
    int n = 0;
    const int s0 = p.seg_ptr[b], s1 = p.seg_ptr[b + 1];
    for (int s = s0; s < s1; ++s) {
        const Seg sg = seg_cache ? seg_cache[s - s0] : p.segs[s];
        const int lo = max(sg.t_lo, t0), hi = min(sg.t_hi, t_end);
        const bool kept = seg_cache ? keep_cache[s - s0] != 0 : !(sg.keep_idx >= 0 && p.keep[sg.keep_idx] == 0);
        if (lo >= hi || !kept) continue;
        if (SE ? ((sg.keep_idx >= 0) != (pair == 0))
               : ((p.seg_select == 1 && sg.keep_idx < 0) || (p.seg_select == 2 && sg.keep_idx >= 0)))
            continue;
        if (n < p.max_segs) {
            StageDesc e;
            e.src = sg.base + size_t(SE ? 0 : pair) * size_t(sg.pair_stride) + size_t(lo + sg.shift) * 512;
            if (!SE && p.plane) {
                // the same row of the source's bin plane (one 2 KB row per frame, the waveform's geometry)
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    if (uint64_t(e.src) - uint64_t(p.pl_wave[k]) < uint64_t(p.pl_floats[k]) * 4u)
                        e.src = reinterpret_cast<const float*>(uint64_t(e.src) + uint64_t(p.pl_delta[k]) * 4u);
            }
            e.j_lo = uint16_t(lo - t0);
            e.j_cnt = uint16_t(hi - lo);
            // exact; the waveform path folds the 1/2 of the two-channel split, a plane holds X itself
            e.gain = (!SE && p.plane) ? sg.gain : 0.5f * sg.gain;
            d[n++] = e;
        }
    }
    if (n == 0) {   // nothing overlaps: one empty stage keeps the slot protocol uniform
        StageDesc e;
        e.src = nullptr; e.j_lo = 0; e.j_cnt = 0; e.gain = 0.f;
        d[n++] = e;
    }
    uint32_t tbits = 0;
    if (p.tmask != nullptr) {
        const int32_t* tm = tm_cache ? tm_cache : p.tmask + size_t(b) * p.n_tmask * 2;
        for (int i = 0; i < p.n_tmask; ++i) {
            const int size = tm[2 * i], off = tm[2 * i + 1];
            const int lo = max(off, t0), hi = min(off + size, t_end);
            if (lo < hi) tbits |= ((1u << (hi - lo)) - 1u) << (lo - t0);
        }
    }
    int4 hdr;
    hdr.x = n; hdr.y = b; hdr.z = t0 | (pair << 24); hdr.w = int(tbits);
    *reinterpret_cast<int4*>(blk) = hdr;
    if (p.fm_bits) {
        // mel epilogues that need bins below 128 only: the bins zeroed by the frequency masks and
        // stft_filter as a 128-bit map, so that a lane picks up its four bits with four shifts
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        auto zero_bins = [&](int off, int size) {
            for (int f = max(off, 0); f < min(off + size, 128); ++f) w[f >> 5] |= 1u << (f & 31);
        };
        if (p.fmask != nullptr) {
            const int32_t* fk = fm_cache ? fm_cache : p.fmask + size_t(b) * p.n_fmask * 2;
            for (int i = 0; i < p.n_fmask; ++i) zero_bins(fk[2 * i + 1], fk[2 * i]);
        }
        if (p.filter_k > 0) zero_bins(1, p.filter_k);
        *reinterpret_cast<uint4*>(blk + 16) = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
        int16_t fm[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) fm[i] = 0;
        if (p.fmask != nullptr) {
            const int32_t* fk = fm_cache ? fm_cache : p.fmask + size_t(b) * p.n_fmask * 2;
            for (int i = 0; i < p.n_fmask && i < 4; ++i) {
                fm[2 * i] = int16_t(fk[2 * i]);
                fm[2 * i + 1] = int16_t(fk[2 * i + 1]);
            }
        }
        *reinterpret_cast<int4*>(blk + 16) = *reinterpret_cast<const int4*>(fm);
    }
}

}  // namespace iris
