// Warp-level 512-point complex FFT: 32 lanes x 16 points, ONE shared-memory exchange.
//
//   n = n2 + 32*i        (lane = n2, register = i)          k = k1 + 16*k2
//   pass 1 (registers):  A[n2][k1] = sum_i x[n2 + 32 i] W16^(i k1)          (16-point FFT)
//   twiddle:             B[n2][k1] = A[n2][k1] * W512^(n2 k1)
//   exchange (shared):   row k1 holds B[.][k1] for all 32 n2
//   pass 2 (registers):  lane L = k1 + 16*p computes the outputs k2 = 2j + p of the 32-point
//                        FFT of its row by one radix-2 DIF step + a 16-point FFT:
//                          u[i] = (B[i] + s*B[i+16]) * (p ? W32^i : 1),  s = p ? -1 : +1
//                          Y[j] = sum_i u[i] W16^(i j) = X[k1 + 16*(2j + p)]
// Mirror bins: X[512-k] of lane (k1, p), register j sits in lane (16-k1, 1-p), register 15-j
// (k1 = 0: same lane; p = 0: register (16-j) & 15), so the split of a packed two-channel
// transform needs one register-indexed-at-compile-time shuffle per bin.
// For the log-mel features only bins < 128 are needed: j < 4 and the mirrors j >= 12, i.e.
// half of the outputs of pass 2 (the dead butterflies are eliminated at compile time).
//
// Everything here compiles for the host too; tests/host/fftwarp_host.cpp emulates the 32
// lanes and checks the index maps and the math against a float64 DFT.
#pragma once
#include "fftcore.cuh"

namespace iris {

// exchange buffer: 16 rows (k1) of 32 complex, row stride padded by 16 B so that the 16
// rows read by a warp's 128-bit loads fall into distinct 16-byte bank groups (2 wavefronts
// for 256 distinct bytes = conflict-free)
constexpr int kXwRowBytes = 32 * 8 + 16;          // 272
constexpr int kXwBytes = 16 * kXwRowBytes;        // 4352 per warp

IRIS_HD int xw_write_off(int k1, int n2) { return k1 * kXwRowBytes + n2 * 8; }        // float2
IRIS_HD int xw_read_off(int k1, int m) { return k1 * kXwRowBytes + m * 16; }          // float4 {B[2m], B[2m+1]}

// lane L = 2 * k1 + par: the two lanes that own the even / odd outputs of row k1 are adjacent.
// Both read the whole row in pass 2 (same 16-byte addresses): neighbouring lanes asking for the
// same address are served by one broadcast, so a 128-bit read of the warp touches 16 distinct
// 16-byte pieces (2 wavefronts) instead of 32 (4 wavefronts).  Row stride 272 B puts rows
// k1 = 0..7 into distinct 16-byte bank groups, so those two wavefronts are conflict-free.
IRIS_HD int warp_k1(int lane) { return lane >> 1; }
IRIS_HD int warp_par(int lane) { return lane & 1; }
IRIS_HD int warp_lane_of(int k1, int par) { return 2 * k1 + par; }
// bin held by register j of a lane after pass 2
IRIS_HD int warp_bin(int lane, int j) { return warp_k1(lane) + 16 * (2 * j + warp_par(lane)); }
// lane holding the mirror bins of this lane (k1 = 0: the lane itself)
IRIS_HD int warp_partner(int lane) {
    return warp_k1(lane) == 0 ? lane : warp_lane_of(16 - warp_k1(lane), 1 - warp_par(lane));
}
// register of the partner that holds the mirror of own register j
IRIS_HD int warp_mirror_reg(int lane, int j) { return (warp_k1(lane) == 0 && warp_par(lane) == 0) ? ((16 - j) & 15) : 15 - j; }

// pass 1 on the 16 registers of a lane, then the inter-pass twiddle v[k1] *= w^k1 with
// w = W512^n2.  Only the lane's base powers w^1, w^2, w^4, w^8 are loaded (2 x 16 bytes per
// lane and frame); the other eleven are products formed on the way (a complex multiply is two
// packed instructions, a 16-byte shared-memory load for every twiddle pair is four wavefronts
// of the shared-memory pipe, which is what bounds the kernel).  Products of at most four
// correctly rounded factors: relative error <= ~3e-7.
IRIS_HD void warp_pass1(cpx (&v)[16], cpx w1, cpx w2, cpx w4, cpx w8) {
    Fft<16>::run(v);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[4] = cmul(v[4], w4);
    v[8] = cmul(v[8], w8);
    {
        const cpx w3 = cmul(w1, w2);
        v[3] = cmul(v[3], w3);
        v[11] = cmul(v[11], cmul(w3, w8));
        const cpx w7 = cmul(w3, w4);
        v[7] = cmul(v[7], w7);
        v[15] = cmul(v[15], cmul(w7, w8));
    }
    {
        const cpx w5 = cmul(w1, w4);
        v[5] = cmul(v[5], w5);
        v[13] = cmul(v[13], cmul(w5, w8));
    }
    {
        const cpx w6 = cmul(w2, w4);
        v[6] = cmul(v[6], w6);
        v[14] = cmul(v[14], cmul(w6, w8));
    }
    v[9] = cmul(v[9], cmul(w1, w8));
    v[10] = cmul(v[10], cmul(w2, w8));
    v[12] = cmul(v[12], cmul(w4, w8));
}

// one DIF element of pass 2: u = (a + s*b) * (odd ? t : 1).  The odd half-warp multiplies by
// the compile-time twiddle t under a predicate (no selects); the even half keeps the sum.
IRIS_HD cpx warp_dif(cpx a, cpx b, float s, bool odd, float tx, float ty) {
    cpx d = caxpy(s, b, a);
    if (odd) d = cmul(d, cpx{tx, ty});
    return d;
}

// W32^(2m), W32^(2m+1) as (cos, sin) of -2 pi i / 32, handed to f as compile-time constants
// (the DIF twiddles t(i) of pass 2)
template <class F>
IRIS_HD void constexpr_for_pair(int m, F f) {
    switch (m) {   // m is a constant of an unrolled loop: the switch folds away
        case 0: f(1.f, 0.f, float(cx_cos2pi(1, 32)), -float(cx_sin2pi(1, 32))); break;
        case 1: f(float(cx_cos2pi(2, 32)), -float(cx_sin2pi(2, 32)), float(cx_cos2pi(3, 32)), -float(cx_sin2pi(3, 32))); break;
        case 2: f(float(cx_cos2pi(4, 32)), -float(cx_sin2pi(4, 32)), float(cx_cos2pi(5, 32)), -float(cx_sin2pi(5, 32))); break;
        case 3: f(float(cx_cos2pi(6, 32)), -float(cx_sin2pi(6, 32)), float(cx_cos2pi(7, 32)), -float(cx_sin2pi(7, 32))); break;
        case 4: f(float(cx_cos2pi(8, 32)), -float(cx_sin2pi(8, 32)), float(cx_cos2pi(9, 32)), -float(cx_sin2pi(9, 32))); break;
        case 5: f(float(cx_cos2pi(10, 32)), -float(cx_sin2pi(10, 32)), float(cx_cos2pi(11, 32)), -float(cx_sin2pi(11, 32))); break;
        case 6: f(float(cx_cos2pi(12, 32)), -float(cx_sin2pi(12, 32)), float(cx_cos2pi(13, 32)), -float(cx_sin2pi(13, 32))); break;
        default: f(float(cx_cos2pi(14, 32)), -float(cx_sin2pi(14, 32)), float(cx_cos2pi(15, 32)), -float(cx_sin2pi(15, 32))); break;
    }
}

}  // namespace iris
