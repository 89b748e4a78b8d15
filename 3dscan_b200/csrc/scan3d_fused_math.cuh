// scan3d_fused_math.cuh -- the register-level arithmetic of the fused kernels: SWAR integer decode of
// 4 pixels per 32-bit word (phase-shift terms, Gray threshold, Gray->binary, fringe order) and the
// conversion of those terms into the wrapped phase.  Pure functions of their arguments (no shared
// memory, no PTX), so the very same source also compiles for the host: tests/fused_math_host.cpp
// runs it on whole scans against the oracle and the reference's golden images without a GPU.
#pragma once
#include <stdint.h>

#include "scan3d_math.cuh"

namespace s3d {

// ---- SWAR pieces -----------------------------------------------------------------------------
// per-byte unsigned a >= b  ->  bit 7 of each byte (the other bits are NOT cleared: callers mask)
__device__ __forceinline__ uint32_t ge_bytes_raw(uint32_t a, uint32_t b)
{
    const uint32_t d = (a | 0x80808080u) - (b & 0x7f7f7f7fu);
    return (a & ~b) | (~(a ^ b) & d);
}
// bytes (b0,b1,b2,b3) -> 16-bit lanes (b0,b1) and (b2,b3)
__device__ __forceinline__ uint32_t lanes_lo(uint32_t w) { return __byte_perm(w, 0, 0x4140); }
__device__ __forceinline__ uint32_t lanes_hi(uint32_t w) { return __byte_perm(w, 0, 0x4342); }

struct Terms {            // up to 4 biased 16-bit terms for 4 pixels: [term][0]=(px0,px1) [1]=(px2,px3)
    uint32_t t[4][2];
};
// phase-shift numerators/denominators for 4 pixels (3/wrapped_phase.cpp:171-173,195-196,217-218)
template <int N>
__device__ __forceinline__ void fringe_terms(const uint32_t* __restrict__ sw, int f0, int wpf, int tid, Terms& T)
{
    uint32_t L[N][2];
#pragma unroll
    for (int k = 0; k < N; k++) {
        const uint32_t w = sw[(f0 + k) * wpf + tid];
        L[k][0] = lanes_lo(w);
        L[k][1] = lanes_hi(w);
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
        if (N == 3) {          // t1 = I0 - I2 (+512) ; t2 = 2*I1 - I0 - I2 (+1024)
            T.t[0][h] = L[0][h] + 0x02000200u - L[2][h];
            T.t[1][h] = 2 * L[1][h] + 0x04000400u - L[0][h] - L[2][h];
        } else if (N == 4) {   // t1 = I3 - I1 ; t2 = I0 - I2
            T.t[0][h] = L[3 % N][h] + 0x02000200u - L[1][h];
            T.t[1][h] = L[0][h] + 0x02000200u - L[2][h];
        } else if (N == 5) {   // t1 = 2(I1 - I3) (+1024) ; t2 = 2*I2 - I0 - I4 (+1024)
            T.t[0][h] = 2 * L[1][h] + 0x04000400u - 2 * L[3 % N][h];
            T.t[1][h] = 2 * L[2][h] + 0x04000400u - L[0][h] - L[4 % N][h];
        } else {               // N == 8: a1 = I6-I2, b1 = I5+I7-I1-I3, a2 = I0-I4, b2 = I1+I7-I3-I5
            T.t[0][h] = L[6 % N][h] + 0x02000200u - L[2][h];
            T.t[1][h] = L[5 % N][h] + L[7 % N][h] + 0x04000400u - L[1][h] - L[3 % N][h];
            T.t[2][h] = L[0][h] + 0x02000200u - L[4 % N][h];
            T.t[3][h] = L[1][h] + L[7 % N][h] + 0x04000400u - L[3 % N][h] - L[5 % N][h];
        }
    }
}

// Gray -> binary (B0 = G0, Bi = B(i-1) xor Gi, 4/phase_unwrap.cpp:187-191) for the 4 pixels at
// once: a prefix xor inside every byte (plane i sits at bit 7 - i%8), then the parity of planes
// 0..7 (bit 0 of the first accumulator) carried into every bit of the second one.
__device__ __forceinline__ void gray_to_binary(uint32_t& accA, uint32_t& accB)
{
    accA ^= (accA >> 1) & 0x7f7f7f7fu;
    accA ^= (accA >> 2) & 0x3f3f3f3fu;
    accA ^= (accA >> 4) & 0x0f0f0f0fu;
    accB ^= (accB >> 1) & 0x7f7f7f7fu;
    accB ^= (accB >> 2) & 0x3f3f3f3fu;
    accB ^= (accB >> 4) & 0x0f0f0f0fu;
    accB ^= (accA & 0x01010101u) * 0xffu;
}
// Gray threshold for 4 pixels, all M planes: byte accumulators with plane i at bit (7 - i%8)
// (4/phase_unwrap.cpp:183: (uchar)img - (uchar)inv >= 0, tie -> 1)
__device__ __forceinline__ void gray_bits(const uint32_t* __restrict__ sw, int g0, int i0, int M, int wpf, int tid,
                                          uint32_t& accA, uint32_t& accB)
{
    accA = 0; accB = 0;
    // shift first, then mask and merge in one 3-input logic op: acc | ((ge >> i) & (0x80808080 >> i))
    // Guards on M are warp-uniform branches and cost issue slots: the planes go in pairs (one test per pair), and the
    // first pair that reaches past M ends the chain -- no test for the planes after it (a guard per plane: +2.2 % kernel time).
    auto plane = [&](int i) {
        const uint32_t ge = ge_bytes_raw(sw[(g0 + i) * wpf + tid], sw[(i0 + i) * wpf + tid]);
        if (i < 8) accA |= (ge >> i) & (0x80808080u >> i);
        else accB |= (ge >> (i - 8)) & (0x80808080u >> (i - 8));
    };
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
        if (i + 1 < M) {
            plane(i);
            if (i + 1 < 15) plane(i + 1);
        } else {
            if (i < M && i < 15) plane(i);
            break;
        }
    }
    gray_to_binary(accA, accB);
}
// fringe order of pixel j from the binary accumulators: code = sum Bi << (M-1-i)  (:193)
__device__ __forceinline__ int code_of(uint32_t binA, uint32_t binB, int j, int M)
{
    const uint32_t a = (binA >> (8 * j)) & 0xffu, b = (binB >> (8 * j)) & 0xffu;
    return (int)(((a << 8) | b) >> (16 - M));
}

// biased 16-bit lane -> exact double without the conversion pipe: the lane value u (< 2^16) is
// dropped into the mantissa of 2^52 and (2^52 + bias) is subtracted
__device__ __forceinline__ double lane_f64(uint32_t u, int bias)
{
    return __hiloint2double(0x43300000, (int)u) - (bias == 512 ? K_2P52_512 : K_2P52_1024);
}

// The pair of pixels (2h, 2h + 1) of a thread shares its term registers: selecting them once per pair (by h, which
// is a run-time value in the rolled pass loop) leaves only compile-time lane extractions per pixel.
struct TermsPair {
    uint32_t r[4];      // T.t[k][h]
};
__device__ __forceinline__ TermsPair terms_pair(const Terms& T, int h)
{
    TermsPair P;
#pragma unroll
    for (int k = 0; k < 4; k++) P.r[k] = h ? T.t[k][1] : T.t[k][0];
    return P;
}

// wrapped phase of pixel u (0 / 1, compile time) of a pair
template <int N>
__device__ __forceinline__ float phase_of_pair(const TermsPair& P, int u, const double* tab)
{
    auto lane = [&](int k) { return u ? (P.r[k] >> 16) : (P.r[k] & 0xffffu); };
    if (N == 8) {
        const double a1 = lane_f64(lane(0), 512), b1 = lane_f64(lane(1), 1024);
        const double a2 = lane_f64(lane(2), 512), b2 = lane_f64(lane(3), 1024);
        const double d1 = dadd(a1, dmul(b1, K_SQRT_HALF));
        const double d2 = dadd(a2, dmul(b2, K_SQRT_HALF));
        return atan2_to_float(d1, d2, 0.0f, 0.0f, tab);
    } else {
        const int t1 = (int)lane(0) - (N == 5 ? 1024 : 512);
        const int t2 = (int)lane(1) - (N == 4 ? 512 : 1024);
        if (N == 5) return atan2f_fdlibm((float)t1, (float)t2);   // 3/wrapped_phase.cpp:220 (float atan2f)
        // exact int -> double without the conversion pipe (|t| < 2^11)
        return atan2_to_float(lane_f64(lane(0), N == 5 ? 1024 : 512), lane_f64(lane(1), N == 4 ? 512 : 1024), 0.0f, 0.0f, tab);
    }
}

// fringe order of pixel u (0 / 1, compile time) of a pair whose accumulators have been shifted down by 16 * h
__device__ __forceinline__ int code_of_pair(uint32_t binA_h, uint32_t binB_h, int u, int M)
{
    const uint32_t a = (binA_h >> (8 * u)) & 0xffu, b = (binB_h >> (8 * u)) & 0xffu;
    return (int)(((a << 8) | b) >> (16 - M));
}

}  // namespace s3d
