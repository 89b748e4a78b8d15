// scan3d_voxel_math.h -- per-point and per-voxel arithmetic of the voxel-grid merge (scan3d_voxel_*), written once
// for the CUDA kernels (scan3d_voxel_kernels.cu) and for a host build of the very same expressions that the CPU tests
// compare with an independent numpy restatement (tests/test_voxel_math_host.py compiles this header with
// g++ -ffp-contract=off).
//
// The sums of a voxel are integers, so the order in which points are added (atomics, warps, adds) cannot change
// them: the merge is bit-reproducible without a sort.  s = voxel_size, S = (double)s, Q = 2^24.
//
//   per point and axis: t = (double)x / S, i = floor(t), f = t - i, q = min((uint64)floor(f Q), Q - 1)
//       (the clamp: for x = -1e-30, t + 1 rounds to 1.0, so floor(f Q) would be Q)
//   dropped: a coordinate not finite, or some i outside [-2^20, 2^20)
//   normal: (0, 0, 0) if a component is not finite, else m = (int64) rint((double)clamp(c, -1, 1) Q), half to even
//   per voxel of n points: coordinate (float)(((double)i + (double)sum q / (Q (double)n)) S);
//       normal X, Y, Z = (double)sum m, l2 = (X X + Y Y) + Z Z, (0, 0, 0) if l2 == 0 else (float)(X / sqrt(l2));
//       colour (sum c + n / 2) / n (integer division); count n.
// Every double operation is one correctly rounded IEEE operation, in this order, no FMA.
#pragma once
#include "scan3d_aux_math.h"

#if defined(__CUDA_ARCH__)
#define S3V_ULL2D(a) __ull2double_rn(a)
#define S3V_LL2D(a) __ll2double_rn(a)
#define S3V_D2LL_RN(a) __double2ll_rn(a)
#define S3V_D2F(a) __double2float_rn(a)
#define S3V_SQRT(a) __dsqrt_rn(a)
#else  // host translation units are built with -ffp-contract=off; the default rounding mode is to nearest
#define S3V_ULL2D(a) ((double)(unsigned long long)(a))
#define S3V_LL2D(a) ((double)(long long)(a))
#define S3V_D2LL_RN(a) ((long long)rint(a))
#define S3V_D2F(a) ((float)(a))
#define S3V_SQRT(a) sqrt((double)(a))
#endif

namespace s3v {

constexpr double Q = 16777216.0;                            // 2^24 fixed-point steps per voxel edge / unit normal
constexpr unsigned long long QMAX = 16777215ull;            // Q - 1
constexpr int KEY_BITS = 21;                                // per axis: i + 2^20 in [0, 2^21)
constexpr long long I_MIN = -(1ll << 20), I_MAX = 1ll << 20; // i in [I_MIN, I_MAX)
constexpr unsigned long long EMPTY_KEY = ~0ull;             // no key packs to it (bit 63 is always 0)

// one axis: *i = floor(x / S), *q = the position inside the voxel in Q steps; false = the point is dropped
S3A_HD bool axis(float x, double S, long long* i, unsigned long long* q)
{
    if (!(x - x == 0.0f)) return false;                     // NaN or +-inf
    const double t = S3A_DIV((double)x, S);
    const double fi = floor(t);
    if (!(fi >= (double)I_MIN && fi < (double)I_MAX)) return false;
    const double f = S3A_SUB(t, fi);
    const unsigned long long qq = (unsigned long long)floor(S3A_MUL(f, Q));   // f Q is exact, in [0, Q]
    *i = (long long)fi;
    *q = qq < QMAX ? qq : QMAX;
    return true;
}

// the 63-bit key of a voxel
S3A_HD unsigned long long pack_key(long long ix, long long iy, long long iz)
{
    return ((unsigned long long)(ix - I_MIN) << (2 * KEY_BITS)) | ((unsigned long long)(iy - I_MIN) << KEY_BITS) |
           (unsigned long long)(iz - I_MIN);
}
S3A_HD long long key_axis(unsigned long long key, int a)   // a = 0 (x), 1 (y), 2 (z)
{
    return (long long)((key >> (KEY_BITS * (2 - a))) & ((1ull << KEY_BITS) - 1)) + I_MIN;
}

// the voxel of (x, y, z) and the point's position inside it; false = dropped
S3A_HD bool point_key(float x, float y, float z, double S, unsigned long long* key, unsigned long long q[3])
{
    long long ix, iy, iz;
    if (!axis(x, S, &ix, &q[0]) || !axis(y, S, &iy, &q[1]) || !axis(z, S, &iz, &q[2])) return false;
    *key = pack_key(ix, iy, iz);
    return true;
}

// fixed-point normal: (0, 0, 0) if any component is not finite, else each component clamped to [-1, 1] in Q steps
S3A_HD void normal_fixed(float nx, float ny, float nz, long long m[3])
{
    if (!(nx - nx == 0.0f && ny - ny == 0.0f && nz - nz == 0.0f)) {
        m[0] = m[1] = m[2] = 0;
        return;
    }
    const float c[3] = {nx, ny, nz};
    for (int k = 0; k < 3; k++) {
        const float v = c[k] < -1.0f ? -1.0f : (c[k] > 1.0f ? 1.0f : c[k]);
        m[k] = S3V_D2LL_RN(S3A_MUL((double)v, Q));
    }
}

// the merged coordinate of axis a of a voxel with n points and position sum sq
S3A_HD float coord(unsigned long long key, int a, unsigned long long sq, unsigned int n, double S)
{
    const double den = S3A_MUL(Q, (double)n);
    const double v = S3A_ADD((double)key_axis(key, a), S3A_DIV(S3V_ULL2D(sq), den));
    return S3V_D2F(S3A_MUL(v, S));
}

// the merged normal from the fixed-point sums
S3A_HD void normal_out(long long sx, long long sy, long long sz, float out[3])
{
    const double X = S3V_LL2D(sx), Y = S3V_LL2D(sy), Z = S3V_LL2D(sz);
    const double l2 = S3A_ADD(S3A_ADD(S3A_MUL(X, X), S3A_MUL(Y, Y)), S3A_MUL(Z, Z));
    if (l2 == 0.0) {
        out[0] = out[1] = out[2] = 0.0f;
        return;
    }
    const double l = S3V_SQRT(l2);
    out[0] = S3V_D2F(S3A_DIV(X, l));
    out[1] = S3V_D2F(S3A_DIV(Y, l));
    out[2] = S3V_D2F(S3A_DIV(Z, l));
}

// the merged colour channel: the mean rounded half up
S3A_HD unsigned char colour(unsigned long long sc, unsigned int n)
{
    return (unsigned char)((sc + n / 2) / n);
}

}  // namespace s3v
