// scan3d_smooth_math.h -- the arithmetic of the surface smoothing (scan3d_voxel_surface_smooth, scan3d_mesh_smooth_dev):
// Taubin lambda|mu fairing with the uniform umbrella operator (Taubin 1995) on fixed-point positions.  Written once for
// the CUDA kernels (scan3d_smooth_kernels.cu) and for a host build of the very same expressions that the CPU tests
// compare with an independent numpy restatement (tests/test_smooth_math_host.py compiles this header with
// g++ -ffp-contract=off).
//
// Every double operation below is one correctly rounded IEEE operation (S3A_*), in this order, no FMA:
//
//   exponent     F = the largest biased exponent field ((bits >> 23) & 0xff) over every coordinate of the mesh, an exact
//                integer max; E = F - 126, so 2^E is the smallest power of two above every |coordinate| (F = 0, all
//                coordinates zero or subnormal, gives E = -126).  E is in [-126, 128] for finite input.
//   fixed point  Q = rint((double)x * 2^(P - E)), half to even, P = 40.  The product is exact (a power-of-two scale
//                that neither overflows nor underflows a double), so only rint rounds, and it is exact wherever
//                |x| >= 2^(E - 17) (a float's 24 significant bits then lie above 2^(E - P)).  |Q| < 2^40.
//   pass         for a free vertex with d >= 1 distinct neighbours w, per axis S = sum Q_w (an exact int64 sum, so the
//                order of the neighbours is irrelevant), m = (double)S / (double)d, Q' = Q + rint(k * (m - (double)Q))
//                with k = (double)lambda or (double)mu.  Held and isolated vertices keep Q.
//   output       a free vertex's coordinate is (float)((double)Q * 2^(E - P)) (the product is exact).
//   displacement (double)x' - (double)x per axis, sqrt((dx dx + dy dy) + dz dz).
//   face normal  for a face of three distinct vertices, d1 = p_b - p_a, d2 = p_c - p_a (double), n = (d1y d2z - d1z d2y,
//                d1z d2x - d1x d2z, d1x d2y - d1y d2x), l2 = (nx nx + ny ny) + nz nz; l2 == 0 or not finite: nothing;
//                else the float unit normal (float)(n_a / sqrt(l2)) in the merge's fixed point (s3v::normal_fixed: clamped
//                to [-1, 1], rint(v * 2^24)) is added to each of the three vertices.
//   normal       s3v::normal_out of the vertex's sums; a vertex whose sums are all zero keeps its normal.
//
// Overflow bound of the int64 sums (checked by the host test).  The input has |Q| < 2^40.  A lambda pass moves Q
// towards the mean of values no larger, but a mu pass moves it away (by up to |mu| (|m| + |Q|)), so the smoothing
// checks every free vertex after every pass: |Q'| <= Q_LIMIT = 2^42 on every axis, and d <= DEGREE_LIMIT = 2^20
// (checked once).  Then |S| <= DEGREE_LIMIT * Q_LIMIT = 2^62 < 2^63 in every pass that reads only checked values, and
// |Q'| <= |Q| + |m| + |Q| + 1 < 2^44 cannot overflow.  A vertex over either limit, or a free vertex whose output
// coordinate rounds to +-inf (possible only for E >= 126), fails the whole call.  The normal sums add at most one
// |m_a| <= 2^24 per face of the vertex, and there are fewer than 2^31 faces, so they stay below 2^55.
#pragma once
#include <string.h>

#include "scan3d_aux_math.h"
#include "scan3d_voxel_math.h"

#if defined(__CUDA_ARCH__)
#define S3T_FBITS(x) __float_as_uint(x)
#define S3T_POW2(e) __longlong_as_double((long long)(1023 + (e)) << 52)
#else
#define S3T_FBITS(x) s3t::float_bits(x)
#define S3T_POW2(e) ldexp(1.0, (e))
#endif

namespace s3t {

constexpr int P = 40;                                       // fixed-point bits below 2^E
constexpr long long Q_LIMIT = 1ll << 42;                    // |Q| of a free vertex after every pass
constexpr unsigned int DEGREE_LIMIT = 1u << 20;             // distinct neighbours of a free vertex
constexpr int E_MIN = -126;                                 // E of an all-zero or subnormal mesh

#if !defined(__CUDA_ARCH__)
inline unsigned int float_bits(float x)
{
    unsigned int u;
    memcpy(&u, &x, 4);
    return u;
}
#endif

// the biased exponent field of x; its max over the mesh gives E
S3A_HD unsigned int exponent_field(float x) { return (S3T_FBITS(x) >> 23) & 0xffu; }
S3A_HD int exponent(unsigned int max_field) { return (int)max_field - 126; }

// x in the fixed point of exponent E
S3A_HD long long quantise(float x, int E) { return S3V_D2LL_RN(S3A_MUL((double)x, S3T_POW2(P - E))); }

// a fixed-point coordinate as the output float
S3A_HD float dequantise(long long q, int E) { return S3V_D2F(S3A_MUL(S3V_LL2D(q), S3T_POW2(E - P))); }

// one axis of one pass: Q' from Q, the neighbours' sum S over d >= 1 of them and k = lambda or mu
S3A_HD long long update(long long q, long long s, unsigned int d, double k)
{
    const double m = S3A_DIV(S3V_LL2D(s), (double)d);
    return q + S3V_D2LL_RN(S3A_MUL(k, S3A_SUB(m, S3V_LL2D(q))));
}

S3A_HD bool over_limit(long long q) { return q > Q_LIMIT || q < -Q_LIMIT; }

// the Euclidean distance between a vertex's old and new float positions
S3A_HD double displacement(const float a[3], const float b[3])
{
    const double dx = S3A_SUB((double)b[0], (double)a[0]), dy = S3A_SUB((double)b[1], (double)a[1]),
                 dz = S3A_SUB((double)b[2], (double)a[2]);
    return S3V_SQRT(S3A_ADD(S3A_ADD(S3A_MUL(dx, dx), S3A_MUL(dy, dy)), S3A_MUL(dz, dz)));
}

// the fixed-point unit normal of face (a, b, c); false when it adds nothing (l2 zero or not finite)
S3A_HD bool face_normal(const float a[3], const float b[3], const float c[3], long long m[3])
{
    double d1[3], d2[3];
    for (int k = 0; k < 3; k++) {
        d1[k] = S3A_SUB((double)b[k], (double)a[k]);
        d2[k] = S3A_SUB((double)c[k], (double)a[k]);
    }
    const double n[3] = {S3A_SUB(S3A_MUL(d1[1], d2[2]), S3A_MUL(d1[2], d2[1])),
                         S3A_SUB(S3A_MUL(d1[2], d2[0]), S3A_MUL(d1[0], d2[2])),
                         S3A_SUB(S3A_MUL(d1[0], d2[1]), S3A_MUL(d1[1], d2[0]))};
    const double l2 = S3A_ADD(S3A_ADD(S3A_MUL(n[0], n[0]), S3A_MUL(n[1], n[1])), S3A_MUL(n[2], n[2]));
    if (!(l2 > 0.0 && l2 - l2 == 0.0)) return false;
    const double l = S3V_SQRT(l2);
    s3v::normal_fixed(S3V_D2F(S3A_DIV(n[0], l)), S3V_D2F(S3A_DIV(n[1], l)), S3V_D2F(S3A_DIV(n[2], l)), m);
    return true;
}

}  // namespace s3t
