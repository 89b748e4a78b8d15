// scan3d_orient_math.h -- the arithmetic of the coherent orientation and the measures of a triangle mesh
// (scan3d_voxel_surface_orient, scan3d_mesh_orient_dev, scan3d_voxel_surface_measure, scan3d_mesh_measure_dev): the
// centre, the per-face fixed-point volume and area terms and their exact int128 sum.  Written once for the CUDA kernels
// (scan3d_orient_kernels.cu) and for a host build of the very same expressions that the CPU tests compare with an
// independent numpy restatement (tests/test_orient_math_host.py compiles this header with g++ -ffp-contract=off).
//
// Every double operation below is one correctly rounded IEEE operation (S3A_*), in this order, no FMA:
//
//   centre       c_k = (float)(((double)lo_k + (double)hi_k) * 0.5), lo / hi the exact float bounding box of the
//                referenced vertices (the vertices of the faces that are not degenerate)
//   exponent     over every referenced vertex and axis, F = the largest biased exponent field ((bits >> 52) & 0x7ff) of
//                the double d = (double)p_k - (double)c_k; E = max(F - 1022, E_MIN), so |d| < 2^E everywhere.  A
//                non-zero d is at least 2^-149 (both floats are multiples of 2^-149), so the clamp only acts when every
//                d is zero; |d| < 2^129 bounds E above.
//   volume term  a = p_a - c, b = p_b - c, q = p_c - c per axis in double; x = (b_y q_z - b_z q_y, b_z q_x - b_x q_z,
//                b_x q_y - b_y q_x); D = (a_x x_x + a_y x_y) + a_z x_z, six times the signed volume of the tetrahedron
//                (c, p_a, p_b, p_c); the term is rint(D * 2^(P - 3E)), half to even.
//   area term    area = s3h::triangle's sqrt(l2) * 0.5 (the hole filling's area, from the float corners in the face's
//                order); the term is rint(area * 2^(P - 2E)).
//   sums         each sum of terms is exact in int128 (two's complement, held as two uint64 words).  The volume is
//                ldexp((double)sum D, 3E - P) / 6 and the area ldexp((double)sum area, 2E - P).  The / 6 comes after
//                the sum, so a mesh whose D are exact (a cube with representable corners) has an exact volume.
//
// Bounds (P = 59).  Every |d| < 2^E, so each product of the cross product is below 2^2E and each of its components
// below 2 * 2^2E; D is then below 3 * 2^E * 2 * 2^2E = 6 * 2^3E, plus a few ulps: below 2^(3E + 3), and the volume term
// below 2^(P + 3) = 2^62.  A side of a face is below 2^(E + 1) per axis, so each component of the area's cross
// product is below 2^(2E + 3), l2 below 3 * 2^(4E + 6), and the area below sqrt(3) * 2^(2E + 2) < 2^(2E + 3): the area
// term is below 2^62 as well.  A mesh has fewer than 2^31 faces, so every sum is below 2^93 in magnitude, far inside
// int128.  The powers of two 2^(P - 3E) and 2^(P - 2E) lie in [2^-328, 2^506] for E in [E_MIN, 129], inside the
// double range, so the scaling is exact and only rint rounds.
//
// Decimation after an orientation (scan3d_voxel_surface_decimate keeps its int64 quadric bound, s3q::sum_bound).  A
// flip (a, b, c) -> (a, c, b) negates the face's cross product n, so u -> -u and e = u . f -> -e, while the ten
// quadric coefficients (u_i u_j, u_i e, e e) and the weight w = |n| / 2 / H^2 do not change.  The per-cell face counts
// and positions do not change either, so an oriented surface is exactly as decimatable as before.  The fill after an
// orientation is another matter: a flip can make a vertex regular, so a fill can close a hole it left open before; the
// one-hole-per-cell argument of the fill's bound is not shown to survive, so an orientation that flipped a face counts
// as a repair (common/scan3d_repair_math.h): a fill after it stops the decimation until the next extraction.
#pragma once
#include "scan3d_aux_math.h"
#include "scan3d_fill_math.h"
#include "scan3d_smooth_math.h"
#include "scan3d_voxel_math.h"

#include <math.h>
#include <string.h>

#if defined(__CUDA_ARCH__)
#define S3O_DBITS(x) (unsigned long long)__double_as_longlong(x)
#else
#define S3O_DBITS(x) s3o::double_bits(x)
#endif

namespace s3o {

constexpr int P = 59;                                       // fixed-point bits below 2^3E (volume) and 2^2E (area)
constexpr int E_MIN = -149;
constexpr int E_MAX = 129;
constexpr int MAX_FACES_LOG2 = 31;                          // fewer than 2^31 faces
static_assert(P + 3 <= 62, "a term stays below 2^62, so it is an int64");
static_assert(MAX_FACES_LOG2 + P + 3 < 127, "2^31 terms of magnitude below 2^62 cannot overflow int128");
static_assert(P - 3 * E_MAX >= -1022 && P - 3 * E_MIN <= 1023, "the scales are normal doubles");
static_assert(P - 2 * E_MAX >= -1022 && P - 2 * E_MIN <= 1023, "the scales are normal doubles");

#if !defined(__CUDA_ARCH__)
inline unsigned long long double_bits(double x)
{
    unsigned long long u;
    memcpy(&u, &x, 8);
    return u;
}
#endif

// the order-preserving key of a float's bits (a larger float has a larger key; -0 below +0), and back
S3A_HD unsigned int order_key(unsigned int bits) { return (bits & 0x80000000u) ? ~bits : bits | 0x80000000u; }
S3A_HD unsigned int key_bits(unsigned int key) { return (key & 0x80000000u) ? key & 0x7fffffffu : ~key; }

// one axis of the centre from the bounding box's float bits
S3A_HD float centre(float lo, float hi) { return S3V_D2F(S3A_MUL(S3A_ADD((double)lo, (double)hi), 0.5)); }

// the biased double exponent field of x - c; its max over the referenced vertices gives E
S3A_HD unsigned int offset_field(float x, float c)
{
    return (unsigned int)((S3O_DBITS(S3A_SUB((double)x, (double)c)) >> 52) & 0x7ffu);
}
S3A_HD int exponent(unsigned int max_field)
{
    const int e = (int)max_field - 1022;
    return e < E_MIN ? E_MIN : e;
}

// the volume term of the face (a, b, q) about the centre c
S3A_HD long long volume_term(const float pa[3], const float pb[3], const float pq[3], const float c[3], int E)
{
    double a[3], b[3], q[3];
    for (int k = 0; k < 3; k++) {
        a[k] = S3A_SUB((double)pa[k], (double)c[k]);
        b[k] = S3A_SUB((double)pb[k], (double)c[k]);
        q[k] = S3A_SUB((double)pq[k], (double)c[k]);
    }
    const double x[3] = {S3A_SUB(S3A_MUL(b[1], q[2]), S3A_MUL(b[2], q[1])),
                         S3A_SUB(S3A_MUL(b[2], q[0]), S3A_MUL(b[0], q[2])),
                         S3A_SUB(S3A_MUL(b[0], q[1]), S3A_MUL(b[1], q[0]))};
    const double D = S3A_ADD(S3A_ADD(S3A_MUL(a[0], x[0]), S3A_MUL(a[1], x[1])), S3A_MUL(a[2], x[2]));
    return S3V_D2LL_RN(S3A_MUL(D, S3T_POW2(P - 3 * E)));
}

// the area term of the face (a, b, q)
S3A_HD long long area_term(const float pa[3], const float pb[3], const float pq[3], int E)
{
    double u[3], area;
    s3h::triangle(pa, pb, pq, u, &area);
    return S3V_D2LL_RN(S3A_MUL(area, S3T_POW2(P - 2 * E)));
}

// (lo, hi) += t, two's complement int128
S3A_HD void add128(unsigned long long* lo, unsigned long long* hi, long long t)
{
    const unsigned long long u = (unsigned long long)t;
    *lo += u;
    *hi += (t < 0 ? ~0ull : 0ull) + (*lo < u ? 1ull : 0ull);
}

// the sign of an int128: -1, 0 or +1
S3A_HD int sign128(unsigned long long lo, unsigned long long hi)
{
    if ((long long)hi < 0) return -1;
    return (hi | lo) ? 1 : 0;
}

// ldexp of the int128 (lo, hi), correctly rounded to double before the scaling (host code)
inline double scaled(unsigned long long lo, unsigned long long hi, int e)
{
    const __int128 v = (__int128)(((unsigned __int128)hi << 64) | lo);
    return ldexp((double)v, e);
}
inline double volume(unsigned long long lo, unsigned long long hi, int E) { return scaled(lo, hi, 3 * E - P) / 6.0; }
inline double area(unsigned long long lo, unsigned long long hi, int E) { return scaled(lo, hi, 2 * E - P); }

}  // namespace s3o
