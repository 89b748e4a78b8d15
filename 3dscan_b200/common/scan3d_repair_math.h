// scan3d_repair_math.h -- the rules of the non-manifold repair (scan3d_voxel_surface_repair, scan3d_mesh_repair_dev)
// that involve arithmetic: the face key and the per-edge keep rule of a non-manifold edge.  Written once for the CUDA
// kernels (scan3d_repair_kernels.cu) and for a host build of the very same expressions that the CPU tests compare
// with an independent numpy restatement (tests/test_repair_math_host.py compiles this header with
// g++ -ffp-contract=off).
//
//   face key     K(f) = (float_bits((float)area_f) << 32) | (2^32 - 1 - f), with area_f the hole filling's triangle
//                area (s3h::triangle: sqrt(l2) * 0.5 in double from the float corners in the face's order).  The area
//                is never negative, so its float bits order the keys by area, ties going to the smaller face index;
//                no two faces have the same key, and no key is 0 (f < 2^31), so 0 marks "no face".
//   edge rule    on an edge with more than 2 faces, f1 is the face of the largest key; f2 the face of the largest key
//                among the faces whose side on the edge runs opposite to f1's, or, when none runs opposite, among
//                the faces other than f1.  Every other face is dropped by the edge.  The kernels keep per edge the
//                largest key of each direction (m[0]: the side runs from the smaller vertex to the larger, m[1] the
//                other way) and the largest key other than f1 (second), all with 64-bit atomicMax.
//
// Decimation after a repair (scan3d_voxel_surface_decimate keeps its int64 quadric bound, s3q::sum_bound, per cell).
// A repair never adds a face and never moves a vertex: a split copy sits exactly on its source, in its source's cell.
// The faces at the copies of one cell are a subset of the faces the cell had before, so every per-cell count the
// decimation's bound and the fill's extension of it (s3h::nets_sum_bound) rest on can only fall, and a surface that was
// decimatable before a repair is decimatable after it.
// The fill's extension assumes one hole per cell over the life of the surface.  After a repair that dropped a face or
// split a vertex that no longer holds: each copy of a cell (up to 24, one per face) can sit on a hole of its own, and a
// dropped face can open a cell whose hole was filled before.  Two holes of 22 edges on one cell already exceed 2^63
// (2^63.85 at r = 256, checked below), and a sequence of fills and repairs can reopen a cell any number of times, so
// no cap on max_edges keeps the bound.  The state rule instead: a fill of the held surface after such a repair makes
// the decimation refuse the surface until the next extraction.
#pragma once
#include "scan3d_fill_math.h"

#if !defined(__CUDA_ARCH__)
#include <string.h>
#endif

namespace s3r {

// the cluster sum bound of the decimation with `holes` holes of N edges on every cell, for r = m in [1, 256]
constexpr double holes_sum_bound(int m, int N, int holes)
{
    const double c = m + 3.0;
    return c * c * c * (s3q::FACES_PER_VERTEX * (3.0 * s3q::AREA_MAX_S2 / ((double)m * m) * s3q::SCALE + 0.5) +
                        holes * (N - 2) * s3h::fill_face_bound(m, N));
}
constexpr bool holes_bound_holds(int N, int holes)
{
    for (int m = 1; m <= (int)s3q::RATIO_MAX; m++)
        if (!(holes_sum_bound(m, N, holes) < 9223372036854775808.0)) return false;
    return true;
}
static_assert(holes_bound_holds(s3h::NETS_MAX_EDGES, 1), "one hole per cell: the fill's own bound");
static_assert(!holes_bound_holds(s3h::NETS_MAX_EDGES, 2),
              "two holes of a cell after a repair break the bound: a fill after a repair must stop the decimation");

S3A_HD unsigned int float_bits(float x)
{
#if defined(__CUDA_ARCH__)
    return __float_as_uint(x);
#else
    unsigned int u;
    memcpy(&u, &x, sizeof(u));
    return u;
#endif
}

// K(f) of face f with the float corners a, b, c
S3A_HD unsigned long long face_key(const float a[3], const float b[3], const float c[3], unsigned int f)
{
    double u[3], area;
    s3h::triangle(a, b, c, u, &area);
    return (unsigned long long)float_bits(S3V_D2F(area)) << 32 | (unsigned long long)(0xffffffffu - f);
}

// whether the face of key k, on an edge with more than 2 faces, is kept by that edge: m0 / m1 the largest keys of the
// two directions (0 = none), second the largest key other than the edge's largest
S3A_HD bool kept_on_edge(unsigned long long k, unsigned long long m0, unsigned long long m1, unsigned long long second)
{
    const unsigned long long f1 = m0 > m1 ? m0 : m1;
    const unsigned long long opposite = m0 > m1 ? m1 : m0;
    const unsigned long long f2 = opposite != 0 ? opposite : second;
    return k == f1 || k == f2;
}

}  // namespace s3r
