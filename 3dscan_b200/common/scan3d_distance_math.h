// scan3d_distance_math.h -- the arithmetic of the sample-to-surface distances (scan3d_voxel_surface_distance,
// scan3d_voxel_surface_distance_dev, scan3d_mesh_distance_dev): the exact nearest face of a triangle mesh within R of a
// sample, signed by the face normal, in the manner of Metro (Cignoni, Rocchini & Scopigno 1998) and MeshLab's Hausdorff
// Distance filter.  Written once for the CUDA kernels (scan3d_distance_kernels.cu) and for a host build of the very same
// expressions that the CPU tests compare with an independent numpy restatement (tests/test_distance_math_host.py
// compiles this header with g++ -ffp-contract=off).
//
// p is a sample (float coordinates as doubles), (a, b, c) a face (float corners as doubles).  Every double operation
// below is one correctly rounded IEEE operation (S3A_*), in this order, no FMA; v . w = (vx wx + vy wy) + vz wz:
//
//   normal       ab = b - a, ac = c - a, N = ab x ac = (ab_y ac_z - ab_z ac_y, ab_z ac_x - ab_x ac_z,
//                ab_x ac_y - ab_y ac_x), l2 = N . N: the hole filling's triangle terms (s3h::triangle)
//   closest      q = Ericson's ClosestPtPointTriangle (Real-Time Collision Detection, 5.1.5) with his region tests in
//                his order, ap = p - a, bp = p - b, cp = p - c:
//                  d1 = ab . ap, d2 = ac . ap;           d1 <= 0 && d2 <= 0:                   q = a
//                  d3 = ab . bp, d4 = ac . bp;           d3 >= 0 && d4 <= d3:                  q = b
//                  vc = d1 d4 - d3 d2;                   vc <= 0 && d1 >= 0 && d3 <= 0:        q = a + (d1 / (d1 - d3)) ab
//                  d5 = ab . cp, d6 = ac . cp;           d6 >= 0 && d5 <= d6:                  q = c
//                  vb = d5 d2 - d1 d6;                   vb <= 0 && d2 >= 0 && d6 <= 0:        q = a + (d2 / (d2 - d6)) ac
//                  va = d3 d6 - d5 d4, e = d4 - d3, g = d5 - d6;
//                                                        va <= 0 && e >= 0 && g >= 0:          q = b + (e / (e + g)) (c - b)
//                  otherwise, inv = 1 / ((va + vb) + vc): q = (a + ab (vb inv)) + ac (vc inv)
//                (a + t v is per axis a + (t v), a product then a sum).
//   fallback     when l2 == 0 (a zero-area face), or the divisor of the region reached is not > 0 (below), q is the closest point
//                of the segments ab, bc, ca instead: on the segment (s, e), u = e - s, t = (p - s) . u; t <= 0: s;
//                else m = u . u, t >= m: e; else s + (t / m) u.  The smaller d2 wins, a tie the earlier segment.
//   distance     d = p - q, d2 = (dx dx + dy dy) + dz dz (the alignment's s3l::dist2 order), s = d . N; the signed
//                distance is (float)(-sqrt(d2)) when s < 0, else (float)sqrt(d2).
//
// No NaN from finite inputs.  Float coordinates are below 2^128 in magnitude, so every difference above is below 2^129,
// every dot or cross product of two differences below 3 2^258 < 2^260, every product of two of those (vc, vb, va) below
// 2^520, and (va + vb) + vc below 2^522: nothing overflows and no Inf appears.  A NaN could then only come from 0 / 0.
// The divisors are d1 - d3 >= d1 >= 0, d2 - d6 >= d2 >= 0 and e + g >= e >= 0 in the edge regions that use them
// (rounding is monotone), (va + vb) + vc in the interior, and m on a segment.  The first four go to the fallback unless
// they are > 0.  The edge divisors can round to 0 on a face of non-zero area: p = (1e20, -1e20, 1) against a = 0,
// b = (1, 1, 0), c = (0, 0, 1) has d1 = d3 = 0, because p - b rounds to p - a; so the fallback covers them too.  On a
// segment, m = u . u > 0 whenever u != 0, since a non-zero difference of floats is at least 2^-149 and its square is a
// normal double.  Every quotient is therefore finite, and so are q, d2 and s.
//
// The index.  S = s3l::cell_edge(R) = R (1 + 2^-20), R = (double)max_distance; the cell of a value v is
// floor(v / S) (s3l::cell_axis).  A face is registered in every cell of its cell box: per axis [cell(lo), cell(hi)],
// lo and hi the smallest and largest float corner coordinate; it has entries(f) = prod (cell(hi) - cell(lo) + 1) of
// them.  A sample p is compared with the faces registered in the 27 cells around its own cell (those in the key range),
// the faces whose cell box meets [cell(p) - 1, cell(p) + 1] on every axis.  Every face whose exact distance from p is
// at most R is among them: the exact closest point q* lies in the face's box, lo <= q*_x <= hi, and since
// v -> floor(v / S) (rounded) is monotone, cell(q*_x) is in [cell(lo), cell(hi)]; |p_x - q*_x| <= R = S / (1 + 2^-20)
// and each rounded quotient v / S with |v / S| < 2^20 is within 2^-33 of the exact one, so the quotients of p_x and q*_x
// differ by less than 1 - 2^-21 + 2^-32 < 1 and their floors by at most 1.  So the box test only removes faces farther
// than R from p, which rounding might otherwise let through; it is part of the rule so that the result is a pure
// function of the samples, the mesh and R.  A vertex of a face (indices in range) whose cell is outside the key range
// [-2^20, 2^20) on some axis, and a mesh with sum entries(f) >= 2^32 over its non-degenerate faces, are configuration
// errors; entries(f) <= 2^63 and is clamped at 2^32 before the sum, which cannot then overflow for fewer than 2^31 faces.
//
// The sums of the statistics (the alignment's scheme).  One sample per thread, 256 per block, sample i in block
// i / 256 at thread i % 256, so the grid depends only on the sample count.  Per block: each warp's 32 values are summed
// by halving, lane l adding lane l + h for h = 16, 8, 4, 2, 1 (a sample that does not match adds +0), then the 8 warp
// sums in order; then one block of 256 threads: thread t adds the partials of blocks t, t + 256, ... to +0 in turn,
// then the 256 totals are summed by halving (t adds t + h for h = 128 ... 1).  That order does not depend on the SM
// count or on scheduling.
#pragma once
#include "scan3d_aux_math.h"
#include "scan3d_align_math.h"
#include "scan3d_voxel_math.h"

namespace s3p {

constexpr int BLOCK = 256;                      // samples per block of the query and of the sum order above
constexpr unsigned long long ENTRY_CLAMP = 1ull << 32;

S3A_HD double dot3(const double v[3], const double w[3])
{
    return S3A_ADD(S3A_ADD(S3A_MUL(v[0], w[0]), S3A_MUL(v[1], w[1])), S3A_MUL(v[2], w[2]));
}

S3A_HD void sub3(const double v[3], const double w[3], double o[3])
{
    for (int k = 0; k < 3; k++) o[k] = S3A_SUB(v[k], w[k]);
}

// o = s + t u per axis
S3A_HD void along(const double s[3], double t, const double u[3], double o[3])
{
    for (int k = 0; k < 3; k++) o[k] = S3A_ADD(s[k], S3A_MUL(t, u[k]));
}

// the closest point of the segment (s, e) to p
S3A_HD void segment_point(const double p[3], const double s[3], const double e[3], double q[3])
{
    double u[3], sp[3];
    sub3(e, s, u);
    sub3(p, s, sp);
    const double t = dot3(sp, u);
    if (t <= 0.0) {
        for (int k = 0; k < 3; k++) q[k] = s[k];
        return;
    }
    const double m = dot3(u, u);
    if (t >= m) {
        for (int k = 0; k < 3; k++) q[k] = e[k];
        return;
    }
    along(s, S3A_DIV(t, m), u, q);
}

S3A_HD double dist2(const double p[3], const double q[3])
{
    double d[3];
    sub3(p, q, d);
    return dot3(d, d);
}

// the fallback: the closest point of ab, bc, ca, the smaller d2 winning, a tie the earlier segment
S3A_HD void edges_point(const double p[3], const double a[3], const double b[3], const double c[3], double q[3])
{
    double r[3], best = 0.0;
    const double* s[3] = {a, b, c};
    for (int k = 0; k < 3; k++) {
        segment_point(p, s[k], s[k == 2 ? 0 : k + 1], r);
        const double d = dist2(p, r);
        if (k == 0 || d < best) {
            best = d;
            for (int j = 0; j < 3; j++) q[j] = r[j];
        }
    }
}

// N = (b - a) x (c - a); returns l2 = N . N
S3A_HD double normal(const double a[3], const double b[3], const double c[3], double N[3])
{
    double ab[3], ac[3];
    sub3(b, a, ab);
    sub3(c, a, ac);
    N[0] = S3A_SUB(S3A_MUL(ab[1], ac[2]), S3A_MUL(ab[2], ac[1]));
    N[1] = S3A_SUB(S3A_MUL(ab[2], ac[0]), S3A_MUL(ab[0], ac[2]));
    N[2] = S3A_SUB(S3A_MUL(ab[0], ac[1]), S3A_MUL(ab[1], ac[0]));
    return dot3(N, N);
}

// q = the closest point of the face (a, b, c) to p, l2 its normal's squared length (Ericson's regions, then the
// fallback)
S3A_HD void closest_point(const double p[3], const double a[3], const double b[3], const double c[3], double l2,
                          double q[3])
{
    if (l2 == 0.0) {
        edges_point(p, a, b, c, q);
        return;
    }
    double ab[3], ac[3], ap[3], bp[3], cp[3];
    sub3(b, a, ab);
    sub3(c, a, ac);
    sub3(p, a, ap);
    const double d1 = dot3(ab, ap), d2 = dot3(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) {
        for (int k = 0; k < 3; k++) q[k] = a[k];
        return;
    }
    sub3(p, b, bp);
    const double d3 = dot3(ab, bp), d4 = dot3(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) {
        for (int k = 0; k < 3; k++) q[k] = b[k];
        return;
    }
    const double vc = S3A_SUB(S3A_MUL(d1, d4), S3A_MUL(d3, d2));
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
        const double den = S3A_SUB(d1, d3);
        if (den > 0.0) along(a, S3A_DIV(d1, den), ab, q);
        else edges_point(p, a, b, c, q);
        return;
    }
    sub3(p, c, cp);
    const double d5 = dot3(ab, cp), d6 = dot3(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) {
        for (int k = 0; k < 3; k++) q[k] = c[k];
        return;
    }
    const double vb = S3A_SUB(S3A_MUL(d5, d2), S3A_MUL(d1, d6));
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
        const double den = S3A_SUB(d2, d6);
        if (den > 0.0) along(a, S3A_DIV(d2, den), ac, q);
        else edges_point(p, a, b, c, q);
        return;
    }
    const double va = S3A_SUB(S3A_MUL(d3, d6), S3A_MUL(d5, d4));
    const double e = S3A_SUB(d4, d3), g = S3A_SUB(d5, d6);
    if (va <= 0.0 && e >= 0.0 && g >= 0.0) {
        const double den = S3A_ADD(e, g);
        double bc[3];
        sub3(c, b, bc);
        if (den > 0.0) along(b, S3A_DIV(e, den), bc, q);
        else edges_point(p, a, b, c, q);
        return;
    }
    const double den = S3A_ADD(S3A_ADD(va, vb), vc);
    if (!(den > 0.0)) {
        edges_point(p, a, b, c, q);
        return;
    }
    const double inv = S3A_DIV(1.0, den);
    double t[3];
    along(a, S3A_MUL(vb, inv), ab, t);
    along(t, S3A_MUL(vc, inv), ac, q);
}

// the squared distance d2 of p from the face (a, b, c) of float corners, and the side s = (p - q) . N
S3A_HD double face_distance(const double p[3], const float fa[3], const float fb[3], const float fc[3], double* s)
{
    const double a[3] = {fa[0], fa[1], fa[2]}, b[3] = {fb[0], fb[1], fb[2]}, c[3] = {fc[0], fc[1], fc[2]};
    double N[3], q[3], d[3];
    const double l2 = normal(a, b, c, N);
    closest_point(p, a, b, c, l2, q);
    sub3(p, q, d);
    *s = dot3(d, N);
    return dot3(d, d);
}

S3A_HD double root(double d2) { return S3L_SQRT(d2); }

// the signed distance of a match, rounded to float
S3A_HD float signed_distance(double d2, double s)
{
    const double r = root(d2);
    return (float)(s < 0.0 ? -r : r);
}

// the cell box [lo, hi] of a face of float corners; false when a corner's cell is outside the key range (or a corner
// is not finite)
S3A_HD bool face_cells(const float* a, const float* b, const float* c, double S, long long lo[3], long long hi[3])
{
    for (int k = 0; k < 3; k++) {
        float l = a[k], h = a[k];
        l = b[k] < l ? b[k] : l;
        h = b[k] > h ? b[k] : h;
        l = c[k] < l ? c[k] : l;
        h = c[k] > h ? c[k] : h;
        if (!s3l::cell_axis((double)l, S, &lo[k]) || !s3l::cell_axis((double)h, S, &hi[k])) return false;
    }
    return true;
}

// entries(f) of a cell box, clamped at 2^32
S3A_HD unsigned long long face_entries(const long long lo[3], const long long hi[3])
{
    const unsigned long long n = (unsigned long long)(hi[0] - lo[0] + 1) * (unsigned long long)(hi[1] - lo[1] + 1) *
                                 (unsigned long long)(hi[2] - lo[2] + 1);
    return n < ENTRY_CLAMP ? n : ENTRY_CLAMP;
}

// candidate (d2, f) beats the best so far: the smaller d2, a tie the smaller face
S3A_HD bool closer(double d2, uint32_t f, double best_d2, uint32_t best_f)
{
    return d2 < best_d2 || (d2 == best_d2 && f < best_f);
}

}  // namespace s3p
