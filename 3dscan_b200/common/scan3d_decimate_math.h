// scan3d_decimate_math.h -- the arithmetic of the surface simplification (scan3d_voxel_surface_decimate): vertex
// clustering on a grid of edge H with quadric placement (Rossignac & Borrel 1993; Lindstrom 2000).  Written once for
// the CUDA kernels (scan3d_decimate_kernels.cu) and for a host build of the very same expressions that the CPU tests
// compare with an independent numpy restatement (tests/test_decimate_math_host.py compiles this header with
// g++ -ffp-contract=off).
//
// H = (double)cell_size.  A vertex's cluster is its voxel of edge H in the merge's sense (s3v::axis, s3v::point_key);
// its fraction along an axis is f = t - floor(t), t = (double)x / H, in [0, 1] (1 only when a tiny negative t rounds
// up, as in s3v::axis).  Every double operation below is one
// correctly rounded IEEE operation (S3A_*), in this order, no FMA:
//
//   face plane   d1 = pb - pa, d2 = pc - pa (per axis, the float coordinates as doubles);
//                n = (d1y d2z - d1z d2y, d1z d2x - d1x d2z, d1x d2y - d1y d2x); l2 = (nx nx + ny ny) + nz nz;
//                l2 == 0: the face adds no quadric; else l = sqrt(l2), u = n / l, w = (l * 0.5) / (H * H)
//   corner       e = (ux fx + uy fy) + uz fz with the corner's own fractions; its 10 coefficients
//                c = (ux ux, ux uy, ux uz, uy uy, uy uz, uz uz, ux e, uy e, uz e, e e), each as w * c_j, rounded to
//                the int64 rint((w * c_j) * 2^P) (half to even) and added to the corner's cluster
//   placement    A = the 3x3 matrix of the first 6 sums * 2^-P (row-major upper triangle), b = the next 3 * 2^-P;
//                ybar_a = (double)sum q_a / (Q (double)n) from the merge's sums (Q = 2^24); tr = (A00 + A11) + A22;
//                tr == 0: y = ybar; else mu = DAMPING * (tr / 3), M = A + mu I, r_a = b_a + mu ybar_a, LDL^T as the
//                alignment's solve6 (D_j = M_jj - sum_k<j (L_jk L_jk) D_k, L_ij = (M_ij - sum_k<j (L_ik L_jk) D_k) / D_j,
//                then z = r - L z forward, y = z / D - L^T y backward); the solve is accepted when mu is finite and
//                > 0, every D_j > mu / 2, and every y_a is finite and in [0, 1]; otherwise y = ybar (a fallback)
//   output       coordinate (float)(((double)i + y_a) * H), the shape of s3v::coord
//   faces        (C(a), C(b), C(c)); collapsed when two are equal; the canonical triple is the cyclic rotation that
//                puts the smallest ordinal first (the winding is kept)
//
// Overflow bound of the int64 sums (checked by the host test).  The surface is surface-nets output (scan3d.h): the
// three vertices of a face lie in three of the four cells around one lattice edge, a box of 1 x 2 x 2 voxels of edge
// s.  Every side of the face is at most that box's diagonal 3 s, so its area is at most (sqrt(3) / 4) (3 s)^2 =
// AREA_MAX_S2 s^2, and w <= AREA_MAX_S2 / r^2 with r = H / s.  |u_a| <= 1 and |e| <= |u| |f| < sqrt(3), so every
// coefficient of a corner is at most 3 w in magnitude before rounding: |rint(w c_j 2^P)| <= face_bound(r) =
// 3 AREA_MAX_S2 / r^2 2^P + 0.5.  A vertex is in at most 24 faces (2 per lattice edge of its cell).  A vertex lies in
// its own cell (up to the float rounding of its coordinate), so a cluster holds the vertices of at most
// floor(r) + 3 cells per axis.  Each cluster sum is therefore at most sum_bound(r) = (floor(r) + 3)^3 * 24 *
// face_bound(r) in magnitude; with P = 40 and r in [1, 256] that is below 2^56.3 (r = 256), under 2^63.
// The bound is per lattice cell, so it survives the non-manifold repair (scan3d_voxel_surface_repair): a split only
// divides a cell's faces among copies at the same position, in the same cell, and dropped faces only lower the count,
// so a repaired raw surface stays decimatable (common/scan3d_repair_math.h).
#pragma once
#include "scan3d_aux_math.h"
#include "scan3d_voxel_math.h"

#if defined(__CUDA_ARCH__)
#define S3Q_UNROLL _Pragma("unroll")
#else
#define S3Q_UNROLL
#endif

namespace s3q {

constexpr int P = 40;                                       // fixed-point bits of the quadric coefficients
constexpr double SCALE = 1099511627776.0;                   // 2^P
constexpr double INV_SCALE = 1.0 / 1099511627776.0;         // 2^-P (exact)
constexpr double DAMPING = 1e-3;                            // mu = DAMPING * trace(A) / 3 pulls y towards the mean
constexpr int NQ = 10;                                      // coefficients per cluster
constexpr double RATIO_MAX = 256.0;                         // cell_size / voxel_size in [1, RATIO_MAX]
constexpr double AREA_MAX_S2 = 3.8971143170299740;          // 9 sqrt(3) / 4, the largest face area in s^2
constexpr int FACES_PER_VERTEX = 24;

enum Placement { PLACED = 0, MEAN = 1, FALLBACK = 2 };      // solved; trace 0 (the mean); the mean after a failure

// the bound on one rounded corner coefficient, and on one cluster sum, for r = H / s (see above)
S3A_HD double face_bound(double r) { return 3.0 * AREA_MAX_S2 / (r * r) * SCALE + 0.5; }
S3A_HD double sum_bound(double r)
{
    const double c = floor(r) + 3.0;
    return c * c * c * FACES_PER_VERTEX * face_bound(r);
}

// the fraction of x in its cluster along one axis (finite x)
S3A_HD double fraction(float x, double H)
{
    const double t = S3A_DIV((double)x, H);
    return S3A_SUB(t, floor(t));
}

// the unit normal u and the weight w of face (a, b, c); false when l2 == 0 (the face adds no quadric)
S3A_HD bool face_plane(const float a[3], const float b[3], const float c[3], double H, double u[3], double* w)
{
    double d1[3], d2[3];
    S3Q_UNROLL
    for (int k = 0; k < 3; k++) {
        d1[k] = S3A_SUB((double)b[k], (double)a[k]);
        d2[k] = S3A_SUB((double)c[k], (double)a[k]);
    }
    const double n[3] = {S3A_SUB(S3A_MUL(d1[1], d2[2]), S3A_MUL(d1[2], d2[1])),
                         S3A_SUB(S3A_MUL(d1[2], d2[0]), S3A_MUL(d1[0], d2[2])),
                         S3A_SUB(S3A_MUL(d1[0], d2[1]), S3A_MUL(d1[1], d2[0]))};
    const double l2 = S3A_ADD(S3A_ADD(S3A_MUL(n[0], n[0]), S3A_MUL(n[1], n[1])), S3A_MUL(n[2], n[2]));
    if (l2 == 0.0) return false;
    const double l = S3V_SQRT(l2);
    S3Q_UNROLL
    for (int k = 0; k < 3; k++) u[k] = S3A_DIV(n[k], l);
    *w = S3A_DIV(S3A_MUL(l, 0.5), S3A_MUL(H, H));
    return true;
}

// a double as the fixed-point integer rint(v * 2^P)
S3A_HD long long to_fixed(double v) { return S3V_D2LL_RN(S3A_MUL(v, SCALE)); }

// the 10 fixed-point coefficients a corner with fractions f adds to its cluster
S3A_HD void corner_coeffs(const double u[3], double w, const double f[3], long long q[NQ])
{
    const double e = S3A_ADD(S3A_ADD(S3A_MUL(u[0], f[0]), S3A_MUL(u[1], f[1])), S3A_MUL(u[2], f[2]));
    const double c[NQ] = {S3A_MUL(u[0], u[0]), S3A_MUL(u[0], u[1]), S3A_MUL(u[0], u[2]), S3A_MUL(u[1], u[1]),
                          S3A_MUL(u[1], u[2]), S3A_MUL(u[2], u[2]), S3A_MUL(u[0], e),    S3A_MUL(u[1], e),
                          S3A_MUL(u[2], e),    S3A_MUL(e, e)};
    S3Q_UNROLL
    for (int j = 0; j < NQ; j++) q[j] = to_fixed(S3A_MUL(w, c[j]));
}

// the position y in [0, 1]^3 (cell units) of a cluster from its quadric sums qs and the merge's position sums sq over
// n vertices; returns PLACED, MEAN (trace 0) or FALLBACK (y = the mean)
S3A_HD int place(const long long qs[NQ], const unsigned long long sq[3], unsigned int n, double y[3])
{
    const double den = S3A_MUL(s3v::Q, (double)n);
    double ybar[3], a[NQ];
    S3Q_UNROLL
    for (int k = 0; k < 3; k++) ybar[k] = S3A_DIV(S3V_ULL2D(sq[k]), den);
    S3Q_UNROLL
    for (int j = 0; j < 9; j++) a[j] = S3A_MUL(S3V_LL2D(qs[j]), INV_SCALE);
    const double tr = S3A_ADD(S3A_ADD(a[0], a[3]), a[5]);
    int status = MEAN;
    if (tr != 0.0) {
        status = FALLBACK;
        const double mu = S3A_MUL(DAMPING, S3A_DIV(tr, 3.0));
        // M_ij by (i, j) over the upper triangle a[0..5]: (0,0) (0,1) (0,2) (1,1) (1,2) (2,2)
        const double M[3][3] = {{S3A_ADD(a[0], mu), a[1], a[2]},
                                {a[1], S3A_ADD(a[3], mu), a[4]},
                                {a[2], a[4], S3A_ADD(a[5], mu)}};
        const double half_mu = S3A_MUL(mu, 0.5);
        double L[3][3] = {}, D[3] = {}, z[3], x[3];
        bool ok = mu > 0.0 && mu - mu == 0.0;
        S3Q_UNROLL
        for (int j = 0; j < 3; j++) {
            double d = M[j][j];
            S3Q_UNROLL
            for (int k = 0; k < j; k++) d = S3A_SUB(d, S3A_MUL(S3A_MUL(L[j][k], L[j][k]), D[k]));
            ok = ok && d > half_mu;
            D[j] = d;
            S3Q_UNROLL
            for (int i = j + 1; i < 3; i++) {
                double v = M[j][i];
                S3Q_UNROLL
                for (int k = 0; k < j; k++) v = S3A_SUB(v, S3A_MUL(S3A_MUL(L[i][k], L[j][k]), D[k]));
                L[i][j] = S3A_DIV(v, d);
            }
        }
        S3Q_UNROLL
        for (int i = 0; i < 3; i++) {
            double v = S3A_ADD(a[6 + i], S3A_MUL(mu, ybar[i]));
            S3Q_UNROLL
            for (int k = 0; k < i; k++) v = S3A_SUB(v, S3A_MUL(L[i][k], z[k]));
            z[i] = v;
        }
        S3Q_UNROLL
        for (int i = 2; i >= 0; i--) {
            double v = S3A_DIV(z[i], D[i]);
            S3Q_UNROLL
            for (int k = i + 1; k < 3; k++) v = S3A_SUB(v, S3A_MUL(L[k][i], x[k]));
            x[i] = v;
        }
        S3Q_UNROLL
        for (int k = 0; k < 3; k++) ok = ok && x[k] >= 0.0 && x[k] <= 1.0;   // false for NaN
        if (ok) {
            S3Q_UNROLL
            for (int k = 0; k < 3; k++) y[k] = x[k];
            return PLACED;
        }
    }
    S3Q_UNROLL
    for (int k = 0; k < 3; k++) y[k] = ybar[k];
    return status;
}

// the output coordinate of axis a of a cluster with integer coordinate i
S3A_HD float coord(long long i, double y, double H) { return S3V_D2F(S3A_MUL(S3A_ADD((double)i, y), H)); }

// a face of distinct cluster ordinals in its canonical rotation (smallest first, winding kept)
S3A_HD void canonical(int a, int b, int c, int out[3])
{
    if (a < b && a < c) {
        out[0] = a; out[1] = b; out[2] = c;
    } else if (b < c) {
        out[0] = b; out[1] = c; out[2] = a;
    } else {
        out[0] = c; out[1] = a; out[2] = b;
    }
}

S3A_HD bool collapsed(int a, int b, int c) { return a == b || b == c || a == c; }

}  // namespace s3q
