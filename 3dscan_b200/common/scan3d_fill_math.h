// scan3d_fill_math.h -- the arithmetic of the hole filling (scan3d_voxel_surface_fill_holes, scan3d_mesh_fill_holes_dev):
// the minimum-weight triangulation of a boundary loop with Liepa's weight (Liepa 2003; the polygon dynamic program of
// Klincsek 1980 and Barequet & Sharir 1995).  Written once for the CUDA kernels (scan3d_fill_kernels.cu) and for a host
// build of the very same expressions that the CPU tests compare with an independent numpy restatement
// (tests/test_fill_math_host.py compiles this header with g++ -ffp-contract=off).
//
// A hole is a loop v_0 ... v_{n-1} (3 <= n <= max_edges); hole edge t runs from v_t to v_{t+1 mod n} and its rim face
// F_t is the one face that holds the reversed side.  Every double operation below is one correctly rounded IEEE
// operation (S3A_*), in this order, no FMA:
//
//   triangle     from the float corners a, b, c in the order of s3q::face_plane: d1 = p_b - p_a, d2 = p_c - p_a,
//                cross = (d1y d2z - d1z d2y, d1z d2x - d1x d2z, d1x d2y - d1y d2x), l2 = (cx cx + cy cy) + cz cz;
//                area = sqrt(l2) * 0.5; the unit normal u = cross / sqrt(l2) when l2 > 0, else none
//   cos          (u1x u2x + u1y u2y) + u1z u2z; -1 when either triangle has no normal
//   cell (i, j)  0 <= i < j <= n - 1: the best triangulation of v_i ... v_j closed by the side v_j -> v_i.  j - i = 1
//                is hole edge i: feasible, weight (cmin, area) = (+inf, 0), its normal is F_i's.  For j - i >= 2 the
//                cell is infeasible when (i, j) != (0, n - 1) and {v_i, v_j} is already an edge of the mesh (the output
//                stays edge-manifold), or when no candidate is feasible.  Candidates k = i + 1 ... j - 1 whose cells
//                (i, k) and (k, j) are feasible give T_k = (v_i, v_k, v_j) with c_k = min(cos(T_k, N(i, k)),
//                cos(T_k, N(k, j))) (N = the triangle chosen for a cell, F_a for a hole edge (a, a + 1)), and for cell
//                (0, n - 1) also with cos(T_k, F_{n-1}); cmin = min(cmin(i, k), cmin(k, j), c_k) and area =
//                (area(i, k) + area(k, j)) + area(T_k).  The larger cmin wins, then the smaller area, then the smaller
//                k.  The hole is filled when cell (0, n - 1) is feasible.
//   faces        n - 2 faces (v_i, v_k, v_j) in preorder from cell (0, n - 1): the cell's face, then cell (i, k), then
//                cell (k, j).  A hole edge's fill face runs v_t -> v_{t+1}, against its rim face, so the winding
//                continues the rim's and a flat continuation has cos = +1.
//
// Cells are stored per hole at cell_index(i, j) = j (j - 1) / 2 + i, and F_{n-1}'s hole-edge cell after them at
// n (n - 1) / 2: cells_of(n) = n (n - 1) / 2 + 1.
//
// Decimation after a fill (scan3d_voxel_surface_decimate keeps its int64 quadric bound, s3q::sum_bound).  A surface-
// nets hole edge is at most 3 s long, so a fill face of a hole of n edges has every side at most (n / 2) 3 s and area
// at most AREA_MAX_S2 (n / 2)^2 s^2; its rounded corner coefficients are at most fill_face_bound(r, n) = 3 AREA_MAX_S2
// (n / 2)^2 / r^2 2^P + 0.5.  A regular vertex is on one hole, so it gains at most n - 2 fill faces beside its 24 nets
// faces, and a cluster sum is at most (floor(r) + 3)^3 (24 face_bound(r) + (N - 2) fill_face_bound(r, N)) for holes of
// at most N edges.  On each [m, m + 1) that is largest at r = m, and over r in [1, 256] it stays below 2^63 up to
// N = NETS_MAX_EDGES = 22 (2^62.85 at r = 256; N = 23 gives 2^63.05).  So an unrefined surface is filled with
// max_edges <= 22, and a filled surface stays decimatable.
#pragma once
#include "scan3d_aux_math.h"
#include "scan3d_decimate_math.h"
#include "scan3d_voxel_math.h"

namespace s3h {

constexpr int NETS_MAX_EDGES = 22;                          // the largest hole of an unrefined surface (see above)
constexpr int MAX_EDGES = 1024;                             // the largest hole of any other mesh
constexpr int INFEASIBLE = -1;                              // Cell::k of an infeasible cell

// one cell of a hole's dynamic program
struct Cell {
    double cmin;                                            // the smallest cos of the triangulation, +inf for an edge
    double area;
    double u[3];                                            // the unit normal of the cell's triangle, or its rim face's
    int k;                                                  // the chosen apex; 0 for a hole edge; INFEASIBLE
    int has;                                                // u is defined
};

// the bound on a cluster sum of the decimation after filling holes of at most N edges, for r = m in [1, 256]
constexpr double fill_face_bound(double r, int N)
{
    return 3.0 * s3q::AREA_MAX_S2 * (N / 2.0) * (N / 2.0) / (r * r) * s3q::SCALE + 0.5;
}
constexpr double nets_sum_bound(int m, int N)
{
    const double c = m + 3.0;
    return c * c * c * (s3q::FACES_PER_VERTEX * (3.0 * s3q::AREA_MAX_S2 / ((double)m * m) * s3q::SCALE + 0.5) +
                        (N - 2) * fill_face_bound(m, N));
}
constexpr bool nets_bound_holds(int N)
{
    for (int m = 1; m <= (int)s3q::RATIO_MAX; m++)
        if (!(nets_sum_bound(m, N) < 9223372036854775808.0)) return false;
    return true;
}

S3A_HD unsigned int cell_index(int i, int j) { return (unsigned int)j * (unsigned int)(j - 1) / 2u + (unsigned int)i; }
S3A_HD unsigned int cells_of(int n) { return (unsigned int)n * (unsigned int)(n - 1) / 2u + 1u; }

// the unit normal (true when defined) and the area of the triangle (a, b, c)
S3A_HD bool triangle(const float a[3], const float b[3], const float c[3], double u[3], double* area)
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
    const double l = S3V_SQRT(l2);
    *area = S3A_MUL(l, 0.5);
    if (!(l2 > 0.0)) return false;
    for (int k = 0; k < 3; k++) u[k] = S3A_DIV(n[k], l);
    return true;
}

S3A_HD double cos_of(const double a[3], bool ha, const double b[3], bool hb)
{
    if (!ha || !hb) return -1.0;
    return S3A_ADD(S3A_ADD(S3A_MUL(a[0], b[0]), S3A_MUL(a[1], b[1])), S3A_MUL(a[2], b[2]));
}

S3A_HD double min2(double a, double b) { return b < a ? b : a; }

// the cell of a hole edge whose rim face has the corners a, b, c
S3A_HD void rim_cell(const float a[3], const float b[3], const float c[3], Cell* out)
{
    double area;
    out->has = triangle(a, b, c, out->u, &area);
    if (!out->has) out->u[0] = out->u[1] = out->u[2] = 0.0;
    out->cmin = __builtin_inf();
    out->area = 0.0;
    out->k = 0;
}

// cell (i, j), j - i >= 2, of a hole of n vertices at positions p from the cells of shorter spans; exists = {v_i, v_j}
// is an edge of the mesh
S3A_HD void solve_cell(const float (*p)[3], const Cell* cells, int n, int i, int j, bool exists, Cell* out)
{
    Cell best;
    best.k = INFEASIBLE;
    best.cmin = best.area = 0.0;
    best.u[0] = best.u[1] = best.u[2] = 0.0;
    best.has = 0;
    const bool closing = i == 0 && j == n - 1;
    if (!exists || closing) {
        const Cell* close = cells + cells_of(n) - 1;
        for (int k = i + 1; k < j; k++) {
            const Cell* L = cells + cell_index(i, k);
            const Cell* R = cells + cell_index(k, j);
            if (L->k < 0 || R->k < 0) continue;
            double u[3], a;
            const bool has = triangle(p[i], p[k], p[j], u, &a);
            double c = min2(cos_of(u, has, L->u, L->has), cos_of(u, has, R->u, R->has));
            if (closing) c = min2(c, cos_of(u, has, close->u, close->has));
            const double cmin = min2(min2(L->cmin, R->cmin), c);
            const double area = S3A_ADD(S3A_ADD(L->area, R->area), a);
            if (best.k < 0 || cmin > best.cmin || (cmin == best.cmin && area < best.area)) {
                best.cmin = cmin;
                best.area = area;
                for (int e = 0; e < 3; e++) best.u[e] = has ? u[e] : 0.0;
                best.has = has;
                best.k = k;
            }
        }
    }
    *out = best;
}

// the n - 2 faces of a filled hole (cell (0, n - 1) feasible) in preorder into out [n - 2][3], as vertex ids of
// verts; stack holds n entries
S3A_HD void emit_faces(const Cell* cells, int n, const unsigned int* verts, unsigned int* stack, int* out)
{
    int top = 0, f = 0;
    stack[top++] = (unsigned int)(n - 1);                   // (i << 16) | j
    while (top > 0) {
        const unsigned int ij = stack[--top];
        const int i = (int)(ij >> 16), j = (int)(ij & 0xffffu);
        if (j - i < 2) continue;
        const int k = cells[cell_index(i, j)].k;
        out[3 * f] = (int)verts[i];
        out[3 * f + 1] = (int)verts[k];
        out[3 * f + 2] = (int)verts[j];
        f++;
        stack[top++] = (unsigned int)k << 16 | (unsigned int)j;
        stack[top++] = (unsigned int)i << 16 | (unsigned int)k;
    }
}

}  // namespace s3h
