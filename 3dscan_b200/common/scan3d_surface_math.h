// scan3d_surface_math.h -- the arithmetic of the surface extraction (scan3d_voxel_surface): a signed distance on the
// merge's voxel lattice, meshed by naive surface nets.  Written once for the CUDA kernels (scan3d_surface_kernels.cu)
// and for a host build of the very same expressions that the CPU tests compare with an independent numpy restatement
// (tests/test_surface_math_host.py compiles this header with g++ -ffp-contract=off).
//
// S = (double)voxel_size; lattice point g = (i, j, k), x_g = ((double)i S, (double)j S, (double)k S).  Cell g is the
// cube with min corner g; its corner g + (a, b, c) is corner number a + 2 b + 4 c.  Every double operation is one
// correctly rounded IEEE operation, in this order, no FMA:
//
//   corner value  f(g) = s3l::residual(x_g, q, n_q) for q the nearest model point (s3l::dist2, s3l::closer, within
//                 max_distance); inside when f < 0 (so -0.0 is outside)
//   edges         the 12 edges of a cell in the order: axis e = x, y, z; for each, the other two axes (p, q) in
//                 increasing order take (0, 0), (1, 0), (0, 1), (1, 1); lower end u (bit e = 0), upper end w
//   crossing      on an edge whose ends are on different sides, t = f_u / (f_u - f_w); the crossing is
//                 ((double)g_e + t) S on axis e and x_u's coordinates on the other two
//   vertex        per axis the sum of the crossings in edge order, from +0, / (double)count, rounded to float
//   normal        g_e = ((d_00 + d_10) + (d_01 + d_11)), d_pq = f_w - f_u of the axis-e edge at (p, q);
//                 l = sqrt((g_x g_x + g_y g_y) + g_z g_z), (float)(g_e / l), or (0, 0, 0) unless 0 < l < inf
//   colour        per channel (sum of the 8 corners' nearest model colours + 4) / 8, integer division
//   quad          lattice edge g -> g + e_a, (b, d) = the next two axes in cyclic order; v0..v3 = the vertices of
//                 cells g - e_b - e_d, g - e_d, g, g - e_b; (v0, v1, v2), (v0, v2, v3) when f(g) < 0 <= f(g + e_a),
//                 else (v0, v2, v1), (v0, v3, v2): the right-hand normal points from inside to outside
//   order key     27 o + k of model voxel o and the offset g - v_o, k = ((dz + 1) 3 + (dy + 1)) 3 + (dx + 1)
#pragma once
#include "scan3d_align_math.h"

namespace s3s {

constexpr int OFFSETS = 27;   // the 27-neighbourhood of a model voxel

S3A_HD void lattice_pos(long long i, long long j, long long k, double S, double x[3])
{
    x[0] = S3A_MUL((double)i, S);
    x[1] = S3A_MUL((double)j, S);
    x[2] = S3A_MUL((double)k, S);
}

S3A_HD bool inside(double f) { return f < 0.0; }

S3A_HD double crossing_t(double fu, double fw) { return S3A_DIV(fu, S3A_SUB(fu, fw)); }

// corner number of the lower end of edge m (0..3) along axis e: the other two axes in increasing order take the bits
// of m (first axis = bit 0)
S3A_HD int edge_lower(int e, int m)
{
    const int p = e == 0 ? 1 : 0, q = e == 2 ? 1 : 2;
    return ((m & 1) << p) | ((m >> 1) << q);
}

// at least one corner inside and one outside
S3A_HD bool mixed(const double f[8])
{
    int n = 0;
    for (int c = 0; c < 8; c++) n += inside(f[c]) ? 1 : 0;
    return n > 0 && n < 8;
}

// the vertex of an active cell g with corner values f[8]
S3A_HD void vertex_position(const long long g[3], const double f[8], double S, float out[3])
{
    double sum[3] = {0.0, 0.0, 0.0};
    int n = 0;
    for (int e = 0; e < 3; e++)
        for (int m = 0; m < 4; m++) {
            const int u = edge_lower(e, m), w = u | (1 << e);
            if (inside(f[u]) == inside(f[w])) continue;
            const double t = crossing_t(f[u], f[w]);
            for (int x = 0; x < 3; x++) {
                const double c = x == e ? S3A_MUL(S3A_ADD((double)g[e], t), S)
                                        : S3A_MUL((double)(g[x] + ((u >> x) & 1)), S);
                sum[x] = S3A_ADD(sum[x], c);
            }
            n++;
        }
    for (int x = 0; x < 3; x++) out[x] = S3V_D2F(S3A_DIV(sum[x], (double)n));
}

// the trilinear gradient of the cell, normalised
S3A_HD void gradient_normal(const double f[8], float out[3])
{
    double gr[3];
    for (int e = 0; e < 3; e++) {
        double d[4];
        for (int m = 0; m < 4; m++) {
            const int u = edge_lower(e, m);
            d[m] = S3A_SUB(f[u | (1 << e)], f[u]);
        }
        gr[e] = S3A_ADD(S3A_ADD(d[0], d[1]), S3A_ADD(d[2], d[3]));
    }
    const double l = S3L_SQRT(S3A_ADD(S3A_ADD(S3A_MUL(gr[0], gr[0]), S3A_MUL(gr[1], gr[1])), S3A_MUL(gr[2], gr[2])));
    if (!(l > 0.0 && l - l == 0.0)) {
        out[0] = out[1] = out[2] = 0.0f;
        return;
    }
    for (int e = 0; e < 3; e++) out[e] = S3V_D2F(S3A_DIV(gr[e], l));
}

// one colour channel from the sum of the 8 corners' nearest model colours
S3A_HD unsigned char colour(unsigned sum) { return (unsigned char)((sum + 4u) / 8u); }

S3A_HD int offset_index(int dx, int dy, int dz) { return ((dz + 1) * 3 + (dy + 1)) * 3 + (dx + 1); }
S3A_HD void offset_of(int k, int d[3])
{
    d[0] = k % 3 - 1;
    d[1] = (k / 3) % 3 - 1;
    d[2] = k / 9 - 1;
}

// the cells of the quad around lattice edge g -> g + e_a: off[c] is cell c's offset from g (v0..v3 above)
S3A_HD void quad_cells(int a, int off[4][3])
{
    const int b = (a + 1) % 3, d = (a + 2) % 3;
    for (int c = 0; c < 4; c++)
        for (int x = 0; x < 3; x++) off[c][x] = 0;
    off[0][b] = -1;
    off[0][d] = -1;
    off[1][d] = -1;
    off[3][b] = -1;
}

// the two triangles of a quad with vertices v[4]; lower_inside = f(g) < 0
S3A_HD void quad_triangles(const int v[4], bool lower_inside, int tri[6])
{
    tri[0] = v[0];
    tri[3] = v[0];
    if (lower_inside) {
        tri[1] = v[1]; tri[2] = v[2];
        tri[4] = v[2]; tri[5] = v[3];
    } else {
        tri[1] = v[2]; tri[2] = v[1];
        tri[4] = v[3]; tri[5] = v[2];
    }
}

}  // namespace s3s
