// Host build of 3dscan_b200/common/scan3d_fill_math.h for tests/test_fill_math_host.py (g++ -ffp-contract=off): the
// triangle terms and the cos rule over arrays, and the whole per-hole DP, so numpy can compare them bit for bit.
#include <math.h>
#include <stdint.h>

#include <vector>

#include "../3dscan_b200/common/scan3d_fill_math.h"

extern "C" {

// triangles [n][3][3] float (corners a, b, c): u [n][3], area [n], has [n]
void s3h_host_triangle(const float* p, long long n, double* u, double* area, uint8_t* has)
{
    for (long long i = 0; i < n; i++) {
        const float* t = p + 9 * i;
        u[3 * i] = u[3 * i + 1] = u[3 * i + 2] = 0.0;
        has[i] = s3h::triangle(t, t + 3, t + 6, u + 3 * i, area + i);
    }
}

void s3h_host_cos(const double* a, const uint8_t* ha, const double* b, const uint8_t* hb, long long n, double* out)
{
    for (long long i = 0; i < n; i++) out[i] = s3h::cos_of(a + 3 * i, ha[i], b + 3 * i, hb[i]);
}

// the DP of one hole of n vertices at p [n][3] with rim faces rims [n][3][3] and exists [n][n] (row-major, 1 = {v_i,
// v_j} is an edge of the mesh) into cmin, area [n][n] and k [n][n] (cells with j > i); faces [n - 2][3] in local ids.
// Returns 1 when the hole is filled.
int s3h_host_polygon(const float* p, const float* rims, const uint8_t* exists, int n, double* cmin, double* area,
                     int* k, int* faces)
{
    std::vector<s3h::Cell> cells(s3h::cells_of(n));
    const float(*pp)[3] = reinterpret_cast<const float(*)[3]>(p);
    for (int t = 0; t < n; t++) {
        const float* r = rims + 9 * t;
        s3h::rim_cell(r, r + 3, r + 6, &cells[t < n - 1 ? s3h::cell_index(t, t + 1) : s3h::cells_of(n) - 1]);
    }
    for (int d = 2; d < n; d++)
        for (int i = 0; i + d < n; i++) {
            const int j = i + d;
            s3h::solve_cell(pp, cells.data(), n, i, j, exists[(size_t)i * n + j] != 0, &cells[s3h::cell_index(i, j)]);
        }
    for (int j = 1; j < n; j++)
        for (int i = 0; i < j; i++) {
            const s3h::Cell& c = cells[s3h::cell_index(i, j)];
            cmin[(size_t)i * n + j] = c.cmin;
            area[(size_t)i * n + j] = c.area;
            k[(size_t)i * n + j] = c.k;
        }
    if (cells[s3h::cell_index(0, n - 1)].k == s3h::INFEASIBLE) return 0;
    std::vector<unsigned int> verts(n), stack(n);
    for (int t = 0; t < n; t++) verts[t] = (unsigned int)t;
    s3h::emit_faces(cells.data(), n, verts.data(), stack.data(), faces);
    return 1;
}

// the caps and the decimation bound: out = {NETS_MAX_EDGES, MAX_EDGES, holds(N), holds(N + 1)}, bound [256] of
// nets_sum_bound(m, N) for m = 1 ... 256
void s3h_host_limits(long long* out, double* bound)
{
    out[0] = s3h::NETS_MAX_EDGES;
    out[1] = s3h::MAX_EDGES;
    out[2] = s3h::nets_bound_holds(s3h::NETS_MAX_EDGES);
    out[3] = s3h::nets_bound_holds(s3h::NETS_MAX_EDGES + 1);
    for (int m = 1; m <= 256; m++) bound[m - 1] = s3h::nets_sum_bound(m, s3h::NETS_MAX_EDGES);
}
}
