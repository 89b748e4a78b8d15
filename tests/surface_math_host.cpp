// Host build of 3dscan_b200/common/scan3d_surface_math.h (the very expressions the CUDA kernels of
// scan3d_surface_kernels.cu evaluate): the per-element functions, and a sequential surface extraction built from them
// with plain loops and a map, so that the CPU test suite can compare both with numpy without a GPU.
// Built by tests/test_surface_math_host.py with g++ -O2 -ffp-contract=off.
#include <stddef.h>
#include <stdint.h>

#include <algorithm>
#include <map>
#include <vector>

#include "../3dscan_b200/common/scan3d_surface_math.h"
#include "../include/scan3d.h"

extern "C" {

void s3s_host_lattice_pos(const long long* g, long long n, float voxel_size, double* x)
{
    for (long long i = 0; i < n; i++) s3s::lattice_pos(g[3 * i], g[3 * i + 1], g[3 * i + 2], (double)voxel_size, x + 3 * i);
}

void s3s_host_residual(const double* p, const float* q, const float* nrm, long long n, double* out)
{
    for (long long i = 0; i < n; i++)
        out[i] = s3l::residual(p + 3 * i, q[3 * i], q[3 * i + 1], q[3 * i + 2], nrm[3 * i], nrm[3 * i + 1], nrm[3 * i + 2]);
}

// per cell (g [n][3], f [n][8]): mixed flag, vertex, normal
void s3s_host_cells(const long long* g, const double* f, long long n, float voxel_size, uint8_t* mixed, float* v,
                    float* nrm)
{
    for (long long i = 0; i < n; i++) {
        mixed[i] = s3s::mixed(f + 8 * i);
        if (mixed[i]) s3s::vertex_position(g + 3 * i, f + 8 * i, (double)voxel_size, v + 3 * i);
        s3s::gradient_normal(f + 8 * i, nrm + 3 * i);
    }
}

void s3s_host_colour(const unsigned* sum, long long n, uint8_t* out)
{
    for (long long i = 0; i < n; i++) out[i] = s3s::colour(sum[i]);
}

void s3s_host_offsets(int* k_of, int* d_of)
{
    for (int dz = -1; dz <= 1; dz++)
        for (int dy = -1; dy <= 1; dy++)
            for (int dx = -1; dx <= 1; dx++) k_of[9 * (dz + 1) + 3 * (dy + 1) + dx + 1] = s3s::offset_index(dx, dy, dz);
    for (int k = 0; k < 27; k++) s3s::offset_of(k, d_of + 3 * k);
}

// axis a, lower side: the quad's cell offsets [4][3] and triangles [6] of v = (0, 1, 2, 3)
void s3s_host_quad(int a, int lower_inside, int* off, int* tri)
{
    int o[4][3];
    s3s::quad_cells(a, o);
    for (int c = 0; c < 4; c++)
        for (int x = 0; x < 3; x++) off[3 * c + x] = o[c][x];
    const int v[4] = {0, 1, 2, 3};
    s3s::quad_triangles(v, lower_inside != 0, tri);
}

// The whole extraction, sequentially.  Model: m voxels (xyz, normals, rgb, their merge indices ijk); those with a zero
// normal are not in it.  Outputs hold up to cap_v vertices and cap_f faces; counts: [vertices, faces, lattice points,
// undefined points].
void s3s_host_extract(const float* mxyz, const float* mnrm, const uint8_t* mrgb, const long long* mijk, long long m,
                      float voxel_size, float max_distance, float* vxyz, float* vnrm, uint8_t* vrgb, int* faces,
                      long long cap_v, long long cap_f, long long* counts)
{
    typedef std::vector<long long> Key;
    const double S = (double)voxel_size, R = (double)max_distance, r2 = S3A_MUL(R, R);
    std::map<Key, unsigned long long> owner;
    for (long long o = 0; o < m; o++) {
        if (mnrm[3 * o] == 0.0f && mnrm[3 * o + 1] == 0.0f && mnrm[3 * o + 2] == 0.0f) continue;
        for (int k = 0; k < 27; k++) {
            int d[3];
            s3s::offset_of(k, d);
            Key g = {mijk[3 * o] + d[0], mijk[3 * o + 1] + d[1], mijk[3 * o + 2] + d[2]};
            bool in = true;
            for (int x = 0; x < 3; x++) in = in && g[x] >= s3v::I_MIN && g[x] + 1 < s3v::I_MAX;
            if (!in) continue;
            const unsigned long long key = 27ull * (unsigned long long)o + (unsigned long long)k;
            auto it = owner.find(g);
            if (it == owner.end()) owner[g] = key;
            else it->second = std::min(it->second, key);
        }
    }
    struct Point {
        double f;
        long long near;
    };
    std::map<Key, Point> pts;
    for (auto& c : owner)
        for (int b = 0; b < 8; b++) pts[Key{c.first[0] + (b & 1), c.first[1] + ((b >> 1) & 1), c.first[2] + (b >> 2)}];
    long long undefined = 0;
    for (auto& pt : pts) {
        double x[3];
        s3s::lattice_pos(pt.first[0], pt.first[1], pt.first[2], S, x);
        double best = 0.0;
        long long bo = -1;
        for (long long o = 0; o < m; o++) {
            if (mnrm[3 * o] == 0.0f && mnrm[3 * o + 1] == 0.0f && mnrm[3 * o + 2] == 0.0f) continue;
            const double d = s3l::dist2(x, mxyz[3 * o], mxyz[3 * o + 1], mxyz[3 * o + 2]);
            if (d <= r2 && (bo < 0 || s3l::closer(d, (uint32_t)o, best, (uint32_t)bo))) {
                best = d;
                bo = o;
            }
        }
        pt.second.near = bo;
        pt.second.f = bo < 0 ? 0.0
                             : s3l::residual(x, mxyz[3 * bo], mxyz[3 * bo + 1], mxyz[3 * bo + 2], mnrm[3 * bo],
                                             mnrm[3 * bo + 1], mnrm[3 * bo + 2]);
        undefined += bo < 0;
    }
    // active cells in key order
    std::vector<std::pair<unsigned long long, Key>> active;
    for (auto& c : owner) {
        double f[8];
        bool def = true;
        for (int b = 0; b < 8; b++) {
            const Point& p = pts[Key{c.first[0] + (b & 1), c.first[1] + ((b >> 1) & 1), c.first[2] + (b >> 2)}];
            def = def && p.near >= 0;
            f[b] = p.f;
        }
        if (def && s3s::mixed(f)) active.push_back({c.second, c.first});
    }
    std::sort(active.begin(), active.end());
    std::map<Key, int> vert;
    for (size_t r = 0; r < active.size(); r++) vert[active[r].second] = (int)r;
    long long nf = 0;
    for (size_t r = 0; r < active.size(); r++) {
        const Key& g = active[r].second;
        const long long gg[3] = {g[0], g[1], g[2]};
        double f[8];
        unsigned sum[3] = {0, 0, 0};
        for (int b = 0; b < 8; b++) {
            const Point& p = pts[Key{g[0] + (b & 1), g[1] + ((b >> 1) & 1), g[2] + (b >> 2)}];
            f[b] = p.f;
            for (int k = 0; k < 3; k++) sum[k] += mrgb[3 * p.near + k];
        }
        if ((long long)r < cap_v) {
            s3s::vertex_position(gg, f, S, vxyz + 3 * r);
            s3s::gradient_normal(f, vnrm + 3 * r);
            for (int k = 0; k < 3; k++) vrgb[3 * r + k] = s3s::colour(sum[k]);
        }
        for (int a = 0; a < 3; a++) {
            Key up = g;
            up[a] += 1;
            if (s3s::inside(pts[up].f) == s3s::inside(f[0])) continue;
            int off[4][3], v[4];
            s3s::quad_cells(a, off);
            bool ok = true;
            for (int c = 0; c < 4 && ok; c++) {
                auto it = vert.find(Key{g[0] + off[c][0], g[1] + off[c][1], g[2] + off[c][2]});
                ok = it != vert.end();
                if (ok) v[c] = it->second;
            }
            if (!ok) continue;
            int tri[6];
            s3s::quad_triangles(v, s3s::inside(f[0]), tri);
            for (int t = 0; t < 2; t++, nf++)
                if (nf < cap_f)
                    for (int k = 0; k < 3; k++) faces[3 * nf + k] = tri[3 * t + k];
        }
    }
    counts[0] = (long long)active.size();
    counts[1] = nf;
    counts[2] = (long long)pts.size();
    counts[3] = undefined;
}

// the field layout of the public structs, for the ctypes mirror
void s3s_host_layout(long long* out)
{
    out[0] = sizeof(scan3d_surface_params);
    out[1] = offsetof(scan3d_surface_params, max_points);
    out[2] = sizeof(scan3d_surface_result);
    out[3] = offsetof(scan3d_surface_result, faces);
    out[4] = offsetof(scan3d_surface_result, lattice_points);
    out[5] = offsetof(scan3d_surface_result, undefined_points);
}
}
