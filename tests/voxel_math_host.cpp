// Host build of 3dscan_b200/common/scan3d_voxel_math.h (the very expressions the CUDA kernels of
// scan3d_voxel_kernels.cu evaluate): a sequential voxel-grid merge built from the header's functions -- a hash map
// and a first-occurrence list -- so that the CPU test suite can compare it with a numpy restatement without a GPU.
// Built by tests/test_voxel_math_host.py with g++ -O2 -ffp-contract=off.
#include <stddef.h>
#include <stdint.h>

#include <unordered_map>
#include <vector>

#include "../3dscan_b200/common/scan3d_voxel_math.h"

namespace {
struct Voxel {
    unsigned long long key;
    unsigned long long q[3] = {0, 0, 0}, c[3] = {0, 0, 0};
    long long m[3] = {0, 0, 0};
    unsigned int n = 0;
};
struct Merge {
    double S;
    std::unordered_map<unsigned long long, size_t> index;
    std::vector<Voxel> voxels;   // in order of their first point
    long long dropped = 0;
};
}  // namespace

extern "C" {

void* s3v_host_begin(float voxel_size)
{
    Merge* g = new Merge;
    g->S = (double)voxel_size;
    return g;
}

void s3v_host_end(void* h) { delete (Merge*)h; }

// xyz f32[n][3]; nrm f32[n][3] and rgb u8[n][3] may be null (zeros)
void s3v_host_add(void* h, const float* xyz, const float* nrm, const uint8_t* rgb, long long n)
{
    Merge* g = (Merge*)h;
    for (long long p = 0; p < n; p++) {
        unsigned long long key, q[3];
        if (!s3v::point_key(xyz[3 * p], xyz[3 * p + 1], xyz[3 * p + 2], g->S, &key, q)) {
            g->dropped++;
            continue;
        }
        auto it = g->index.find(key);
        size_t k;
        if (it == g->index.end()) {
            k = g->voxels.size();
            g->index.emplace(key, k);
            g->voxels.push_back(Voxel{key});
        } else {
            k = it->second;
        }
        Voxel& v = g->voxels[k];
        long long m[3] = {0, 0, 0};
        if (nrm) s3v::normal_fixed(nrm[3 * p], nrm[3 * p + 1], nrm[3 * p + 2], m);
        for (int a = 0; a < 3; a++) {
            v.q[a] += q[a];
            v.m[a] += m[a];
            v.c[a] += rgb ? rgb[3 * p + a] : 0;
        }
        v.n++;
    }
}

// the merged voxels (outputs sized for s3v_host_count); returns the voxel count
long long s3v_host_finish(void* h, float* xyz, float* nrm, uint8_t* rgb, uint32_t* cnt, long long* dropped)
{
    const Merge* g = (const Merge*)h;
    for (size_t o = 0; o < g->voxels.size(); o++) {
        const Voxel& v = g->voxels[o];
        for (int a = 0; a < 3; a++) {
            xyz[3 * o + a] = s3v::coord(v.key, a, v.q[a], v.n, g->S);
            rgb[3 * o + a] = s3v::colour(v.c[a], v.n);
        }
        s3v::normal_out(v.m[0], v.m[1], v.m[2], nrm + 3 * o);
        cnt[o] = v.n;
    }
    *dropped = g->dropped;
    return (long long)g->voxels.size();
}

long long s3v_host_count(void* h) { return (long long)((Merge*)h)->voxels.size(); }
}
