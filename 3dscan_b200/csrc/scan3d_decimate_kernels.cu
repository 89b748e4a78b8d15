// scan3d_decimate_kernels.cu -- the simplification of the held voxel surface (scan3d_voxel_surface_decimate): vertex
// clustering on a grid of edge H with quadric placement.  The arithmetic is in common/scan3d_decimate_math.h, shared
// with the host test; this file owns the per-cluster sums, the duplicate-face table and the emission.
//
// The clusters are the voxels of a second VoxelTable: launch_voxel_add over the surface's vertices keys them, sums
// their positions, normals and colours and numbers them by first vertex, exactly as the merge does.  The quadric sums
// are int64 atomics indexed by cluster ordinal, so they do not depend on scheduling.  Duplicate faces are found with
// an open-addressing table of face indices keyed on the canonical cluster triple: the first face of each triple claims
// a slot with atomicCAS, later ones compare triples and lower the slot to the smallest face index with atomicMin.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "../common/scan3d_decimate_math.h"

namespace s3d {

namespace {

constexpr int DT = 256;                                 // threads per block of the face kernels
constexpr unsigned FULL = 0xffffffffu;

unsigned grid(uint64_t n, int threads) { return n ? (unsigned)((n + threads - 1) / threads) : 1u; }

// the exact sum of v over the lanes of grp (every lane of grp calls it): three 32-bit reductions of 16 + 16 + 32 bits,
// recombined modulo 2^64, so the int64 two's-complement sum is exact
__device__ __forceinline__ long long group_sum64(unsigned grp, long long v)
{
    const unsigned long long u = (unsigned long long)v;
    const uint32_t lo = __reduce_add_sync(grp, (uint32_t)(u & 0xffffu));
    const uint32_t mid = __reduce_add_sync(grp, (uint32_t)((u >> 16) & 0xffffu));
    const uint32_t hi = __reduce_add_sync(grp, (uint32_t)(u >> 32));
    return (long long)(((unsigned long long)hi << 32) + ((unsigned long long)mid << 16) + (unsigned long long)lo);
}

__device__ __forceinline__ bool same_triple(const int* a, const int* b)
{
    return a[0] == b[0] && a[1] == b[1] && a[2] == b[2];
}

__device__ __forceinline__ void canonical_of(const int32_t* __restrict__ ctri, uint32_t f, int out[3])
{
    s3q::canonical(ctri[3 * (size_t)f], ctri[3 * (size_t)f + 1], ctri[3 * (size_t)f + 2], out);
}

}  // namespace

// One thread per face: its cluster triple into ctri, and its plane's coefficients into the sums of its corners'
// clusters.  Lanes whose corners share a cluster (neighbouring faces mostly do) add one group sum with one set of
// atomics.
__global__ void __launch_bounds__(DT) k_dec_quadrics(VoxelTable t, const float* __restrict__ xyz,
                                                     const int32_t* __restrict__ tri, uint32_t n_faces, double H,
                                                     const uint32_t* __restrict__ point_slot,
                                                     int32_t* __restrict__ ctri, unsigned long long* __restrict__ quad)
{
    const uint32_t f = blockIdx.x * DT + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int32_t v[3] = {0, 0, 0};
    uint32_t c[3] = {VOXEL_NO_SLOT, VOXEL_NO_SLOT, VOXEL_NO_SLOT};
    double u[3], w = 0.0;
    bool plane = false;
    if (f < n_faces) {
        for (int k = 0; k < 3; k++) {
            v[k] = tri[3 * (size_t)f + k];
            const uint32_t s = point_slot[v[k]];   // always a slot: the surface lies inside the key range (scan3d.h)
            c[k] = s == VOXEL_NO_SLOT ? VOXEL_NO_SLOT : t.ordinal[s];
            ctri[3 * (size_t)f + k] = (int32_t)c[k];
        }
        plane = s3q::face_plane(xyz + 3 * (size_t)v[0], xyz + 3 * (size_t)v[1], xyz + 3 * (size_t)v[2], H, u, &w);
    }
    for (int k = 0; k < 3; k++) {
        const bool has = plane && c[k] != VOXEL_NO_SLOT;
        long long q[s3q::NQ];
        if (has) {
            const double fr[3] = {s3q::fraction(xyz[3 * (size_t)v[k]], H), s3q::fraction(xyz[3 * (size_t)v[k] + 1], H),
                                  s3q::fraction(xyz[3 * (size_t)v[k] + 2], H)};
            s3q::corner_coeffs(u, w, fr, q);
        } else {
#pragma unroll
            for (int j = 0; j < s3q::NQ; j++) q[j] = 0;
        }
        const uint32_t key = has ? c[k] : VOXEL_NO_SLOT;
        const unsigned grp = __match_any_sync(FULL, key);
        const bool leader = lane == __ffs(grp) - 1;
#pragma unroll
        for (int j = 0; j < s3q::NQ; j++) {
            const long long sum = group_sum64(grp, q[j]);
            if (has && leader) atomicAdd(quad + (size_t)key * s3q::NQ + j, (unsigned long long)sum);
        }
    }
}

// One thread per face: a face of three distinct clusters finds or claims the slot of its canonical triple (slot_of[f]);
// a collapsed face counts in state->collapsed and gets no slot.
__global__ void __launch_bounds__(DT) k_dec_insert(const int32_t* __restrict__ ctri, uint32_t n_faces, uint32_t* table,
                                                   uint32_t cap, uint32_t* __restrict__ slot_of, DecimateState* state)
{
    const uint32_t f = blockIdx.x * DT + threadIdx.x;
    bool col = false;
    if (f < n_faces) {
        const int a = ctri[3 * (size_t)f], b = ctri[3 * (size_t)f + 1], c = ctri[3 * (size_t)f + 2];
        uint32_t slot = VOXEL_NO_SLOT;
        col = s3q::collapsed(a, b, c) || a < 0 || b < 0 || c < 0;
        if (!col) {
            int k[3];
            s3q::canonical(a, b, c, k);
            const unsigned long long key =
                mix64(((unsigned long long)(uint32_t)k[0] << 32) | (uint32_t)k[1]) ^ (unsigned long long)(uint32_t)k[2];
            uint32_t s = hash_home(key, cap);
            for (uint32_t p = 0; p < cap; p++) {
                uint32_t g = __ldcg(table + s);     // a slot's triple never changes once set
                if (g == VOXEL_NO_SLOT) {
                    g = atomicCAS(table + s, VOXEL_NO_SLOT, f);
                    if (g == VOXEL_NO_SLOT) {
                        slot = s;
                        break;
                    }
                }
                int kg[3];
                canonical_of(ctri, g, kg);
                if (same_triple(k, kg)) {
                    atomicMin(table + s, f);
                    slot = s;
                    break;
                }
                s = s + 1 == cap ? 0 : s + 1;
            }
        }
        slot_of[f] = slot;
    }
    const unsigned m = __ballot_sync(FULL, col);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&state->collapsed, (uint32_t)__popc(m));
}

// keep[f] = face f is the first face of its canonical triple
__global__ void __launch_bounds__(DT) k_dec_flags(const uint32_t* __restrict__ table,
                                                  const uint32_t* __restrict__ slot_of, uint32_t n_faces,
                                                  uint8_t* __restrict__ keep)
{
    const uint32_t f = blockIdx.x * DT + threadIdx.x;
    if (f >= n_faces) return;
    const uint32_t s = slot_of[f];
    keep[f] = s != VOXEL_NO_SLOT && table[s] == f;
}

// one output vertex per cluster, in ordinal order: the placement, the merge's normal and colour
__global__ void k_dec_vertices(VoxelTable t, const unsigned long long* __restrict__ quad, double H,
                               float* __restrict__ xyz2, float* __restrict__ nrm2, uint8_t* __restrict__ rgb2,
                               DecimateState* state)
{
    const uint32_t total = t.state->total[1];
    uint32_t fallbacks = 0;
    for (uint32_t o = blockIdx.x * blockDim.x + threadIdx.x; o < total; o += gridDim.x * blockDim.x) {
        const uint32_t s = t.ord2slot[o];
        const unsigned long long key = t.keys[s];
        const VoxelSlot a = t.acc[s];
        long long qs[s3q::NQ];
#pragma unroll
        for (int j = 0; j < s3q::NQ; j++) qs[j] = (long long)quad[(size_t)o * s3q::NQ + j];
        double y[3];
        fallbacks += s3q::place(qs, a.q, a.n, y) == s3q::FALLBACK;
        for (int k = 0; k < 3; k++) {
            xyz2[3 * (size_t)o + k] = s3q::coord(s3v::key_axis(key, k), y[k], H);
            rgb2[3 * (size_t)o + k] = s3v::colour(a.c[k], a.n);
        }
        s3v::normal_out((long long)a.m[0], (long long)a.m[1], (long long)a.m[2], nrm2 + 3 * (size_t)o);
    }
    fallbacks = __reduce_add_sync(FULL, fallbacks);
    if ((threadIdx.x & 31) == 0 && fallbacks) atomicAdd(&state->fallbacks, fallbacks);
}

// kept face f goes to rank r of its keep flag with its cluster triple in its original rotation
__global__ void __launch_bounds__(POINT_BLOCK) k_dec_faces(const uint8_t* __restrict__ keep,
                                                           const uint32_t* __restrict__ offsets, uint32_t n_faces,
                                                           const int32_t* __restrict__ ctri,
                                                           int32_t* __restrict__ faces2)
{
    const uint32_t f = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const bool k = f < n_faces && keep[f] != 0;
    const uint32_t r = offsets[blockIdx.x] + block_rank(k);
    if (!k) return;
#pragma unroll
    for (int j = 0; j < 3; j++) faces2[3 * (size_t)r + j] = ctri[3 * (size_t)f + j];
}

cudaError_t DecimateWorkspace::run(const SurfaceMesh& in, double H, SurfaceMesh& out, int sm_count, cudaStream_t st,
                                   int64_t* launches)
{
    const uint32_t n_vertices = (uint32_t)in.vertices, n_faces = (uint32_t)in.faces;
    // the cluster table is sized as the merge's for max_voxels = the vertex count
    const size_t av = n_vertices ? n_vertices : 1, af = n_faces ? n_faces : 1;
    const uint32_t table_cap = (uint32_t)(2 * af);
    cudaError_t e = clusters.reset((uint32_t)av, H, sm_count, st);
    if (e == cudaSuccess)
        e = grow_group(Grow(point_slot, av), Grow(vert_flags, av),
                       Grow(vert_counts, (av + POINT_BLOCK - 1) / POINT_BLOCK + 1), Grow(quad, s3q::NQ * av));
    if (e == cudaSuccess)
        e = grow_group(Grow(ctri, 3 * af), Grow(table, table_cap), Grow(slot_of, af), Grow(keep, af),
                       Grow(face_counts, (af + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    if (e == cudaSuccess) e = state.ensure(1);
    if (e == cudaSuccess) e = cudaMemsetAsync(quad, 0, s3q::NQ * av * sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(table, 0xff, (size_t)table_cap * sizeof(uint32_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(state, 0, sizeof(DecimateState), st);
    if (e != cudaSuccess) return e;
    const VoxelTable& t = clusters.view;
    DecimateState* ds = state;
    // an empty surface still runs every launch: one block that reads a vertex count of 0
    const uint32_t plane = n_vertices ? n_vertices : 1;
    e = launch_voxel_add(t, in.xyz, in.nrm, in.rgb, n_vertices ? nullptr : &ds->zero, plane, point_slot, vert_flags,
                         vert_counts, 0, st, launches);
    if (e != cudaSuccess) return e;
    k_dec_quadrics<<<grid(n_faces, DT), DT, 0, st>>>(t, in.xyz, in.tri, n_faces, H, point_slot, ctri, quad);
    k_dec_insert<<<grid(n_faces, DT), DT, 0, st>>>(ctri, n_faces, table, table_cap, slot_of, ds);
    k_dec_flags<<<grid(n_faces, DT), DT, 0, st>>>(table, slot_of, n_faces, keep);
    e = launch_point_offsets(keep, n_faces, face_counts, &ds->faces, st);
    if (e != cudaSuccess) return e;
    k_dec_vertices<<<4 * sm_count, 256, 0, st>>>(t, quad, H, out.xyz, out.nrm, out.rgb, ds);
    k_dec_faces<<<grid(n_faces, POINT_BLOCK), POINT_BLOCK, 0, st>>>(keep, face_counts, n_faces, ctri, out.tri);
    *launches += 7;
    return cudaGetLastError();
}

}  // namespace s3d
