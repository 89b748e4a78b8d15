// scan3d_surface_kernels.cu -- the triangle surface of the merged voxel model (scan3d_voxel_surface): point-to-plane
// distance to the nearest model point at the corners of the merge's voxel lattice, meshed by naive surface nets.  The
// arithmetic is in common/scan3d_surface_math.h, shared with the host test; this file owns the lattice table, the
// vertex order and the face offsets.
//
// The lattice points are held in an open-addressing table (scan3d_hash.cuh) with one slot per distinct point.  Every
// pair (o, k) of a model voxel o and one of its 27 offsets k inserts its cell and takes the cell's order key
// 27 o + k with atomicMin; the candidate cells then insert their other 7 corners, and each lattice point is evaluated
// once against the alignment's cell index of the model (AlignWorkspace::index).  The flag of (o, k) is set when (o, k)
// owns (has the smallest key of) an active cell, so the compaction's k_count + k_scan over the 27 max_voxels flags rank
// the vertices by their key whatever the hash or the scheduling did.  Faces are counted per block of SURFACE_VB
// vertices and scanned; the emission (one thread per vertex) writes each vertex's faces at its block's offset plus
// its rank inside the block.  Inserting stops once more than max_points slots are taken (the condition is reported at
// the entry's synchronisation), so an undersized max_points can neither hang nor overrun the table.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "../common/scan3d_surface_math.h"

namespace s3d {

namespace {

constexpr int ST = 256;                                 // threads per block of the table kernels
constexpr int SURFACE_VB = 256;                         // vertices per block of the face counts and the emission
constexpr unsigned FULL = 0xffffffffu;
constexpr unsigned long long NO_OWNER = ~0ull;
static_assert(SURFACE_VB % 32 == 0 && SURFACE_VB <= 1024, "vertex block");

__device__ __forceinline__ bool has_normal(const float* nrm, uint32_t o)
{
    return nrm[3 * (size_t)o] != 0.0f || nrm[3 * (size_t)o + 1] != 0.0f || nrm[3 * (size_t)o + 2] != 0.0f;
}

__device__ __forceinline__ void key_cell(unsigned long long key, long long g[3])
{
    g[0] = s3v::key_axis(key, 0);
    g[1] = s3v::key_axis(key, 1);
    g[2] = s3v::key_axis(key, 2);
}

// the cell g of pair idx = 27 o + k: false when o is not a model voxel or a corner of g is outside the key range.  The
// model voxel's own merge index is its key in the accumulator.
__device__ __forceinline__ bool pair_cell(const VoxelTable& t, int par, const float* nrm, unsigned long long idx,
                                          long long g[3])
{
    const unsigned long long o = idx / s3s::OFFSETS;
    const uint32_t m = min(t.state->total[par], t.max_voxels);
    if (o >= m || !has_normal(nrm, (uint32_t)o)) return false;
    int d[3];
    s3s::offset_of((int)(idx - o * s3s::OFFSETS), d);
    key_cell(t.keys[t.ord2slot[o]], g);
    for (int x = 0; x < 3; x++) {
        g[x] += d[x];
        if (g[x] < s3v::I_MIN || g[x] + 1 >= s3v::I_MAX) return false;
    }
    return true;
}

__device__ __forceinline__ uint32_t lattice_insert(const SurfaceTable& s, long long a, long long b, long long c,
                                                   uint32_t* claims)
{
    bool claimed;
    const uint32_t slot = find_or_insert(s.keys, s.cap, s3v::pack_key(a, b, c), &claimed);
    if (slot == VOXEL_NO_SLOT) s.state->overflow = 1;
    else if (claimed) atomicAdd(claims, 1u);
    return slot;
}

// the slots and values of the 8 corners of cell g (slot0 = g's own); false when one is not held or undefined
__device__ __forceinline__ bool corners(const SurfaceTable& s, const long long g[3], uint32_t slot0, double f[8],
                                        uint32_t sl[8])
{
#pragma unroll
    for (int c = 0; c < 8; c++) {
        const uint32_t q = c == 0 ? slot0
                                  : find_slot(s.keys, s.cap, s3v::pack_key(g[0] + (c & 1), g[1] + ((c >> 1) & 1),
                                                                           g[2] + (c >> 2)));
        if (q == VOXEL_NO_SLOT || s.nearest[q] == VOXEL_NO_SLOT) return false;
        sl[c] = q;
        f[c] = s.f[q];
    }
    return true;
}

// the quads of active cell g: bit a is set when lattice edge g -> g + e_a has one; nb[a] = the slots of its 4 cells
__device__ __forceinline__ int cell_quads(const SurfaceTable& s, const long long g[3], uint32_t slot, double f0,
                                          uint32_t nb[3][4])
{
    int mask = 0;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        long long h[3] = {g[0], g[1], g[2]};
        h[a] += 1;
        const uint32_t up = find_slot(s.keys, s.cap, s3v::pack_key(h[0], h[1], h[2]));
        if (up == VOXEL_NO_SLOT || s3s::inside(s.f[up]) == s3s::inside(f0)) continue;
        int off[4][3];
        s3s::quad_cells(a, off);
        bool ok = true;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            if (c == 2) {
                nb[a][c] = slot;
                continue;
            }
            const long long x = g[0] + off[c][0], y = g[1] + off[c][1], z = g[2] + off[c][2];
            const uint32_t q = x < s3v::I_MIN || y < s3v::I_MIN || z < s3v::I_MIN
                                   ? VOXEL_NO_SLOT
                                   : find_slot(s.keys, s.cap, s3v::pack_key(x, y, z));
            ok = ok && q != VOXEL_NO_SLOT && s.vert[q] != VOXEL_NO_SLOT;
            nb[a][c] = q;
        }
        if (ok) mask |= 1 << a;
    }
    return mask;
}

}  // namespace

// every (o, k): insert cell g and take its order key
__global__ void __launch_bounds__(ST) k_surface_cells(SurfaceTable s, VoxelTable t, int par, const float* __restrict__ nrm,
                                                      unsigned long long n)
{
    __shared__ uint32_t s_claims;
    __shared__ int s_stop;
    if (threadIdx.x == 0) {
        s_claims = 0;
        s_stop = *(volatile uint32_t*)&s.state->occupied > s.max_points;
    }
    __syncthreads();
    const unsigned long long idx = (unsigned long long)blockIdx.x * ST + threadIdx.x;
    long long g[3];
    if (!s_stop && idx < n && pair_cell(t, par, nrm, idx, g)) {
        const uint32_t slot = lattice_insert(s, g[0], g[1], g[2], &s_claims);
        if (slot != VOXEL_NO_SLOT) atomicMin(&s.owner[slot], idx);
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_claims) atomicAdd(&s.state->occupied, s_claims);
}

// every candidate cell: insert its other 7 corners
__global__ void __launch_bounds__(ST) k_surface_corners(SurfaceTable s)
{
    __shared__ uint32_t s_claims;
    __shared__ int s_stop;
    if (threadIdx.x == 0) {
        s_claims = 0;
        s_stop = *(volatile uint32_t*)&s.state->occupied > s.max_points;
    }
    __syncthreads();
    const uint32_t i = blockIdx.x * ST + threadIdx.x;
    if (!s_stop && i < s.cap && s.owner[i] != NO_OWNER) {
        long long g[3];
        key_cell(s.keys[i], g);
        for (int c = 1; c < 8; c++) lattice_insert(s, g[0] + (c & 1), g[1] + ((c >> 1) & 1), g[2] + (c >> 2), &s_claims);
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_claims) atomicAdd(&s.state->occupied, s_claims);
}

// every lattice point: f and its nearest model point, once
__global__ void __launch_bounds__(ST) k_surface_eval(SurfaceTable s, AlignIndex ix, double Sa, double r2)
{
    __shared__ uint32_t s_undef;
    if (threadIdx.x == 0) s_undef = 0;
    __syncthreads();
    const uint32_t i = blockIdx.x * ST + threadIdx.x;
    const unsigned long long key = i < s.cap ? s.keys[i] : s3v::EMPTY_KEY;
    if (key != s3v::EMPTY_KEY) {
        long long g[3];
        key_cell(key, g);
        double x[3];
        s3s::lattice_pos(g[0], g[1], g[2], s.S, x);
        uint32_t e;
        const uint32_t o = align_nearest(ix, x, Sa, r2, &e);
        if (o != VOXEL_NO_SLOT) {
            const float4 q = ix.entries[2 * (size_t)e], nq = ix.entries[2 * (size_t)e + 1];
            s.f[i] = s3l::residual(x, q.x, q.y, q.z, nq.x, nq.y, nq.z);
        } else {
            atomicAdd(&s_undef, 1u);
        }
        s.nearest[i] = o;
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_undef) atomicAdd(&s.state->undefined, (unsigned long long)s_undef);
}

// flags[27 o + k] = (o, k) owns an active cell; the cell is marked active (vert = 0 until its ordinal is known)
__global__ void __launch_bounds__(ST) k_surface_flag(SurfaceTable s, VoxelTable t, int par, const float* __restrict__ nrm,
                                                     unsigned long long n, uint8_t* __restrict__ flags)
{
    const unsigned long long idx = (unsigned long long)blockIdx.x * ST + threadIdx.x;
    if (idx >= n) return;
    uint8_t flag = 0;
    long long g[3];
    if (pair_cell(t, par, nrm, idx, g)) {
        const uint32_t slot = find_slot(s.keys, s.cap, s3v::pack_key(g[0], g[1], g[2]));
        double f[8];
        uint32_t sl[8];
        if (slot != VOXEL_NO_SLOT && s.owner[slot] == idx && corners(s, g, slot, f, sl) && s3s::mixed(f)) {
            flag = 1;
            s.vert[slot] = 0;
        }
    }
    flags[idx] = flag;
}

// vertex ordinal = rank of the flag (block b of POINT_BLOCK flags starts at offsets[b]); the faces of each vertex are
// added to the count of its block of SURFACE_VB vertices
__global__ void __launch_bounds__(POINT_BLOCK) k_surface_assign(SurfaceTable s, VoxelTable t, int par,
                                                                const float* __restrict__ nrm, unsigned long long n,
                                                                const uint8_t* __restrict__ flags,
                                                                const uint32_t* __restrict__ offsets,
                                                                uint32_t* __restrict__ vert_slot,
                                                                uint32_t* __restrict__ face_counts)
{
    __shared__ uint32_t wsum[POINT_BLOCK / 32];
    const unsigned long long idx = (unsigned long long)blockIdx.x * POINT_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool fl = idx < n && flags[idx] != 0;
    const unsigned b = __ballot_sync(FULL, fl);
    if (lane == 0) wsum[w] = __popc(b);
    __syncthreads();
    if (!fl) return;
    uint32_t before = 0;
    for (int k = 0; k < w; k++) before += wsum[k];
    const uint32_t r = offsets[blockIdx.x] + before + __popc(b & ((1u << lane) - 1));
    long long g[3];
    pair_cell(t, par, nrm, idx, g);
    const uint32_t slot = find_slot(s.keys, s.cap, s3v::pack_key(g[0], g[1], g[2]));
    if (r >= s.max_points) {
        s.state->overflow = 1;
        return;
    }
    s.vert[slot] = r;
    vert_slot[r] = slot;
    uint32_t nb[3][4];
    const int nf = 2 * __popc(cell_quads(s, g, slot, s.f[slot], nb));
    if (nf) atomicAdd(&face_counts[r / SURFACE_VB], (uint32_t)nf);
}

// one thread per vertex: position, normal, colour and the vertex's faces
__global__ void __launch_bounds__(SURFACE_VB) k_surface_emit(SurfaceTable s, const uint8_t* __restrict__ vox_rgb,
                                                             const uint32_t* __restrict__ vert_slot,
                                                             const uint32_t* __restrict__ face_offsets, uint32_t vertices,
                                                             float* __restrict__ xyz, float* __restrict__ nrm,
                                                             uint8_t* __restrict__ rgb, int32_t* __restrict__ faces)
{
    __shared__ uint32_t wsum[SURFACE_VB / 32];
    const uint32_t r = blockIdx.x * SURFACE_VB + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int mask = 0;
    uint32_t nb[3][4];
    double f[8];
    if (r < vertices) {
        const uint32_t slot = vert_slot[r];
        long long g[3];
        key_cell(s.keys[slot], g);
        uint32_t sl[8];
        corners(s, g, slot, f, sl);
        float v[3], nv[3];
        s3s::vertex_position(g, f, s.S, v);
        s3s::gradient_normal(f, nv);
        unsigned sum[3] = {0u, 0u, 0u};
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const size_t o = s.nearest[sl[c]];
#pragma unroll
            for (int k = 0; k < 3; k++) sum[k] += vox_rgb[3 * o + k];
        }
#pragma unroll
        for (int k = 0; k < 3; k++) {
            xyz[3 * (size_t)r + k] = v[k];
            nrm[3 * (size_t)r + k] = nv[k];
            rgb[3 * (size_t)r + k] = s3s::colour(sum[k]);
        }
        mask = cell_quads(s, g, slot, f[0], nb);
    }
    const uint32_t nf = 2 * __popc(mask);
    uint32_t incl = nf;                                  // inclusive prefix sum over the warp, then over the warps
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t x = __shfl_up_sync(FULL, incl, off);
        if (lane >= off) incl += x;
    }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    uint32_t base = face_offsets[blockIdx.x] + incl - nf;
    for (int k = 0; k < w; k++) base += wsum[k];
    if (!mask) return;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        if (!(mask >> a & 1)) continue;
        int v[4], tri[6];
#pragma unroll
        for (int c = 0; c < 4; c++) v[c] = (int)s.vert[nb[a][c]];
        s3s::quad_triangles(v, s3s::inside(f[0]), tri);
#pragma unroll
        for (int k = 0; k < 6; k++) faces[3 * (size_t)base + k] = tri[k];
        base += 2;
    }
}

// slots of the lattice table for max_points: at most half of them are ever taken
static uint32_t surface_table_capacity(uint32_t max_points, int sm_count)
{
    // Inserting stops once more than max_points slots are taken.  Blocks that passed that check before claim at most
    // one slot per thread (cells) or seven (corners): the crossing block and every resident one (2048 threads per SM).
    // Twice that bound keeps the table at most half full, so probe sequences stay short and always end.
    const unsigned long long c = 2ull * ((unsigned long long)max_points + 7ull * (2048ull * (unsigned)sm_count + ST));
    return (uint32_t)(c < 0xffffffffull ? c : 0xffffffffull);
}

cudaError_t SurfaceWorkspace::count(const AlignIndex& ix, const VoxelTable& t, int par, const float* vox_nrm,
                                    float max_distance, uint32_t max_points, int sm_count, cudaStream_t st,
                                    int64_t* launches)
{
    const uint32_t cap = surface_table_capacity(max_points, sm_count);
    const size_t nvb = (max_points + SURFACE_VB - 1) / SURFACE_VB;
    const unsigned long long n = (unsigned long long)s3s::OFFSETS * t.max_voxels;
    cudaError_t e = grow_group(Grow(keys, cap), Grow(owner, cap), Grow(f, cap), Grow(nearest, cap), Grow(vert, cap));
    if (e == cudaSuccess) e = grow_group(Grow(vert_slot, max_points), Grow(face_counts, nvb + 1));
    if (e == cudaSuccess) e = grow_group(Grow(flags, n), Grow(flag_counts, (n + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    if (e == cudaSuccess) e = state.ensure(1);
    if (e != cudaSuccess) return e;
    view = SurfaceTable{keys, owner, f, nearest, vert, state, cap, max_points, t.S};
    e = cudaMemsetAsync(keys, 0xff, (size_t)cap * sizeof(*view.keys), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(owner, 0xff, (size_t)cap * sizeof(*view.owner), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(vert, 0xff, (size_t)cap * sizeof(*view.vert), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(state, 0, sizeof(*view.state), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(face_counts, 0, nvb * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    const SurfaceTable& s = view;
    const unsigned gp = (unsigned)((n + ST - 1) / ST), gs = (unsigned)((s.cap + (unsigned long long)ST - 1) / ST);
    const double R = (double)max_distance;
    k_surface_cells<<<gp, ST, 0, st>>>(s, t, par, vox_nrm, n);
    k_surface_corners<<<gs, ST, 0, st>>>(s);
    k_surface_eval<<<gs, ST, 0, st>>>(s, ix, s3l::cell_edge(max_distance), R * R);
    k_surface_flag<<<gp, ST, 0, st>>>(s, t, par, vox_nrm, n, flags);
    e = launch_point_offsets(flags, (size_t)n, flag_counts, &s.state->vertices, st);
    if (e != cudaSuccess) return e;
    k_surface_assign<<<(unsigned)((n + POINT_BLOCK - 1) / POINT_BLOCK), POINT_BLOCK, 0, st>>>(
        s, t, par, vox_nrm, n, flags, flag_counts, vert_slot, face_counts);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    e = launch_block_scan(face_counts, (int)nvb, &s.state->faces, st);
    *launches += 8;
    return e;
}

cudaError_t SurfaceWorkspace::emit(const uint8_t* vox_rgb, uint32_t vertices, SurfaceMesh& out, cudaStream_t st,
                                   int64_t* launches)
{
    const unsigned blocks = vertices ? (vertices + SURFACE_VB - 1) / SURFACE_VB : 1;
    k_surface_emit<<<blocks, SURFACE_VB, 0, st>>>(view, vox_rgb, vert_slot, face_counts, vertices, out.xyz, out.nrm,
                                                  out.rgb, out.tri);
    *launches += 1;
    return cudaGetLastError();
}

}  // namespace s3d
