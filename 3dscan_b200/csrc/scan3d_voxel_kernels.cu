// scan3d_voxel_kernels.cu -- the voxel-grid merge of registered views (scan3d_voxel_*): one output point per occupied
// voxel, averaged over every point of every add that fell into it.  The arithmetic is in common/scan3d_voxel_math.h,
// shared with the host test; this file owns the hash table and the output order.
//
// The table is open addressing with linear probing over a 64-bit key array; each slot has integer accumulators
// (VoxelSlot), so concurrent atomics commute and the sums do not depend on scheduling.  Output order is the order of
// each voxel's first point: an add (or chunk) gives its new voxels the ordinals voxels_so_far + rank, where rank
// orders them by their first point inside the add.  That takes a grid-wide step after the inserts, so an add is
// 5 launches: insert, flag, the compaction's k_count + k_scan over the flags, assign.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "../common/scan3d_voxel_math.h"

namespace s3d {

namespace {

constexpr int VT = 256;                 // threads per block of the insert / flag kernels
constexpr unsigned FULL = 0xffffffffu;

}  // namespace

// One thread per point.  Lanes whose points share a voxel (consecutive raster points usually do) are grouped with
// __match_any_sync on the key; the group's lowest lane probes the table once and adds the group's sums with one set
// of atomics.  A warp's sums fit 32 bits (32 * 2^24 for positions and normals, 32 * 255 for colours).
__global__ void __launch_bounds__(VT) k_voxel_insert(VoxelTable t, const float* __restrict__ xyz,
                                                     const float* __restrict__ nrm, const uint8_t* __restrict__ rgb,
                                                     const uint32_t* __restrict__ n_dev, uint32_t plane,
                                                     uint32_t* __restrict__ point_slot)
{
    __shared__ uint32_t s_claims;
    __shared__ int s_stop;
    if (threadIdx.x == 0) {
        s_claims = 0;
        // past the capacity: stop inserting (the condition is reported by the getters), so the table never fills
        s_stop = *(volatile uint32_t*)&t.state->occupied > t.max_voxels;
    }
    __syncthreads();
    const uint32_t n = n_dev ? min(*n_dev, plane) : plane;
    const uint32_t i = blockIdx.x * VT + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool live = i < n;
    unsigned long long key = s3v::EMPTY_KEY, q[3] = {0, 0, 0};
    long long m[3] = {0, 0, 0};
    uint32_t c[3] = {0, 0, 0};
    bool ok = false;
    if (live) {
        ok = s3v::point_key(xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], t.S, &key, q);
        if (nrm) s3v::normal_fixed(nrm[3 * (size_t)i], nrm[3 * (size_t)i + 1], nrm[3 * (size_t)i + 2], m);
        if (rgb) {
            c[0] = rgb[3 * (size_t)i];
            c[1] = rgb[3 * (size_t)i + 1];
            c[2] = rgb[3 * (size_t)i + 2];
        }
    }
    const unsigned dropped = __ballot_sync(FULL, live && !ok);
    if (lane == 0 && dropped) atomicAdd(&t.state->dropped, (unsigned long long)__popc(dropped));
    const bool has = ok && !s_stop;
    if (!has) key = s3v::EMPTY_KEY;
    const unsigned grp = __match_any_sync(FULL, key);
    const int leader = __ffs(grp) - 1;
    uint32_t slot = VOXEL_NO_SLOT;
    if (has && lane == leader) {
        bool claimed;
        slot = find_or_insert(t.keys, t.cap, key, &claimed);
        if (claimed) atomicAdd(&s_claims, 1u);
    }
    slot = __shfl_sync(FULL, slot, leader);
    uint32_t sq[3], sm[3], sc[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        sq[k] = __reduce_add_sync(grp, (uint32_t)q[k]);
        sm[k] = __reduce_add_sync(grp, (uint32_t)(int32_t)m[k]);   // two's complement: the int32 sum is exact
        sc[k] = __reduce_add_sync(grp, c[k]);
    }
    if (has && lane == leader && slot != VOXEL_NO_SLOT) {
        VoxelSlot* a = t.acc + slot;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            atomicAdd(&a->q[k], (unsigned long long)sq[k]);
            if (nrm) atomicAdd(&a->m[k], (unsigned long long)(long long)(int32_t)sm[k]);
            if (rgb) atomicAdd(&a->c[k], (unsigned long long)sc[k]);
        }
        atomicAdd(&a->n, (uint32_t)__popc(grp));
        atomicMax(&a->first_inv, ~i);   // the group's first point is its lowest lane
    }
    if (live) point_slot[i] = has ? slot : VOXEL_NO_SLOT;
    __syncthreads();
    if (threadIdx.x == 0 && s_claims) atomicAdd(&t.state->occupied, s_claims);
}

// flag[i] = point i is the first point of a voxel that has no ordinal yet
__global__ void __launch_bounds__(VT) k_voxel_flag(VoxelTable t, const uint32_t* __restrict__ n_dev, uint32_t plane,
                                                   const uint32_t* __restrict__ point_slot, uint8_t* __restrict__ flags)
{
    const uint32_t i = blockIdx.x * VT + threadIdx.x;
    if (i >= plane) return;
    const uint32_t n = n_dev ? min(*n_dev, plane) : plane;
    uint8_t f = 0;
    if (i < n) {
        const uint32_t s = point_slot[i];
        f = s != VOXEL_NO_SLOT && t.ordinal[s] == VOXEL_NO_SLOT && t.acc[s].first_inv == ~i;
    }
    flags[i] = f;
}

// ordinal = voxels so far + rank of the flagged point; block b of POINT_BLOCK flags starts at offsets[b].  The running
// total ping-pongs between state->total[par] (read) and [par ^ 1] (written once), so no block reads a value another
// block of this launch writes.
__global__ void __launch_bounds__(POINT_BLOCK) k_voxel_assign(VoxelTable t, const uint8_t* __restrict__ flags,
                                                              uint32_t plane, const uint32_t* __restrict__ offsets,
                                                              const uint32_t* __restrict__ point_slot, int par)
{
    __shared__ uint32_t wsum[POINT_BLOCK / 32];
    const uint32_t i = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool f = i < plane && flags[i] != 0;
    const unsigned b = __ballot_sync(FULL, f);
    if (lane == 0) wsum[w] = __popc(b);
    __syncthreads();
    const uint32_t base = t.state->total[par];
    if (f) {
        uint32_t before = 0;
        for (int k = 0; k < w; k++) before += wsum[k];
        const uint32_t ord = base + offsets[blockIdx.x] + before + __popc(b & ((1u << lane) - 1));
        const uint32_t s = point_slot[i];
        t.ordinal[s] = ord;
        if (ord < t.max_voxels) t.ord2slot[ord] = s;
        else t.state->overflow = 1;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) t.state->total[par ^ 1] = base + t.state->chunk_new;
}

// the merged voxels in ordinal order
__global__ void k_voxel_finish(VoxelTable t, int par, float* __restrict__ out_xyz, float* __restrict__ out_nrm,
                               uint8_t* __restrict__ out_rgb, uint32_t* __restrict__ out_cnt)
{
    const uint32_t total = min(t.state->total[par], t.max_voxels);
    for (uint32_t o = blockIdx.x * blockDim.x + threadIdx.x; o < total; o += gridDim.x * blockDim.x) {
        const uint32_t s = t.ord2slot[o];
        const unsigned long long key = t.keys[s];
        const VoxelSlot a = t.acc[s];
        for (int k = 0; k < 3; k++) {
            out_xyz[3 * (size_t)o + k] = s3v::coord(key, k, a.q[k], a.n, t.S);
            out_rgb[3 * (size_t)o + k] = s3v::colour(a.c[k], a.n);
        }
        s3v::normal_out((long long)a.m[0], (long long)a.m[1], (long long)a.m[2], out_nrm + 3 * (size_t)o);
        out_cnt[o] = a.n;
    }
}

uint32_t voxel_table_capacity(uint32_t max_voxels, int sm_count)
{
    // k_voxel_insert stops claiming slots once more than max_voxels are taken.  Blocks that passed that check before
    // claim at most one slot per thread: the crossing block and every resident one (2048 threads per SM).  Twice
    // that bound keeps the table at most half full, so probe sequences stay short and always end.
    const unsigned long long c = 2ull * ((unsigned long long)max_voxels + 2048ull * (unsigned)sm_count + VT);
    return (uint32_t)(c < 0xffffffffull ? c : 0xffffffffull);
}

cudaError_t launch_voxel_add(const VoxelTable& t, const float* xyz, const float* nrm, const uint8_t* rgb,
                             const uint32_t* n_dev, uint32_t plane, uint32_t* point_slot, uint8_t* flags,
                             uint32_t* block_counts, int par, cudaStream_t st)
{
    const unsigned grid = (unsigned)((plane + VT - 1) / VT);
    k_voxel_insert<<<grid, VT, 0, st>>>(t, xyz, nrm, rgb, n_dev, plane, point_slot);
    k_voxel_flag<<<grid, VT, 0, st>>>(t, n_dev, plane, point_slot, flags);
    cudaError_t e = launch_point_offsets(flags, plane, block_counts, &t.state->chunk_new, st);
    if (e != cudaSuccess) return e;
    k_voxel_assign<<<(unsigned)((plane + POINT_BLOCK - 1) / POINT_BLOCK), POINT_BLOCK, 0, st>>>(t, flags, plane,
                                                                                               block_counts, point_slot, par);
    return cudaGetLastError();
}

cudaError_t launch_voxel_finish(const VoxelTable& t, int par, float* xyz, float* nrm, uint8_t* rgb, uint32_t* cnt,
                                int sm_count, cudaStream_t st)
{
    k_voxel_finish<<<4 * sm_count, 256, 0, st>>>(t, par, xyz, nrm, rgb, cnt);
    return cudaGetLastError();
}

}  // namespace s3d
