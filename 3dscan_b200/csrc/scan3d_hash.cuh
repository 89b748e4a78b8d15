// scan3d_hash.cuh -- the open-addressing hash of 63-bit keys (s3v::pack_key) shared by the voxel-grid merge
// (scan3d_voxel_kernels.cu), the alignment's cell index (scan3d_align_kernels.cu) and the surface's lattice table
// (scan3d_surface_kernels.cu), and the undirected-edge tables of the smoothing and the hole filling (edge_key): linear
// probing over a 64-bit key array whose free slots hold s3v::EMPTY_KEY.  The callers size their tables so that at most
// half the slots are taken, which keeps probe sequences short and makes them end.  Also the nearest-model-point search
// of the cell index, shared by the alignment and the surface.
#pragma once
#include "scan3d_internal.h"
#include "../common/scan3d_align_math.h"

namespace s3d {

// splitmix64's finaliser: the table position must not follow the raster order of the keys
__device__ __forceinline__ unsigned long long mix64(unsigned long long x)
{
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

__device__ __forceinline__ uint32_t hash_home(unsigned long long key, uint32_t cap)
{
    return (uint32_t)(((mix64(key) >> 32) * (unsigned long long)cap) >> 32);
}

// the key of the undirected edge {a, b}: (min << 32) | max (the smoothing's and the hole filling's edge tables)
__device__ __forceinline__ unsigned long long edge_key(uint32_t a, uint32_t b)
{
    return a < b ? (unsigned long long)a << 32 | b : (unsigned long long)b << 32 | a;
}

// The key's slot, inserting it if absent.  At most cap probes, so a full table cannot hang the caller.
// *claimed = this call took a new slot.  VOXEL_NO_SLOT if the table is full.
__device__ __forceinline__ uint32_t find_or_insert(unsigned long long* keys, uint32_t cap, unsigned long long key,
                                                   bool* claimed)
{
    uint32_t s = hash_home(key, cap);
    *claimed = false;
    for (uint32_t p = 0; p < cap; p++) {
        unsigned long long k = __ldcg(keys + s);   // keys never change once set: a stale EMPTY only costs a CAS
        if (k == s3v::EMPTY_KEY) {
            k = atomicCAS(keys + s, s3v::EMPTY_KEY, key);
            if (k == s3v::EMPTY_KEY) {
                *claimed = true;
                return s;
            }
        }
        if (k == key) return s;
        s = s + 1 == cap ? 0 : s + 1;
    }
    return VOXEL_NO_SLOT;
}

// The key's slot in a table no kernel is inserting into, VOXEL_NO_SLOT if absent.
__device__ __forceinline__ uint32_t find_slot(const unsigned long long* __restrict__ keys, uint32_t cap,
                                              unsigned long long key)
{
    uint32_t s = hash_home(key, cap);
    for (uint32_t p = 0; p < cap; p++) {
        const unsigned long long k = keys[s];
        if (k == key) return s;
        if (k == s3v::EMPTY_KEY) return VOXEL_NO_SLOT;
        s = s + 1 == cap ? 0 : s + 1;
    }
    return VOXEL_NO_SLOT;
}

// The exact nearest model point to p within r2 in the alignment's cell index (AlignWorkspace::index, cell edge S): the
// smallest s3l::dist2, a tie going to the smaller ordinal.  Returns its ordinal and sets *entry to its entry, or
// VOXEL_NO_SLOT when no model point qualifies.
__device__ __forceinline__ uint32_t align_nearest(const AlignIndex& ix, const double p[3], double S, double r2,
                                                  uint32_t* entry)
{
    long long c[3];
    if (!s3l::cell_of(p, S, c)) return VOXEL_NO_SLOT;
    double best = 0.0;
    uint32_t best_o = VOXEL_NO_SLOT, best_e = 0;
    for (int dz = -1; dz <= 1; dz++)
        for (int dy = -1; dy <= 1; dy++)
            for (int dx = -1; dx <= 1; dx++) {
                const long long a = c[0] + dx, b = c[1] + dy, e = c[2] + dz;
                if (a < s3v::I_MIN || a >= s3v::I_MAX || b < s3v::I_MIN || b >= s3v::I_MAX || e < s3v::I_MIN ||
                    e >= s3v::I_MAX)
                    continue;
                const uint32_t slot = find_slot(ix.keys, ix.cap, s3v::pack_key(a, b, e));
                if (slot == VOXEL_NO_SLOT) continue;
                const uint2 cell = ix.cells[slot];
                for (uint32_t u = cell.y - cell.x; u < cell.y; u++) {
                    const float4 q = ix.entries[2 * (size_t)u];
                    const double d = s3l::dist2(p, q.x, q.y, q.z);
                    const uint32_t o = __float_as_uint(q.w);
                    if (d <= r2 && (best_o == VOXEL_NO_SLOT || s3l::closer(d, o, best, best_o))) {
                        best = d;
                        best_o = o;
                        best_e = u;
                    }
                }
            }
    *entry = best_e;
    return best_o;
}

}  // namespace s3d
