// scan3d_hash.cuh -- the open-addressing hash of 63-bit keys (s3v::pack_key) shared by the voxel-grid merge
// (scan3d_voxel_kernels.cu) and the alignment's cell index (scan3d_align_kernels.cu): linear probing over a 64-bit key
// array whose free slots hold s3v::EMPTY_KEY.  Both callers size their tables so that at most half the slots are taken,
// which keeps probe sequences short and makes them end.
#pragma once
#include "scan3d_internal.h"
#include "../common/scan3d_voxel_math.h"

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

}  // namespace s3d
