// scan3d_union_find.cuh -- the lock-free union-find of ECL-CC (Jaiganesh & Burtscher, HPDC 2018), shared by the
// connected components (scan3d_components_kernels.cu, over vertices) and the non-manifold repair
// (scan3d_repair_kernels.cu, over face corners).
//
// A union links the larger of the two roots under the smaller with atomicCAS and retries from the new roots when
// another thread linked first, so parent[x] <= x always holds and each root is the smallest element of its set whatever
// the interleaving.  The finds use path halving: a non-root's parent only ever moves to another of its ancestors, and a
// CAS only ever targets a root, so the halving stores never race with a link.  parent is read with relaxed atomic
// loads, so a thread always sees the links other threads made.
#pragma once
#include <stdint.h>

#include <cuda/atomic>

namespace s3d {

__device__ __forceinline__ uint32_t load_parent(uint32_t* parent, uint32_t x)
{
    return cuda::atomic_ref<uint32_t, cuda::thread_scope_device>(parent[x]).load(cuda::memory_order_relaxed);
}

__device__ __forceinline__ void store_parent(uint32_t* parent, uint32_t x, uint32_t p)
{
    cuda::atomic_ref<uint32_t, cuda::thread_scope_device>(parent[x]).store(p, cuda::memory_order_relaxed);
}

// the root of x, halving the path on the way
__device__ __forceinline__ uint32_t find(uint32_t* parent, uint32_t x)
{
    for (;;) {
        const uint32_t p = load_parent(parent, x);
        if (p == x) return x;
        const uint32_t g = load_parent(parent, p);
        if (g == p) return p;
        store_parent(parent, x, g);
        x = g;
    }
}

__device__ __forceinline__ void unite(uint32_t* parent, uint32_t a, uint32_t b)
{
    a = find(parent, a);
    b = find(parent, b);
    while (a != b) {
        if (a > b) {
            const uint32_t t = a;
            a = b;
            b = t;
        }
        const uint32_t old = atomicCAS(&parent[b], b, a);
        if (old == b) return;
        a = find(parent, a);
        b = find(parent, old);
    }
}

}  // namespace s3d
