// scan3d_components_kernels.cu -- connected components of a triangle mesh (scan3d_voxel_surface_components,
// scan3d_mesh_components_dev) and the compaction of the held voxel surface to its kept components.
//
// Labels: the lock-free union-find of scan3d_union_find.cuh (ECL-CC) over the vertices.  Every face unites its first
// vertex with the other two.  Each root is the smallest vertex of its component whatever the interleaving, and the
// flags "v is a root" ranked by k_count + k_scan give the ids (rank of the smallest vertex).
//
// Selection: one block finds the threshold key K of the keep rule by a radix select over key(c) = faces << 32 |
// (2^32 - 1 - c), which orders the components by faces descending and then by id ascending with no two keys equal.
// The kept components are the eligible ones (faces >= min_faces) with key >= K.  Counts are integer atomics and the
// selection works on integers only, so every output is a pure function of the mesh.
#include "scan3d_internal.h"
#include "scan3d_union_find.cuh"

namespace s3d {

namespace {

constexpr int CT = 256;                                 // threads per block of the union-find kernels
constexpr int SELECT_THREADS = 1024;
constexpr unsigned FULL = 0xffffffffu;
static_assert(POINT_BLOCK == 1024, "the emission kernels rank one flag per thread of a POINT_BLOCK block");

__device__ __forceinline__ unsigned long long key_of(uint32_t faces, uint32_t c)
{
    return (unsigned long long)faces << 32 | (unsigned long long)(0xffffffffu - c);
}

__device__ __forceinline__ bool keep_component(const uint32_t* comp_f, const ComponentsState* st, uint32_t c,
                                               unsigned long long min_faces)
{
    const uint32_t f = comp_f[c];
    return f >= min_faces && key_of(f, c) >= st->threshold;
}

}  // namespace

__global__ void __launch_bounds__(CT) k_cc_init(uint32_t* __restrict__ parent, uint32_t n)
{
    const uint32_t v = blockIdx.x * CT + threadIdx.x;
    if (v < n) parent[v] = v;
}

// one thread per face: union(v0, v1), union(v0, v2); a face with an index outside [0, n) sets st->bad and is skipped
__global__ void __launch_bounds__(CT) k_cc_hook(const int32_t* __restrict__ faces, uint32_t n_faces, uint32_t n,
                                                uint32_t* parent, ComponentsState* st)
{
    const uint32_t f = blockIdx.x * CT + threadIdx.x;
    if (f >= n_faces) return;
    const int32_t a = faces[3 * (size_t)f], b = faces[3 * (size_t)f + 1], c = faces[3 * (size_t)f + 2];
    if ((uint32_t)a >= n || (uint32_t)b >= n || (uint32_t)c >= n) {
        st->bad = 1;
        return;
    }
    unite(parent, (uint32_t)a, (uint32_t)b);
    unite(parent, (uint32_t)a, (uint32_t)c);
}

// parent[v] = the root of v; flags[v] = v is a root.  The walk does not halve: a halving store could overwrite the
// root another thread has just stored with an ancestor that is not the root.  The only stores here are roots.
__global__ void __launch_bounds__(CT) k_cc_compress(uint32_t* parent, uint8_t* __restrict__ flags, uint32_t n)
{
    const uint32_t v = blockIdx.x * CT + threadIdx.x;
    if (v >= n) return;
    uint32_t r = v, p;
    while ((p = load_parent(parent, r)) != r) r = p;
    store_parent(parent, v, r);
    flags[v] = r == v;
}

// every root writes its id: the rank of its flag (block b of POINT_BLOCK flags starts at offsets[b])
__global__ void __launch_bounds__(POINT_BLOCK) k_cc_root_ids(const uint8_t* __restrict__ flags,
                                                             const uint32_t* __restrict__ offsets, uint32_t n,
                                                             int32_t* __restrict__ label)
{
    const uint32_t v = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const bool root = v < n && flags[v] != 0;
    const uint32_t r = block_rank(root);
    if (root) label[v] = (int32_t)(offsets[blockIdx.x] + r);
}

// every other vertex reads its root's id
__global__ void __launch_bounds__(CT) k_cc_labels(const uint32_t* __restrict__ parent, uint32_t n, int32_t* label)
{
    const uint32_t v = blockIdx.x * CT + threadIdx.x;
    if (v >= n) return;
    const uint32_t r = parent[v];
    if (r != v) label[v] = label[r];
}

// count[c] += the lanes of the warp whose c is the same (c < 0: none); every lane of the warp calls it.  Neighbouring
// vertices and faces mostly share a component, so one atomic per distinct c keeps a large component's counters from
// serialising the whole grid.
__device__ __forceinline__ void add_per_warp(uint32_t* count, int32_t c)
{
    const unsigned m = __match_any_sync(FULL, c);
    if (c >= 0 && (int)(threadIdx.x & 31) == __ffs(m) - 1) atomicAdd(&count[c], (uint32_t)__popc(m));
}

// vertices and faces per component (a face counts for the component of its first vertex)
__global__ void __launch_bounds__(CT) k_cc_count(const int32_t* __restrict__ label, const int32_t* __restrict__ faces,
                                                 uint32_t n, uint32_t n_faces, uint32_t* __restrict__ comp_v,
                                                 uint32_t* __restrict__ comp_f)
{
    const uint32_t i = blockIdx.x * CT + threadIdx.x;
    add_per_warp(comp_v, i < n ? label[i] : -1);
    add_per_warp(comp_f, i < n_faces ? label[faces[3 * (size_t)i]] : -1);
}

// one block: st->threshold (K), st->kept and st->largest from the face counts of the st->components components
__global__ void __launch_bounds__(SELECT_THREADS) k_cc_select(const uint32_t* __restrict__ comp_f, ComponentsState* st,
                                                              unsigned long long min_faces,
                                                              unsigned long long max_components)
{
    constexpr int U = 4;                                 // loads in flight per thread
    __shared__ uint32_t hist[256];
    __shared__ unsigned long long s_eligible, s_prefix, s_need;
    __shared__ uint32_t s_largest;
    __shared__ int s_done;
    const uint32_t C = st->components;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        s_eligible = 0;
        s_largest = 0;
    }
    __syncthreads();
    uint32_t eligible = 0, largest = 0;
    for (uint32_t c = threadIdx.x; c < C; c += SELECT_THREADS) {
        const uint32_t f = comp_f[c];
        eligible += f >= min_faces;
        largest = max(largest, f);
    }
    for (int o = 16; o; o >>= 1) {
        eligible += __shfl_xor_sync(FULL, eligible, o);
        largest = max(largest, __shfl_xor_sync(FULL, largest, o));
    }
    if (lane == 0) {
        atomicAdd(&s_eligible, (unsigned long long)eligible);
        atomicMax(&s_largest, largest);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        s_prefix = 0;                                    // K = 0 keeps every eligible component
        s_need = max_components;
        s_done = max_components == 0 || s_eligible <= max_components;
    }
    __syncthreads();
    // radix select of the max_components-th largest eligible key, 8 bits at a time from the top; it stops early when
    // every key of the chosen bin is kept (K = the bin's smallest key)
    for (int shift = 56; shift >= 0 && !s_done; shift -= 8) {
        for (int b = threadIdx.x; b < 256; b += SELECT_THREADS) hist[b] = 0;
        __syncthreads();
        const unsigned long long hi = shift == 56 ? 0ull : ~0ull << (shift + 8), prefix = s_prefix;
        for (uint32_t base = 0; base < C; base += U * SELECT_THREADS) {   // the same trip count for every thread
            uint32_t f[U];
#pragma unroll
            for (int j = 0; j < U; j++) {
                const uint32_t c = base + j * SELECT_THREADS + threadIdx.x;
                f[j] = c < C ? comp_f[c] : 0u;
            }
#pragma unroll
            for (int j = 0; j < U; j++) {
                const uint32_t c = base + j * SELECT_THREADS + threadIdx.x;
                const unsigned long long k = key_of(f[j], c);
                const int d = c < C && f[j] >= min_faces && (k & hi) == prefix ? (int)(k >> shift & 255) : 256;
                const unsigned m = __match_any_sync(FULL, d);
                if (d < 256 && lane == __ffs(m) - 1) atomicAdd(&hist[d], (uint32_t)__popc(m));
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long need = s_need;
            for (int b = 255; b >= 0; b--) {
                if (need <= hist[b]) {
                    s_prefix = prefix | (unsigned long long)b << shift;
                    s_done = need == hist[b];
                    break;
                }
                need -= hist[b];
            }
            s_need = need;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        st->threshold = s_prefix;
        st->kept = (uint32_t)(max_components && max_components < s_eligible ? max_components : s_eligible);
        st->largest = s_largest;
    }
}

// keep flags of the vertices, the faces and the components
__global__ void __launch_bounds__(CT) k_cc_keep(const int32_t* __restrict__ label, const int32_t* __restrict__ faces,
                                                const uint32_t* __restrict__ comp_f, const ComponentsState* st,
                                                unsigned long long min_faces, uint32_t n, uint32_t n_faces,
                                                uint8_t* __restrict__ keep_v, uint8_t* __restrict__ keep_f,
                                                uint8_t* __restrict__ kept)
{
    const uint32_t i = blockIdx.x * CT + threadIdx.x;
    if (i < n) keep_v[i] = keep_component(comp_f, st, (uint32_t)label[i], min_faces);
    if (i < n_faces) keep_f[i] = keep_component(comp_f, st, (uint32_t)label[faces[3 * (size_t)i]], min_faces);
    if (i < st->components) kept[i] = keep_component(comp_f, st, i, min_faces);
}

// kept vertex v goes to rank r of its keep flag: its bytes are copied and new_index[v] = r
__global__ void __launch_bounds__(POINT_BLOCK) k_cc_emit_vertices(const uint8_t* __restrict__ keep_v,
                                                                  const uint32_t* __restrict__ offsets, uint32_t n,
                                                                  const float* __restrict__ xyz,
                                                                  const float* __restrict__ nrm,
                                                                  const uint8_t* __restrict__ rgb, float* __restrict__ xyz2,
                                                                  float* __restrict__ nrm2, uint8_t* __restrict__ rgb2,
                                                                  int32_t* __restrict__ new_index)
{
    const uint32_t v = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const bool keep = v < n && keep_v[v] != 0;
    const uint32_t r = offsets[blockIdx.x] + block_rank(keep);
    if (!keep) return;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        xyz2[3 * (size_t)r + k] = xyz[3 * (size_t)v + k];
        nrm2[3 * (size_t)r + k] = nrm[3 * (size_t)v + k];
        rgb2[3 * (size_t)r + k] = rgb[3 * (size_t)v + k];
    }
    new_index[v] = (int32_t)r;
}

// kept face f goes to rank r of its keep flag, with its indices remapped
__global__ void __launch_bounds__(POINT_BLOCK) k_cc_emit_faces(const uint8_t* __restrict__ keep_f,
                                                               const uint32_t* __restrict__ offsets, uint32_t n_faces,
                                                               const int32_t* __restrict__ faces,
                                                               const int32_t* __restrict__ new_index,
                                                               int32_t* __restrict__ faces2)
{
    const uint32_t f = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const bool keep = f < n_faces && keep_f[f] != 0;
    const uint32_t r = offsets[blockIdx.x] + block_rank(keep);
    if (!keep) return;
#pragma unroll
    for (int k = 0; k < 3; k++) faces2[3 * (size_t)r + k] = new_index[faces[3 * (size_t)f + k]];
}

namespace {
// at least one block, so that every launch runs for an empty mesh too
unsigned grid(uint32_t n, int threads) { return n ? (unsigned)((n + (uint64_t)threads - 1) / threads) : 1u; }

// the labelling scratch for n vertices, and the state zeroed
cudaError_t reset_labels(ComponentsWorkspace& w, uint32_t n, cudaStream_t st)
{
    const size_t a = n ? n : 1;
    cudaError_t e =
        grow_group(Grow(w.parent, a), Grow(w.flags, a), Grow(w.vert_counts, (a + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    if (e == cudaSuccess) e = w.state.ensure(1);
    if (e == cudaSuccess) e = cudaMemsetAsync(w.state, 0, sizeof(ComponentsState), st);
    return e;
}

cudaError_t launch_labels(ComponentsWorkspace& w, const int32_t* faces, uint32_t n_faces, uint32_t n, int32_t* label,
                          cudaStream_t st, int64_t* launches)
{
    k_cc_init<<<grid(n, CT), CT, 0, st>>>(w.parent, n);
    k_cc_hook<<<grid(n_faces, CT), CT, 0, st>>>(faces, n_faces, n, w.parent, w.state);
    k_cc_compress<<<grid(n, CT), CT, 0, st>>>(w.parent, w.flags, n);
    cudaError_t e = launch_point_offsets(w.flags, n, w.vert_counts, &w.state.get()->components, st);
    if (e != cudaSuccess) return e;
    k_cc_root_ids<<<grid(n, POINT_BLOCK), POINT_BLOCK, 0, st>>>(w.flags, w.vert_counts, n, label);
    k_cc_labels<<<grid(n, CT), CT, 0, st>>>(w.parent, n, label);
    *launches += 7;
    return cudaGetLastError();
}
}  // namespace

cudaError_t ComponentsWorkspace::labels(const int32_t* faces, uint32_t n_faces, uint32_t n, int32_t* out,
                                        cudaStream_t st, int64_t* launches)
{
    const cudaError_t e = reset_labels(*this, n, st);
    return e != cudaSuccess ? e : launch_labels(*this, faces, n_faces, n, out, st, launches);
}

cudaError_t ComponentsWorkspace::select(const SurfaceMesh& in, unsigned long long min_faces,
                                        unsigned long long max_components, cudaStream_t st, int64_t* launches)
{
    const uint32_t n = (uint32_t)in.vertices, n_faces = (uint32_t)in.faces;
    const size_t av = n ? n : 1, af = n_faces ? n_faces : 1;
    cudaError_t e = reset_labels(*this, n, st);
    if (e == cudaSuccess) e = grow_group(Grow(label, av), Grow(comp_v, av), Grow(comp_f, av), Grow(kept, av));
    if (e == cudaSuccess) e = grow_group(Grow(keep_f, af), Grow(face_counts, (af + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    if (e == cudaSuccess) e = cudaMemsetAsync(comp_v, 0, (size_t)n * sizeof(uint32_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(comp_f, 0, (size_t)n * sizeof(uint32_t), st);
    if (e == cudaSuccess) e = launch_labels(*this, in.tri, n_faces, n, label, st, launches);
    if (e != cudaSuccess) return e;
    const uint32_t m = n > n_faces ? n : n_faces;
    k_cc_count<<<grid(m, CT), CT, 0, st>>>(label, in.tri, n, n_faces, comp_v, comp_f);
    k_cc_select<<<1, SELECT_THREADS, 0, st>>>(comp_f, state, min_faces, max_components);
    k_cc_keep<<<grid(m, CT), CT, 0, st>>>(label, in.tri, comp_f, state, min_faces, n, n_faces, flags, keep_f, kept);
    e = launch_point_offsets(flags, n, vert_counts, &state.get()->vertices, st);
    if (e != cudaSuccess) return e;
    *launches += 7;
    return launch_point_offsets(keep_f, n_faces, face_counts, &state.get()->faces, st);
}

cudaError_t ComponentsWorkspace::emit(const SurfaceMesh& in, SurfaceMesh& out, cudaStream_t st, int64_t* launches)
{
    const uint32_t n = (uint32_t)in.vertices, n_faces = (uint32_t)in.faces;
    k_cc_emit_vertices<<<grid(n, POINT_BLOCK), POINT_BLOCK, 0, st>>>(flags, vert_counts, n, in.xyz, in.nrm, in.rgb,
                                                                     out.xyz, out.nrm, out.rgb, label);
    k_cc_emit_faces<<<grid(n_faces, POINT_BLOCK), POINT_BLOCK, 0, st>>>(keep_f, face_counts, n_faces, in.tri, label,
                                                                        out.tri);
    *launches += 2;
    return cudaGetLastError();
}

}  // namespace s3d
