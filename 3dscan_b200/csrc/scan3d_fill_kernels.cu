// scan3d_fill_kernels.cu -- hole filling of a triangle mesh by the minimum-weight triangulation of its boundary loops
// (scan3d_voxel_surface_fill_holes, scan3d_mesh_fill_holes_dev).  The arithmetic and the per-hole dynamic program are
// in common/scan3d_fill_math.h, shared with the host test; this file owns the boundary structure and the launches.
//
// Count: the faces' sides go into the smoothing's table of undirected edges with an atomic side count per slot and the
// face of a side on it; each edge of count 1 gives its hole edge (the reversed side) to the per-vertex in / out counts,
// head and rim face.  Every vertex with one hole edge in and one out walks the successors, stopping at the first vertex
// smaller than itself, so only a loop's smallest vertex walks the whole loop; it flags itself when the loop closes
// through regular vertices within max_edges edges.  The flags, loop lengths and DP sizes are summed per block of
// vertices and scanned (k_scan), which ranks the holes by their smallest vertex.
// Fill, after the host read the totals: one thread per hole gathers its vertices; one block per hole runs the DP
// diagonal by diagonal, one thread per cell, every cell in the header's fixed candidate order; the faces per block of
// holes are scanned, and one thread per filled hole writes its faces in preorder at its rank.  Every count is an
// integer and every choice is made by one thread in a fixed order, so the result is bit-reproducible.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "../common/scan3d_fill_math.h"

namespace s3d {

static_assert(s3h::NETS_MAX_EDGES == SCAN3D_FILL_NETS_MAX_EDGES && s3h::MAX_EDGES == SCAN3D_FILL_MAX_EDGES,
              "the header's caps are the ABI's");
static_assert(s3h::nets_bound_holds(SCAN3D_FILL_NETS_MAX_EDGES) && !s3h::nets_bound_holds(SCAN3D_FILL_NETS_MAX_EDGES + 1),
              "SCAN3D_FILL_NETS_MAX_EDGES is the largest hole that keeps the decimation's quadric sums below 2^63");
static_assert(sizeof(s3h::Cell) == 48, "a DP cell is 48 bytes");

// the kernels' view of a FillWorkspace's counting scratch
struct FillBuffers {
    unsigned long long* keys;      // [cap] edge keys, s3v::EMPTY_KEY = free
    uint32_t* sides;               // [cap] sides on each edge, zeroed
    uint32_t* face;                // [cap] the face of a side on the edge (the only one for a count of 1)
    uint32_t cap;
    uint32_t* out_n;               // [vertices] zeroed
    uint32_t* in_n;                // [vertices] zeroed
    uint32_t* next;                // [vertices] head of the vertex's hole edge (when out_n is 1)
    uint32_t* rim;                 // [vertices] rim face of that hole edge
    uint32_t* len;                 // [vertices]
    uint32_t* block_counts;        // [3][stride] zeroed
    uint32_t stride;
    FillState* state;              // zeroed
};

namespace {

constexpr int ST = 256;                                 // threads per block of the per-item kernels
constexpr int DP_THREADS = 256;                         // threads per hole of the DP
constexpr unsigned FULL = 0xffffffffu;
static_assert(POINT_BLOCK == 1024, "the hole ranks scan one vertex or hole per thread of a POINT_BLOCK block");

unsigned grid(uint64_t n, int threads) { return n ? (unsigned)((n + threads - 1) / threads) : 1u; }

__device__ __forceinline__ bool regular(const uint32_t* out_n, const uint32_t* in_n, uint32_t v)
{
    return out_n[v] == 1 && in_n[v] == 1;
}

// exclusive prefix of x over the POINT_BLOCK threads of the block (every thread calls it)
__device__ __forceinline__ uint32_t block_exclusive(uint32_t x)
{
    __shared__ uint32_t wsum[POINT_BLOCK / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t s = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, s, o);
        if (lane >= o) s += t;
    }
    __syncthreads();                                    // an earlier call's readers are done with wsum
    if (lane == 31) wsum[w] = s;
    __syncthreads();
    uint32_t before = 0;
    for (int k = 0; k < w; k++) before += wsum[k];
    return before + s - x;
}

__device__ __forceinline__ void add_warp(uint32_t* count, uint32_t x)
{
    const uint32_t s = __reduce_add_sync(FULL, x);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(count, s);
}

}  // namespace

// one thread per face: its sides with distinct ends into the edge table; a face with an index outside [0, n) sets
// state->bad and adds nothing
__global__ void __launch_bounds__(ST) k_fh_sides(const int32_t* __restrict__ faces, uint32_t nf, uint32_t n,
                                                 FillBuffers b)
{
    const uint32_t f = blockIdx.x * ST + threadIdx.x;
    if (f >= nf) return;
    const uint32_t v[3] = {(uint32_t)faces[3 * (size_t)f], (uint32_t)faces[3 * (size_t)f + 1],
                           (uint32_t)faces[3 * (size_t)f + 2]};
    if (v[0] >= n || v[1] >= n || v[2] >= n) {
        b.state->bad = 1;
        return;
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const uint32_t a = v[k], c = v[k == 2 ? 0 : k + 1];
        if (a == c) continue;
        bool claimed;
        const uint32_t s = find_or_insert(b.keys, b.cap, edge_key(a, c), &claimed);
        if (s == VOXEL_NO_SLOT) continue;               // the table holds 2 slots per side: not reached
        atomicAdd(&b.sides[s], 1u);
        b.face[s] = f;
    }
}

// one thread per slot: an edge of count 1 is a boundary edge; its hole edge, the reversed side, leaves the side's head
__global__ void __launch_bounds__(ST) k_fh_edges(const int32_t* __restrict__ faces, FillBuffers b)
{
    const uint32_t s = blockIdx.x * ST + threadIdx.x;
    const unsigned long long key = s < b.cap ? b.keys[s] : s3v::EMPTY_KEY;
    const bool boundary = key != s3v::EMPTY_KEY && b.sides[s] == 1;
    add_warp(&b.state->boundary, boundary);
    if (!boundary) return;
    const uint32_t f = b.face[s];
    const uint32_t v[3] = {(uint32_t)faces[3 * (size_t)f], (uint32_t)faces[3 * (size_t)f + 1],
                           (uint32_t)faces[3 * (size_t)f + 2]};
    // the one side (a, c) of the face on this edge; the hole edge runs c -> a
    uint32_t a = v[2], c = v[0];
    if (edge_key(v[0], v[1]) == key) {
        a = v[0];
        c = v[1];
    } else if (edge_key(v[1], v[2]) == key) {
        a = v[1];
        c = v[2];
    }
    atomicAdd(&b.out_n[c], 1u);
    atomicAdd(&b.in_n[a], 1u);
    b.next[c] = a;
    b.rim[c] = f;
}

// per vertex: a coordinate that is not finite sets state->bad; a regular vertex walks its loop and, when it is the
// loop's smallest vertex and the loop closes through regular vertices within max_edges edges, records the loop's
// length; the holes, their edges and their DP cells are summed per block
__global__ void __launch_bounds__(POINT_BLOCK) k_fh_walk(const float* __restrict__ xyz, uint32_t n, uint32_t max_edges,
                                                         FillBuffers b)
{
    const uint32_t v = blockIdx.x * POINT_BLOCK + threadIdx.x;
    uint32_t L = 0;
    bool bad = false;
    if (v < n) {
#pragma unroll
        for (int k = 0; k < 3; k++) bad |= !(xyz[3 * (size_t)v + k] - xyz[3 * (size_t)v + k] == 0.0f);
        if (regular(b.out_n, b.in_n, v)) {
            uint32_t u = b.next[v], edges = 1;
            while (u != v) {
                if (u < v || edges == max_edges || !regular(b.out_n, b.in_n, u)) {
                    edges = 0;
                    break;
                }
                u = b.next[u];
                edges++;
            }
            L = edges;
        }
        b.len[v] = L;
    }
    if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) atomicOr(&b.state->bad, 1u);
    const uint32_t cells = L ? s3h::cells_of((int)L) : 0u;
    add_warp(&b.block_counts[blockIdx.x], L != 0);
    add_warp(&b.block_counts[b.stride + blockIdx.x], L);
    add_warp(&b.block_counts[2 * (size_t)b.stride + blockIdx.x], cells);
    const unsigned long long c64 = __reduce_add_sync(FULL, cells);   // < 32 * 2^19
    if ((threadIdx.x & 31) == 0 && c64) atomicAdd(&b.state->cells64, c64);
}

// per vertex: each hole, ranked by its smallest vertex, with its offsets; its thread walks it into verts
__global__ void __launch_bounds__(POINT_BLOCK) k_fh_holes(FillBuffers b, uint32_t n, FillHole* __restrict__ holes,
                                                          uint32_t* __restrict__ verts)
{
    const uint32_t v = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const uint32_t L = v < n ? b.len[v] : 0u;
    const uint32_t r = b.block_counts[blockIdx.x] + block_exclusive(L != 0);
    const uint32_t vo = b.block_counts[b.stride + blockIdx.x] + block_exclusive(L);
    const uint32_t co = b.block_counts[2 * (size_t)b.stride + blockIdx.x] +
                        block_exclusive(L ? s3h::cells_of((int)L) : 0u);
    if (!L) return;
    holes[r] = FillHole{v, L, vo, co};
    uint32_t u = v;
    for (uint32_t t = 0; t < L; t++) {
        verts[vo + t] = u;
        u = b.next[u];
    }
}

// one block per hole: the rim cells, then the DP diagonal by diagonal; the hole's face count for the emission
__global__ void __launch_bounds__(DP_THREADS, 1) k_fh_dp(const FillHole* __restrict__ holes, uint32_t n_holes,
                                                      const uint32_t* __restrict__ verts,
                                                      const uint32_t* __restrict__ rim, const float* __restrict__ xyz,
                                                      const int32_t* __restrict__ faces,
                                                      const unsigned long long* __restrict__ keys, uint32_t cap,
                                                      s3h::Cell* cells_all, uint32_t* __restrict__ hole_faces,
                                                      uint32_t* __restrict__ face_counts, FillState* state)
{
    __shared__ float p[s3h::MAX_EDGES][3];
    const uint32_t h = blockIdx.x;
    if (h >= n_holes) return;
    const FillHole hole = holes[h];
    const int n = (int)hole.n;
    const uint32_t* v = verts + hole.vert;
    s3h::Cell* cells = cells_all + hole.cell;
    for (int t = threadIdx.x; t < n; t += DP_THREADS) {
        const uint32_t a = v[t], f = rim[a];
        float c[3][3];
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const uint32_t w = (uint32_t)faces[3 * (size_t)f + k];
#pragma unroll
            for (int e = 0; e < 3; e++) c[k][e] = xyz[3 * (size_t)w + e];
        }
#pragma unroll
        for (int e = 0; e < 3; e++) p[t][e] = xyz[3 * (size_t)a + e];
        s3h::rim_cell(c[0], c[1], c[2], cells + (t < n - 1 ? s3h::cell_index(t, t + 1) : s3h::cells_of(n) - 1));
    }
    __syncthreads();
    for (int d = 2; d < n; d++) {
        for (int i = threadIdx.x; i + d < n; i += DP_THREADS) {
            const int j = i + d;
            const bool exists = !(i == 0 && j == n - 1) && find_slot(keys, cap, edge_key(v[i], v[j])) != VOXEL_NO_SLOT;
            s3h::solve_cell(p, cells, n, i, j, exists, cells + s3h::cell_index(i, j));
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const uint32_t added = cells[s3h::cell_index(0, n - 1)].k != s3h::INFEASIBLE ? (uint32_t)n - 2 : 0u;
        hole_faces[h] = added;
        if (added) {
            atomicAdd(&face_counts[h / POINT_BLOCK], added);
            atomicAdd(&state->filled, 1u);
        }
    }
}

// one thread per hole: a filled hole's faces at its rank, nothing at all when they exceed the capacity
__global__ void __launch_bounds__(POINT_BLOCK) k_fh_emit(const FillHole* __restrict__ holes, uint32_t n_holes,
                                                         const uint32_t* __restrict__ hole_faces,
                                                         const uint32_t* __restrict__ face_counts,
                                                         const uint32_t* __restrict__ verts, uint32_t* stack,
                                                         const s3h::Cell* __restrict__ cells, int32_t* out,
                                                         unsigned long long capacity, const FillState* state)
{
    const uint32_t h = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const uint32_t f = h < n_holes ? hole_faces[h] : 0u;
    const uint32_t at = face_counts[blockIdx.x] + block_exclusive(f);
    if (!f || state->added > capacity) return;
    const FillHole hole = holes[h];
    s3h::emit_faces(cells + hole.cell, (int)hole.n, verts + hole.vert, stack + hole.vert, out + 3 * (size_t)at);
}

FillBuffers FillWorkspace::view()
{
    return FillBuffers{keys, sides, face, table, out_n, in_n, next, rim, len, block_counts, stride, state};
}

cudaError_t FillWorkspace::count(const float* xyz, const int32_t* faces, uint32_t n, uint32_t nf, uint32_t max_edges,
                                 cudaStream_t st, int64_t* launches)
{
    const size_t av = n ? n : 1;
    const uint32_t cap = 6ull * nf > 64 ? (uint32_t)(6ull * nf) : 64u;   // two slots per side: at most half are taken
    const int nb = (int)grid(n, POINT_BLOCK);
    table = cap;
    stride = (uint32_t)nb + 1;
    cudaError_t e = grow_group(Grow(keys, cap), Grow(sides, cap), Grow(face, cap));
    if (e == cudaSuccess)
        e = grow_group(Grow(out_n, av), Grow(in_n, av), Grow(next, av), Grow(rim, av), Grow(len, av),
                       Grow(block_counts, 3 * (size_t)stride));
    if (e == cudaSuccess) e = state.ensure(1);
    if (e != cudaSuccess) return e;
    const FillBuffers b = view();
    e = cudaMemsetAsync(b.keys, 0xff, (size_t)cap * sizeof(*b.keys), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.sides, 0, (size_t)cap * sizeof(*b.sides), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.out_n, 0, av * sizeof(*b.out_n), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.in_n, 0, av * sizeof(*b.in_n), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.block_counts, 0, 3 * (size_t)stride * sizeof(*b.block_counts), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.state, 0, sizeof(*b.state), st);
    if (e != cudaSuccess) return e;
    k_fh_sides<<<grid(nf, ST), ST, 0, st>>>(faces, nf, n, b);
    k_fh_edges<<<grid(cap, ST), ST, 0, st>>>(faces, b);
    k_fh_walk<<<nb, POINT_BLOCK, 0, st>>>(xyz, n, max_edges, b);
    e = launch_block_scan(b.block_counts, nb, &b.state->holes, st);
    if (e == cudaSuccess) e = launch_block_scan(b.block_counts + stride, nb, &b.state->loop_edges, st);
    if (e == cudaSuccess) e = launch_block_scan(b.block_counts + 2 * stride, nb, &b.state->cells, st);
    *launches += 6;
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t FillWorkspace::fill(const FillState& counts, const float* xyz, const int32_t* faces, uint32_t n,
                                int32_t* out, uint64_t capacity, cudaStream_t st, int64_t* launches)
{
    const uint32_t H = counts.holes;
    const size_t ah = H ? H : 1, ae = counts.loop_edges ? counts.loop_edges : 1;
    const int nbh = (int)grid(H, POINT_BLOCK);
    cudaError_t e = grow_group(Grow(holes, ah), Grow(hole_faces, ah), Grow(face_counts, (size_t)nbh + 1));
    if (e == cudaSuccess) e = grow_group(Grow(verts, ae), Grow(stack, ae));
    if (e == cudaSuccess) e = cells.ensure(counts.cells64 ? (size_t)counts.cells64 : 1);
    if (e == cudaSuccess) e = cudaMemsetAsync(face_counts, 0, ((size_t)nbh + 1) * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    const int nb = (int)grid(n, POINT_BLOCK);
    const FillBuffers b = view();
    k_fh_holes<<<nb, POINT_BLOCK, 0, st>>>(b, n, holes, verts);
    k_fh_dp<<<H ? H : 1, DP_THREADS, 0, st>>>(holes, H, verts, rim, xyz, faces, keys, table, cells, hole_faces,
                                             face_counts, state);
    e = launch_block_scan(face_counts, nbh, &state.get()->added, st);
    if (e != cudaSuccess) return e;
    k_fh_emit<<<nbh, POINT_BLOCK, 0, st>>>(holes, H, hole_faces, face_counts, verts, stack, cells, out,
                                           (unsigned long long)capacity, state);
    *launches += 4;
    return cudaGetLastError();
}

}  // namespace s3d
