// scan3d_repair_kernels.cu -- the repair of the non-manifold edges and vertices of a triangle mesh
// (scan3d_voxel_surface_repair, scan3d_mesh_repair_dev).  The face key and the per-edge keep rule are in
// common/scan3d_repair_math.h, shared with the host test; this file owns the tables and the launches.
//
// Faces: degenerate faces are flagged per face; duplicates go through an open-addressing table of face indices keyed
// on the sorted triple, where the first face of a triple claims a slot with atomicCAS and later ones compare triples
// and lower the slot to the smallest face index with atomicMin.  The surviving faces' sides go into the smoothing's
// edge table with an atomic face count and the 64-bit atomicMax of the face keys per direction; a second pass takes
// the largest key other than the edge's largest, and a third decides the drops, so the rule needs no sort.
// Fans: the kept faces' sides count again per edge, keeping the two faces of an edge with at most two; every edge in
// exactly two kept faces unites the corners of its two ends in the lock-free union-find of scan3d_union_find.cuh, over
// corners 3 f + k.  Each root is then the smallest corner of its fan; the roots that are not their vertex's smallest
// kept corner get new vertices, ranked by k_count + k_scan over corners.  Every count is an integer atomic and every
// choice an order-independent max or min, so the result is a pure function of the mesh and the flags.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "scan3d_union_find.cuh"
#include "../common/scan3d_repair_math.h"

namespace s3d {

// the kernels' view of a RepairWorkspace
struct RepairBuffers {
    unsigned long long* keys;      // [cap] edge keys, s3v::EMPTY_KEY = free
    uint32_t* sides;               // [cap] surviving faces on the edge, zeroed
    uint32_t* kept_n;              // [cap] kept faces on the edge, zeroed
    unsigned long long* best;      // [cap][3] largest key from the smaller end, from the larger end, other than f1; 0
    uint32_t* pair;                // [cap][2]
    uint32_t cap;
    uint32_t* triples;             // [dup_cap] VOXEL_NO_SLOT = free
    uint32_t dup_cap;
    uint32_t* triple_slot;         // [faces]
    unsigned long long* key;       // [faces]
    uint32_t* side_slot;           // [faces][3]
    uint8_t* status;               // [faces]
    uint8_t* keep;                 // [faces]
    uint32_t* parent;              // [3 faces]
    uint8_t* fresh;                // [3 faces]
    uint32_t* first;               // [vertices] 0xffffffff until a kept corner lowers it
    uint32_t* fans;                // [vertices] zeroed
    RepairState* state;            // zeroed
};

namespace {

constexpr int RT = 256;                                 // threads per block of the per-item kernels
constexpr unsigned FULL = 0xffffffffu;
static_assert(POINT_BLOCK == 1024, "the emission kernels rank one flag per thread of a POINT_BLOCK block");
static_assert(SCAN3D_REPAIR_FACES == 1 && SCAN3D_REPAIR_VERTICES == 2, "the ABI's flags");

unsigned grid(uint64_t n, int threads) { return n ? (unsigned)((n + threads - 1) / threads) : 1u; }

// count += the lanes of the warp with x set (every lane of the warp calls it)
__device__ __forceinline__ void add_warp(uint32_t* count, bool x)
{
    const unsigned m = __ballot_sync(FULL, x);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, (uint32_t)__popc(m));
}

__device__ __forceinline__ void load_face(const int32_t* __restrict__ faces, uint32_t f, uint32_t v[3])
{
#pragma unroll
    for (int k = 0; k < 3; k++) v[k] = (uint32_t)faces[3 * (size_t)f + k];
}

__device__ __forceinline__ void sort3(const uint32_t v[3], uint32_t s[3])
{
    const uint32_t lo = min(v[0], min(v[1], v[2])), hi = max(v[0], max(v[1], v[2]));
    s[0] = lo;
    s[1] = v[0] + v[1] + v[2] - lo - hi;                // modulo 2^32: exact
    s[2] = hi;
}

// the corner of vertex x in face f (x is one of its corners)
__device__ __forceinline__ int corner_of(const int32_t* __restrict__ faces, uint32_t f, uint32_t x)
{
    return (uint32_t)faces[3 * (size_t)f] == x ? 0 : (uint32_t)faces[3 * (size_t)f + 1] == x ? 1 : 2;
}

// the slot of face f's sorted triple s in the duplicate table, which ends up holding the triple's smallest face
__device__ __forceinline__ uint32_t insert_triple(const int32_t* __restrict__ faces, uint32_t f, const uint32_t s[3],
                                                  uint32_t* table, uint32_t cap)
{
    const unsigned long long key = mix64((unsigned long long)s[0] << 32 | s[1]) ^ (unsigned long long)s[2];
    uint32_t slot = hash_home(key, cap);
    for (uint32_t p = 0; p < cap; p++) {
        uint32_t g = __ldcg(table + slot);              // a slot's triple never changes once set
        if (g == VOXEL_NO_SLOT) {
            g = atomicCAS(table + slot, VOXEL_NO_SLOT, f);
            if (g == VOXEL_NO_SLOT) return slot;
        }
        uint32_t w[3], t[3];
        load_face(faces, g, w);
        sort3(w, t);
        if (t[0] == s[0] && t[1] == s[1] && t[2] == s[2]) {
            atomicMin(table + slot, f);
            return slot;
        }
        slot = slot + 1 == cap ? 0 : slot + 1;
    }
    return VOXEL_NO_SLOT;                               // the table holds 2 slots per face: not reached
}

}  // namespace

// one thread per vertex and per face: a coordinate that is not finite or a face index outside [0, n) sets state->bad;
// the corners' parents; a degenerate face is counted, a face of three distinct vertices survives step 1 and, with
// SCAN3D_REPAIR_FACES, claims or joins the slot of its sorted triple
__global__ void __launch_bounds__(RT) k_rp_init(const float* __restrict__ xyz, const int32_t* __restrict__ faces,
                                                uint32_t n, uint32_t nf, int flags, RepairBuffers b)
{
    const uint32_t i = blockIdx.x * RT + threadIdx.x;
    bool bad = false, degenerate = false;
    if (i < n) {
#pragma unroll
        for (int k = 0; k < 3; k++) bad |= !(xyz[3 * (size_t)i + k] - xyz[3 * (size_t)i + k] == 0.0f);
    }
    if (i < nf) {
        uint32_t v[3];
        load_face(faces, i, v);
#pragma unroll
        for (int k = 0; k < 3; k++) b.parent[3 * (size_t)i + k] = 3 * i + k;
        uint8_t st = 0;
        uint32_t slot = VOXEL_NO_SLOT;
        if (v[0] >= n || v[1] >= n || v[2] >= n) {
            bad = true;
        } else if (v[0] == v[1] || v[1] == v[2] || v[0] == v[2]) {
            degenerate = true;
        } else {
            st = 1;
            if (flags & SCAN3D_REPAIR_FACES) {
                uint32_t s[3];
                sort3(v, s);
                slot = insert_triple(faces, i, s, b.triples, b.dup_cap);
            }
        }
        b.status[i] = st;
        b.triple_slot[i] = slot;
    }
    add_warp(&b.state->degenerate, degenerate);
    if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) b.state->bad = 1;
}

// one thread per face: a duplicate (not the smallest face of its triple) is dropped; every other surviving face gets
// its key, and its sides go into the edge table with the count and the largest key per direction
__global__ void __launch_bounds__(RT) k_rp_sides(const float* __restrict__ xyz, const int32_t* __restrict__ faces,
                                                 uint32_t nf, int flags, RepairBuffers b)
{
    const uint32_t f = blockIdx.x * RT + threadIdx.x;
    bool dup = false;
    if (f < nf && b.status[f]) {
        dup = (flags & SCAN3D_REPAIR_FACES) && b.triples[b.triple_slot[f]] != f;
        if (dup) {
            b.status[f] = 0;
        } else {
            uint32_t v[3];
            load_face(faces, f, v);
            const unsigned long long K = s3r::face_key(xyz + 3 * (size_t)v[0], xyz + 3 * (size_t)v[1],
                                                       xyz + 3 * (size_t)v[2], f);
            b.key[f] = K;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const uint32_t a = v[k], c = v[k == 2 ? 0 : k + 1];
                bool claimed;
                const uint32_t s = find_or_insert(b.keys, b.cap, edge_key(a, c), &claimed);   // 2 slots per side
                b.side_slot[3 * (size_t)f + k] = s;
                atomicAdd(&b.sides[s], 1u);
                atomicMax(&b.best[3 * (size_t)s + (a > c)], K);
            }
        }
    }
    add_warp(&b.state->duplicate, dup);
}

// one thread per surviving face (SCAN3D_REPAIR_FACES): its key into the largest other than f1 of each edge with more
// than 2 faces where it is not f1
__global__ void __launch_bounds__(RT) k_rp_second(uint32_t nf, int flags, RepairBuffers b)
{
    const uint32_t f = blockIdx.x * RT + threadIdx.x;
    if (f >= nf || !(flags & SCAN3D_REPAIR_FACES) || !b.status[f]) return;
    const unsigned long long K = b.key[f];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const uint32_t s = b.side_slot[3 * (size_t)f + k];
        if (b.sides[s] <= 2) continue;
        const unsigned long long m0 = b.best[3 * (size_t)s], m1 = b.best[3 * (size_t)s + 1];
        if (K != (m0 > m1 ? m0 : m1)) atomicMax(&b.best[3 * (size_t)s + 2], K);
    }
}

// one thread per face: the keep flag (a surviving face that no edge drops); a kept face's sides count again, the
// first two faces of each edge are recorded, and its corners lower their vertices' smallest kept corner
__global__ void __launch_bounds__(RT) k_rp_drop(const int32_t* __restrict__ faces, uint32_t nf, int flags,
                                                RepairBuffers b)
{
    const uint32_t f = blockIdx.x * RT + threadIdx.x;
    bool dropped = false;
    if (f < nf) {
        bool kept = b.status[f] != 0;
        if (kept && (flags & SCAN3D_REPAIR_FACES)) {
            const unsigned long long K = b.key[f];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const uint32_t s = b.side_slot[3 * (size_t)f + k];
                if (b.sides[s] > 2 &&
                    !s3r::kept_on_edge(K, b.best[3 * (size_t)s], b.best[3 * (size_t)s + 1], b.best[3 * (size_t)s + 2]))
                    dropped = true;
            }
            kept = !dropped;
        }
        b.keep[f] = kept;
        if (kept) {
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const uint32_t s = b.side_slot[3 * (size_t)f + k];
                const uint32_t at = atomicAdd(&b.kept_n[s], 1u);
                if (at < 2) b.pair[2 * (size_t)s + at] = f;
                atomicMin(&b.first[faces[3 * (size_t)f + k]], 3 * f + k);
            }
        }
    }
    add_warp(&b.state->nonmanifold_faces, dropped);
}

// one thread per slot: the edge counts; an edge in exactly two kept faces f, g is inconsistent when both run it the
// same way, and with SCAN3D_REPAIR_VERTICES it joins the corners of each of its ends in f and g
__global__ void __launch_bounds__(RT) k_rp_edges(const int32_t* __restrict__ faces, int flags, RepairBuffers b)
{
    const uint32_t s = blockIdx.x * RT + threadIdx.x;
    const unsigned long long key = s < b.cap ? b.keys[s] : s3v::EMPTY_KEY;
    const bool used = key != s3v::EMPTY_KEY;
    const uint32_t kn = used ? b.kept_n[s] : 0u;
    bool inconsistent = false;
    if (kn == 2) {
        const uint32_t a = (uint32_t)(key >> 32), c = (uint32_t)key;
        const uint32_t f = b.pair[2 * (size_t)s], g = b.pair[2 * (size_t)s + 1];
        const int fa = corner_of(faces, f, a), ga = corner_of(faces, g, a);
        const bool f_up = (uint32_t)faces[3 * (size_t)f + (fa == 2 ? 0 : fa + 1)] == c;   // f runs a -> c
        const bool g_up = (uint32_t)faces[3 * (size_t)g + (ga == 2 ? 0 : ga + 1)] == c;
        inconsistent = f_up == g_up;
        if (flags & SCAN3D_REPAIR_VERTICES) {
            unite(b.parent, 3 * f + fa, 3 * g + ga);
            unite(b.parent, 3 * f + corner_of(faces, f, c), 3 * g + corner_of(faces, g, c));
        }
    }
    add_warp(&b.state->nonmanifold_edges, used && b.sides[s] > 2);
    add_warp(&b.state->boundary, kn == 1);
    add_warp(&b.state->inconsistent, inconsistent);
}

// one thread per corner of a kept face: parent = its fan's root (the fan's smallest corner).  The walk does not halve
// (the only stores are roots, as in the components' compression).  With SCAN3D_REPAIR_VERTICES a root that is not its
// vertex's smallest kept corner is fresh (its fan gets a new vertex), and the vertex's first fresh root counts it split.
__global__ void __launch_bounds__(RT) k_rp_roots(const int32_t* __restrict__ faces, uint32_t corners, int flags,
                                                 RepairBuffers b)
{
    const uint32_t c = blockIdx.x * RT + threadIdx.x;
    bool split = false;
    if (c < corners) {
        bool fresh = false;
        if (b.keep[c / 3]) {
            uint32_t r = c, p;
            while ((p = load_parent(b.parent, r)) != r) r = p;
            store_parent(b.parent, c, r);
            if (r == c && (flags & SCAN3D_REPAIR_VERTICES)) {
                const uint32_t v = (uint32_t)faces[c];
                fresh = b.first[v] != c;
                split = fresh && atomicAdd(&b.fans[v], 1u) == 0;
            }
        }
        b.fresh[c] = fresh;
    }
    add_warp(&b.state->split, split);
}

// one thread per corner: a fresh root becomes vertex n + its rank; its source vertex into source and, when xyz_out is
// set, the source's bytes into the new vertex
__global__ void __launch_bounds__(POINT_BLOCK) k_rp_vertices(const uint8_t* __restrict__ fresh,
                                                             const uint32_t* __restrict__ offsets, uint32_t corners,
                                                             const int32_t* __restrict__ faces, uint32_t n,
                                                             uint32_t* __restrict__ new_id, int32_t* __restrict__ source,
                                                             const float* __restrict__ xyz, const float* __restrict__ nrm,
                                                             const uint8_t* __restrict__ rgb, float* __restrict__ xyz_out,
                                                             float* __restrict__ nrm_out, uint8_t* __restrict__ rgb_out)
{
    const uint32_t c = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const bool is_new = c < corners && fresh[c] != 0;
    const uint32_t r = offsets[blockIdx.x] + block_rank(is_new);
    if (!is_new) return;
    const uint32_t v = (uint32_t)faces[c], w = n + r;
    new_id[c] = w;
    source[r] = (int32_t)v;
    if (!xyz_out) return;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        xyz_out[3 * (size_t)w + k] = xyz[3 * (size_t)v + k];
        nrm_out[3 * (size_t)w + k] = nrm[3 * (size_t)v + k];
        rgb_out[3 * (size_t)w + k] = rgb[3 * (size_t)v + k];
    }
}

// one thread per face: kept face f goes to rank r of its keep flag, each corner remapped to its fan's vertex
__global__ void __launch_bounds__(POINT_BLOCK) k_rp_faces(const uint8_t* __restrict__ keep,
                                                          const uint32_t* __restrict__ offsets, uint32_t nf,
                                                          const int32_t* __restrict__ faces, int flags,
                                                          const uint32_t* __restrict__ parent,
                                                          const uint32_t* __restrict__ first,
                                                          const uint32_t* __restrict__ new_id, int32_t* __restrict__ out)
{
    const uint32_t f = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const bool kept = f < nf && keep[f] != 0;
    const uint32_t r = offsets[blockIdx.x] + block_rank(kept);
    if (!kept) return;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const uint32_t v = (uint32_t)faces[3 * (size_t)f + k];
        uint32_t w = v;
        if (flags & SCAN3D_REPAIR_VERTICES) {
            const uint32_t root = parent[3 * f + k];
            if (root != first[v]) w = new_id[root];
        }
        out[3 * (size_t)r + k] = (int32_t)w;
    }
}

RepairBuffers RepairWorkspace::view()
{
    return RepairBuffers{keys,   sides,       kept_n, best,     pair,   table, triples, dup_table, triple_slot, key,
                         side_slot, status,   keep,   parent,   fresh,  first, fans,    state};
}

cudaError_t RepairWorkspace::count(const float* xyz, const int32_t* faces, uint32_t n, uint32_t nf, int flags,
                                   cudaStream_t st, int64_t* launches)
{
    const size_t av = n ? n : 1, af = nf ? nf : 1, corners = 3 * (size_t)nf;
    const uint32_t cap = 6ull * nf > 64 ? (uint32_t)(6ull * nf) : 64u;   // two slots per side: at most half are taken
    const uint32_t dup_cap = 2ull * nf > 64 ? (uint32_t)(2ull * nf) : 64u;
    table = cap;
    dup_table = dup_cap;
    cudaError_t e = grow_group(Grow(keys, cap), Grow(sides, cap), Grow(kept_n, cap), Grow(best, 3 * (size_t)cap),
                               Grow(pair, 2 * (size_t)cap), Grow(triples, dup_cap));
    if (e == cudaSuccess)
        e = grow_group(Grow(triple_slot, af), Grow(key, af), Grow(side_slot, 3 * af), Grow(status, af), Grow(keep, af),
                       Grow(face_counts, (af + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    if (e == cudaSuccess)
        e = grow_group(Grow(parent, 3 * af), Grow(fresh, 3 * af), Grow(new_id, 3 * af),
                       Grow(corner_counts, (3 * af + POINT_BLOCK - 1) / POINT_BLOCK + 1), Grow(first, av),
                       Grow(fans, av));
    if (e == cudaSuccess) e = state.ensure(1);
    if (e != cudaSuccess) return e;
    const RepairBuffers b = view();
    e = cudaMemsetAsync(b.keys, 0xff, (size_t)cap * sizeof(*b.keys), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.sides, 0, (size_t)cap * sizeof(*b.sides), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.kept_n, 0, (size_t)cap * sizeof(*b.kept_n), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.best, 0, 3 * (size_t)cap * sizeof(*b.best), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.triples, 0xff, (size_t)dup_cap * sizeof(*b.triples), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.first, 0xff, av * sizeof(*b.first), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.fans, 0, av * sizeof(*b.fans), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.state, 0, sizeof(*b.state), st);
    if (e != cudaSuccess) return e;
    const uint32_t m = n > nf ? n : nf;
    k_rp_init<<<grid(m, RT), RT, 0, st>>>(xyz, faces, n, nf, flags, b);
    k_rp_sides<<<grid(nf, RT), RT, 0, st>>>(xyz, faces, nf, flags, b);
    k_rp_second<<<grid(nf, RT), RT, 0, st>>>(nf, flags, b);
    k_rp_drop<<<grid(nf, RT), RT, 0, st>>>(faces, nf, flags, b);
    k_rp_edges<<<grid(cap, RT), RT, 0, st>>>(faces, flags, b);
    k_rp_roots<<<grid(corners, RT), RT, 0, st>>>(faces, (uint32_t)corners, flags, b);
    e = launch_point_offsets(b.fresh, corners, corner_counts, &b.state->added, st);
    if (e == cudaSuccess) e = launch_point_offsets(b.keep, nf, face_counts, &b.state->faces, st);
    *launches += 10;
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t RepairWorkspace::emit(const int32_t* faces, uint32_t n, uint32_t nf, int flags, int32_t* faces_out,
                                  int32_t* source_out, const float* xyz, const float* nrm, const uint8_t* rgb,
                                  float* xyz_out, float* nrm_out, uint8_t* rgb_out, cudaStream_t st, int64_t* launches)
{
    const uint32_t corners = 3 * nf;
    k_rp_vertices<<<grid(corners, POINT_BLOCK), POINT_BLOCK, 0, st>>>(fresh, corner_counts, corners, faces, n, new_id,
                                                                       source_out, xyz, nrm, rgb, xyz_out, nrm_out,
                                                                       rgb_out);
    k_rp_faces<<<grid(nf, POINT_BLOCK), POINT_BLOCK, 0, st>>>(keep, face_counts, nf, faces, flags, parent, first,
                                                              new_id, faces_out);
    *launches += 2;
    return cudaGetLastError();
}

}  // namespace s3d
