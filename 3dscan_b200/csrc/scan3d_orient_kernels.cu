// scan3d_orient_kernels.cu -- the coherent orientation and the measures of a triangle mesh (scan3d_voxel_surface_orient,
// scan3d_mesh_orient_dev, scan3d_voxel_surface_measure, scan3d_mesh_measure_dev).  The centre, the fixed-point terms and
// the int128 sums are in common/scan3d_orient_math.h, shared with the host test; this file owns the tables and the
// launches.
//
// The faces' sides go into the smoothing's edge table with an atomic count, the first two faces of each edge recorded.
// Orientability is a 2-colouring solved by the lock-free union-find of scan3d_union_find.cuh over 2 nf nodes: node 2 f
// is "f as wound", node 2 f + 1 "f flipped".  A consistent edge of count 2 between f and g unites (2 f, 2 g) and
// (2 f + 1, 2 g + 1), an inconsistent one (2 f, 2 g + 1) and (2 f + 1, 2 g).  Roots are the smallest node of their set,
// so an orientable patch of smallest face f0 has the two roots 2 f0 and 2 f0 + 1, and a non-orientable one the single
// root 2 f0: find(2 f) >> 1 is the patch, its parity sigma, and find(2 f) == find(2 f + 1) marks a non-orientable
// patch.  Per patch (indexed by f0) the faces, the faces of sigma = +1, the int128 sum of sigma * D and an open flag are
// summed; every sum is an integer, so the decision is a pure function of the faces.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "scan3d_union_find.cuh"
#include "../common/scan3d_orient_math.h"

namespace s3d {

// the kernels' view of an OrientWorkspace
struct OrientBuffers {
    unsigned long long* keys;      // [cap] edge keys, s3v::EMPTY_KEY = free
    uint32_t* sides;               // [cap] faces on the edge, zeroed
    uint32_t* pair;                // [cap][2] the first two faces on the edge
    uint32_t cap;
    uint32_t* side_slot;           // [faces][3]
    uint8_t* status;               // [faces] 1 = indices in range and not degenerate
    uint32_t* parent;              // [2 faces]
    uint32_t* root;                // [faces] find(2 f) of an active face
    uint8_t* is_root;              // [faces] f is the smallest face of its patch
    uint32_t* size;                // [faces] per patch: faces, zeroed
    uint32_t* npos;                // [faces] per patch: faces of sigma = +1, zeroed
    unsigned long long* v0;        // [faces][2] per patch: sum of sigma D, int128, zeroed
    uint8_t* open;                 // [faces] per patch: a face on an edge whose count is not 2, zeroed
    uint8_t* nonorientable;        // [faces] per patch, zeroed
    uint8_t* flip;                 // [faces]
    uint8_t* ref;                  // [vertices] in a face that is not degenerate, zeroed
    uint8_t* kept;                 // [vertices] in a face that keeps its winding, zeroed
    OrientState* state;
};

namespace {

constexpr int OT = 256;                                 // threads per block
constexpr unsigned FULL = 0xffffffffu;

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

// the corner of vertex x in face f (x is one of its corners)
__device__ __forceinline__ int corner_of(const int32_t* __restrict__ faces, uint32_t f, uint32_t x)
{
    return (uint32_t)faces[3 * (size_t)f] == x ? 0 : (uint32_t)faces[3 * (size_t)f + 1] == x ? 1 : 2;
}

// whether faces f and g run the edge {a, c} the same way
__device__ __forceinline__ bool same_way(const int32_t* __restrict__ faces, uint32_t f, uint32_t g, uint32_t a,
                                         uint32_t c)
{
    const int fa = corner_of(faces, f, a), ga = corner_of(faces, g, a);
    const bool f_up = (uint32_t)faces[3 * (size_t)f + (fa == 2 ? 0 : fa + 1)] == c;   // f runs a -> c
    const bool g_up = (uint32_t)faces[3 * (size_t)g + (ga == 2 ? 0 : ga + 1)] == c;
    return f_up == g_up;
}

// (lo, hi) += the 128-bit value in two 64-bit atomics, the carry of the low word propagated
__device__ __forceinline__ void atomic_add128(unsigned long long* p, unsigned long long lo, unsigned long long hi)
{
    const unsigned long long old = atomicAdd(p, lo);
    atomicAdd(p + 1, hi + (old + lo < lo ? 1ull : 0ull));
}

// the centre of the bounding box held in the state
__device__ __forceinline__ void load_centre(const OrientState* st, float c[3])
{
#pragma unroll
    for (int k = 0; k < 3; k++)
        c[k] = s3o::centre(__uint_as_float(s3o::key_bits(st->box_lo[k])), __uint_as_float(s3o::key_bits(st->box_hi[k])));
}

}  // namespace

// one thread per face: the face-index check, the degenerate faces, the referenced vertices, the sides into the edge
// table with the first two faces of each edge, and the two union-find nodes
__global__ void __launch_bounds__(OT) k_or_sides(const int32_t* __restrict__ faces, uint32_t n, uint32_t nf,
                                                 OrientBuffers b)
{
    const uint32_t f = blockIdx.x * OT + threadIdx.x;
    bool bad = false, degenerate = false;
    if (f < nf) {
        uint32_t v[3];
        load_face(faces, f, v);
        b.parent[2 * (size_t)f] = 2 * f;
        b.parent[2 * (size_t)f + 1] = 2 * f + 1;
        uint8_t st = 0;
        if (v[0] >= n || v[1] >= n || v[2] >= n) {
            bad = true;
        } else if (v[0] == v[1] || v[1] == v[2] || v[0] == v[2]) {
            degenerate = true;
        } else {
            st = 1;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const uint32_t a = v[k], c = v[k == 2 ? 0 : k + 1];
                b.ref[a] = 1;
                bool claimed;
                const uint32_t s = find_or_insert(b.keys, b.cap, edge_key(a, c), &claimed);   // 2 slots per side
                b.side_slot[3 * (size_t)f + k] = s;
                const uint32_t at = atomicAdd(&b.sides[s], 1u);
                if (at < 2) b.pair[2 * (size_t)s + at] = f;
            }
        }
        b.status[f] = st;
    }
    add_warp(&b.state->degenerate, degenerate);
    if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) b.state->bad = 1;
}

// one thread per vertex: the finiteness check; the referenced vertices' count and bounding box
__global__ void __launch_bounds__(OT) k_or_box(const float* __restrict__ xyz, uint32_t n, OrientBuffers b)
{
    const uint32_t i = blockIdx.x * OT + threadIdx.x;
    bool bad = false, used = false;
    unsigned lo[3] = {FULL, FULL, FULL}, hi[3] = {0u, 0u, 0u};
    if (i < n) {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const float x = xyz[3 * (size_t)i + k];
            bad |= !(x - x == 0.0f);
            lo[k] = hi[k] = s3o::order_key(__float_as_uint(x));
        }
        used = b.ref[i] != 0;
        if (!used) {
#pragma unroll
            for (int k = 0; k < 3; k++) lo[k] = FULL, hi[k] = 0u;
        }
    }
    add_warp(&b.state->referenced, used);
    if (__any_sync(FULL, bad) && (threadIdx.x & 31) == 0) b.state->bad = 1;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const unsigned l = __reduce_min_sync(FULL, lo[k]), h = __reduce_max_sync(FULL, hi[k]);
        if ((threadIdx.x & 31) == 0) {
            if (l != FULL) atomicMin(&b.state->box_lo[k], l);
            if (h != 0u) atomicMax(&b.state->box_hi[k], h);
        }
    }
}

// one thread per slot and per vertex: the edge counts, and the unions of an edge of count 2; the largest exponent field
// of a referenced vertex's offset from the centre
__global__ void __launch_bounds__(OT) k_or_edges(const float* __restrict__ xyz, const int32_t* __restrict__ faces,
                                                 uint32_t n, OrientBuffers b)
{
    const uint32_t i = blockIdx.x * OT + threadIdx.x;
    const unsigned long long key = i < b.cap ? b.keys[i] : s3v::EMPTY_KEY;
    const bool used = key != s3v::EMPTY_KEY;
    const uint32_t cnt = used ? b.sides[i] : 0u;
    bool inconsistent = false;
    if (cnt == 2) {
        const uint32_t a = (uint32_t)(key >> 32), c = (uint32_t)key;
        const uint32_t f = b.pair[2 * (size_t)i], g = b.pair[2 * (size_t)i + 1];
        inconsistent = same_way(faces, f, g, a, c);
        unite(b.parent, 2 * f, 2 * g + inconsistent);
        unite(b.parent, 2 * f + 1, 2 * g + !inconsistent);
    }
    add_warp(&b.state->edges, used);
    add_warp(&b.state->boundary, cnt == 1);
    add_warp(&b.state->nonmanifold, cnt > 2);
    add_warp(&b.state->inconsistent, inconsistent);
    unsigned field = 0;
    if (i < n && b.ref[i]) {
        float c[3];
        load_centre(b.state, c);
#pragma unroll
        for (int k = 0; k < 3; k++) field = max(field, s3o::offset_field(xyz[3 * (size_t)i + k], c[k]));
    }
    field = __reduce_max_sync(FULL, field);
    if ((threadIdx.x & 31) == 0 && field) atomicMax(&b.state->exp_field, field);
}

// one thread per face: an active face's root, its patch's counters and open and non-orientable flags; the volume and
// area terms, summed exactly per patch (sigma D, per warp and patch) and over the mesh (D and area, per block)
__global__ void __launch_bounds__(OT) k_or_faces(const float* __restrict__ xyz, const int32_t* __restrict__ faces,
                                                 uint32_t nf, OrientBuffers b)
{
    __shared__ long long t_patch[OT], t_vol[OT], t_area[OT];
    __shared__ unsigned long long part[OT / 32][4];
    const uint32_t f = blockIdx.x * OT + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool active = f < nf && b.status[f] != 0;
    uint32_t f0 = VOXEL_NO_SLOT;
    bool pos = false;
    long long D = 0, A = 0;
    if (active) {
        const uint32_t r = find(b.parent, 2 * f), r1 = find(b.parent, 2 * f + 1);
        f0 = r >> 1;
        pos = (r & 1) == 0;
        b.root[f] = r;
        if (r == r1 && !b.nonorientable[f0]) b.nonorientable[f0] = 1;
        bool open = false;
#pragma unroll
        for (int k = 0; k < 3; k++) open |= b.sides[b.side_slot[3 * (size_t)f + k]] != 2;
        if (open && !b.open[f0]) b.open[f0] = 1;
        uint32_t v[3];
        load_face(faces, f, v);
        float p[3][3], c[3];
#pragma unroll
        for (int j = 0; j < 3; j++)
#pragma unroll
            for (int k = 0; k < 3; k++) p[j][k] = xyz[3 * (size_t)v[j] + k];
        load_centre(b.state, c);
        const int E = s3o::exponent(b.state->exp_field);
        D = s3o::volume_term(p[0], p[1], p[2], c, E);
        A = s3o::area_term(p[0], p[1], p[2], E);
        b.is_root[f] = r == 2 * f;
    } else if (f < nf) {
        b.is_root[f] = 0;
    }
    t_patch[threadIdx.x] = pos ? D : -D;
    t_vol[threadIdx.x] = D;
    t_area[threadIdx.x] = A;
    const unsigned grp = __match_any_sync(FULL, f0), posm = __ballot_sync(FULL, pos);
    __syncwarp();
    if (active && lane == __ffs(grp) - 1) {
        atomicAdd(&b.size[f0], (uint32_t)__popc(grp));
        if (posm & grp) atomicAdd(&b.npos[f0], (uint32_t)__popc(posm & grp));
        unsigned long long lo = 0, hi = 0;
        for (unsigned m = grp; m; m &= m - 1) s3o::add128(&lo, &hi, t_patch[(w << 5) + __ffs(m) - 1]);
        atomic_add128(b.v0 + 2 * (size_t)f0, lo, hi);
    }
    if (lane == 0) {
        unsigned long long vl = 0, vh = 0, al = 0, ah = 0;
        for (int k = 0; k < 32; k++) {
            s3o::add128(&vl, &vh, t_vol[(w << 5) + k]);
            s3o::add128(&al, &ah, t_area[(w << 5) + k]);
        }
        part[w][0] = vl, part[w][1] = vh, part[w][2] = al, part[w][3] = ah;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long s[4] = {0, 0, 0, 0};
        for (int k = 0; k < OT / 32; k++) {
            s[0] += part[k][0];
            s[1] += part[k][1] + (s[0] < part[k][0] ? 1ull : 0ull);
            s[2] += part[k][2];
            s[3] += part[k][3] + (s[2] < part[k][2] ? 1ull : 0ull);
        }
        atomic_add128(b.state->volume, s[0], s[1]);
        atomic_add128(b.state->area, s[2], s[3]);
    }
}

// one thread per face and per slot: the flip of an active face by its patch's rule, the vertices of the faces that
// keep their winding, the closed and non-orientable patches at their smallest face; the inconsistent edges left, those
// of non-orientable patches
__global__ void __launch_bounds__(OT) k_or_decide(const int32_t* __restrict__ faces, uint32_t nf, OrientBuffers b)
{
    const uint32_t i = blockIdx.x * OT + threadIdx.x;
    bool flipped = false, closed = false, nonorientable = false, left = false;
    if (i < nf) {
        bool flip = false;
        if (b.status[i]) {
            const uint32_t r = b.root[i], f0 = r >> 1;
            const bool nonor = b.nonorientable[f0] != 0;
            if (!nonor) {
                const bool is_closed = !b.open[f0];
                const int s = s3o::sign128(b.v0[2 * (size_t)f0], b.v0[2 * (size_t)f0 + 1]);
                const bool keep = is_closed && s != 0 ? s > 0 : 2ull * b.npos[f0] >= (unsigned long long)b.size[f0];
                flip = (r & 1) == (uint32_t)keep;
            }
            if (!flip) {
#pragma unroll
                for (int k = 0; k < 3; k++) b.kept[faces[3 * (size_t)i + k]] = 1;
            }
            if (b.is_root[i]) {
                closed = !b.open[f0];
                nonorientable = nonor;
            }
        }
        b.flip[i] = flip;
        flipped = flip;
    }
    if (i < b.cap) {
        const unsigned long long key = b.keys[i];
        if (key != s3v::EMPTY_KEY && b.sides[i] == 2) {
            const uint32_t f = b.pair[2 * (size_t)i];
            left = b.nonorientable[b.root[f] >> 1] &&
                   same_way(faces, f, b.pair[2 * (size_t)i + 1], (uint32_t)(key >> 32), (uint32_t)key);
        }
    }
    add_warp(&b.state->flipped, flipped);
    add_warp(&b.state->closed, closed);
    add_warp(&b.state->nonorientable, nonorientable);
    add_warp(&b.state->inconsistent_after, left);
}

// one thread per face and per vertex, nothing written when the state holds an error: a flipped face (a, b, c) becomes
// (a, c, b); a referenced vertex whose every face flipped is counted and its normal, when given, negated
__global__ void __launch_bounds__(OT) k_or_apply(int32_t* __restrict__ faces, float* __restrict__ nrm, uint32_t n,
                                                 uint32_t nf, OrientBuffers b)
{
    if (b.state->bad) return;
    const uint32_t i = blockIdx.x * OT + threadIdx.x;
    if (i < nf && b.flip[i]) {
        const int32_t t = faces[3 * (size_t)i + 1];
        faces[3 * (size_t)i + 1] = faces[3 * (size_t)i + 2];
        faces[3 * (size_t)i + 2] = t;
    }
    const bool turned = i < n && b.ref[i] && !b.kept[i];
    if (turned && nrm) {
        uint32_t* u = reinterpret_cast<uint32_t*>(nrm) + 3 * (size_t)i;
#pragma unroll
        for (int k = 0; k < 3; k++) u[k] ^= 0x80000000u;
    }
    add_warp(&b.state->flipped_normals, turned);
}

OrientBuffers OrientWorkspace::view()
{
    return OrientBuffers{keys, sides, pair,  table, side_slot, status,        parent, root, is_root,
                         size, npos,  v0,    open,  nonorientable, flip,      ref,    kept, state};
}

cudaError_t OrientWorkspace::count(const float* xyz, const int32_t* faces, uint32_t n, uint32_t nf, cudaStream_t st,
                                   int64_t* launches)
{
    const size_t av = n ? n : 1, af = nf ? nf : 1;
    const uint32_t cap = 6ull * nf > 64 ? (uint32_t)(6ull * nf) : 64u;   // two slots per side: at most half are taken
    table = cap;
    cudaError_t e = grow_group(Grow(keys, cap), Grow(sides, cap), Grow(pair, 2 * (size_t)cap));
    if (e == cudaSuccess)
        e = grow_group(Grow(side_slot, 3 * af), Grow(status, af), Grow(parent, 2 * af), Grow(root, af),
                       Grow(is_root, af), Grow(face_counts, (af + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    if (e == cudaSuccess)
        e = grow_group(Grow(size, af), Grow(npos, af), Grow(v0, 2 * af), Grow(open, af), Grow(nonorientable, af),
                       Grow(flip, af));
    if (e == cudaSuccess) e = grow_group(Grow(ref, av), Grow(kept, av));
    if (e == cudaSuccess) e = state.ensure(1);
    if (e != cudaSuccess) return e;
    const OrientBuffers b = view();
    e = cudaMemsetAsync(b.keys, 0xff, (size_t)cap * sizeof(*b.keys), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.sides, 0, (size_t)cap * sizeof(*b.sides), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.size, 0, af * sizeof(*b.size), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.npos, 0, af * sizeof(*b.npos), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.v0, 0, 2 * af * sizeof(*b.v0), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.open, 0, af, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.nonorientable, 0, af, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.ref, 0, av, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.kept, 0, av, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.state, 0, sizeof(*b.state), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.state->box_lo, 0xff, sizeof(b.state->box_lo), st);
    if (e != cudaSuccess) return e;
    k_or_sides<<<grid(nf, OT), OT, 0, st>>>(faces, n, nf, b);
    k_or_box<<<grid(n, OT), OT, 0, st>>>(xyz, n, b);
    k_or_edges<<<grid(cap > n ? cap : n, OT), OT, 0, st>>>(xyz, faces, n, b);
    k_or_faces<<<grid(nf, OT), OT, 0, st>>>(xyz, faces, nf, b);
    e = launch_point_offsets(b.is_root, nf, face_counts, &b.state->patches, st);
    k_or_decide<<<grid(cap, OT), OT, 0, st>>>(faces, nf, b);
    *launches += 7;
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t OrientWorkspace::apply(int32_t* faces, float* nrm, uint32_t n, uint32_t nf, cudaStream_t st,
                                   int64_t* launches)
{
    k_or_apply<<<grid(nf > n ? nf : n, OT), OT, 0, st>>>(faces, nrm, n, nf, view());
    *launches += 1;
    return cudaGetLastError();
}

}  // namespace s3d
