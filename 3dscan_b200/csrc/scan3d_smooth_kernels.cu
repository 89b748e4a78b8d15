// scan3d_smooth_kernels.cu -- Taubin lambda|mu smoothing of a triangle mesh (scan3d_voxel_surface_smooth,
// scan3d_mesh_smooth_dev).  The arithmetic is in common/scan3d_smooth_math.h, shared with the host test; this file owns
// the neighbour structure, the passes and the normals.
//
// Build: the faces' sides go into an open-addressing table of undirected edges keyed (min << 32 | max) with an atomic
// side count per slot, which deduplicates the neighbours and gives each edge's count.  One pass over the slots gives
// the degrees and the held flags; per-block degree sums, k_scan and an in-block scan give the row starts, and a scatter
// fills each vertex's row of neighbours through per-vertex cursors.  The order inside a row depends on scheduling, but
// the positions are int64 fixed point and a row's sum is exact, so no result does.
// Passes: one gather per pass, ping-pong between two position buffers, no atomics.  A vertex of up to HUB neighbours
// is summed by its own thread; the warp then sums each larger row together, so a hub does not hold one thread for
// long.  End: the face normals are added as fixed-point integers (atomics aggregated per warp), then one vertex kernel
// writes the positions and normals unless the device found an error.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "../common/scan3d_smooth_math.h"

namespace s3d {

// the kernels' view of a SmoothWorkspace
struct SmoothBuffers {
    unsigned long long* keys;      // [cap] edge keys, s3v::EMPTY_KEY = free
    uint32_t* sides;               // [cap] sides on each edge, zeroed
    uint32_t cap;
    uint32_t* degree;              // [vertices] distinct neighbours, zeroed
    uint8_t* held;                 // [vertices] zeroed
    uint32_t* block_counts;        // [cdiv(vertices, POINT_BLOCK) + 1]
    uint32_t* cursor;              // [vertices] row start, then (after the scatter) row end
    uint32_t* rows;                // [cap] neighbour indices (2 per edge, at most 2 * 3 nf)
    long long* q[2];               // [vertices][3] fixed-point positions, ping-pong
    unsigned long long* nsum;      // [vertices][3] fixed-point normal sums (int64 two's complement), zeroed
    SmoothState* state;            // zeroed
};

namespace {

constexpr int ST = 256;                                 // threads per block of the per-item kernels
constexpr uint32_t HUB = 64;                            // rows longer than this are summed by the whole warp
constexpr unsigned FULL = 0xffffffffu;
static_assert(POINT_BLOCK == 1024, "the row starts scan one degree per thread of a POINT_BLOCK block");

unsigned grid(uint64_t n, int threads) { return n ? (unsigned)((n + threads - 1) / threads) : 1u; }

// the lanes of the warp whose v is the same take consecutive values of counter[v] (v == VOXEL_NO_SLOT: none); returns
// this lane's.  Every lane of the warp calls it.
__device__ __forceinline__ uint32_t take_per_warp(uint32_t* counter, uint32_t v)
{
    const unsigned m = __match_any_sync(FULL, v);
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    uint32_t base = 0;
    if (v != VOXEL_NO_SLOT && lane == leader) base = atomicAdd(&counter[v], (uint32_t)__popc(m));
    base = __shfl_sync(FULL, base, leader);
    return base + __popc(m & ((1u << lane) - 1));
}

__device__ __forceinline__ void flag_warp(uint32_t* flag, bool f)
{
    if (__any_sync(FULL, f) && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}

__device__ __forceinline__ void count_warp(uint32_t* count, bool f)
{
    const unsigned m = __ballot_sync(FULL, f);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, (uint32_t)__popc(m));
}

__device__ __forceinline__ bool is_free(const uint32_t* degree, const uint8_t* held, uint32_t v)
{
    return degree[v] != 0 && !held[v];
}

// a vertex's position after the passes: its fixed point for a free vertex, else its input bytes
__device__ __forceinline__ void final_position(const float* xyz, const long long* q, bool free, int E, uint32_t v,
                                               float p[3])
{
#pragma unroll
    for (int k = 0; k < 3; k++) p[k] = free ? s3t::dequantise(q[3 * (size_t)v + k], E) : xyz[3 * (size_t)v + k];
}

}  // namespace

// the largest exponent field of the coordinates; a coordinate that is not finite sets state->bad
__global__ void __launch_bounds__(ST) k_sm_exponent(const float* __restrict__ xyz, uint32_t n, SmoothState* state)
{
    const uint32_t v = blockIdx.x * ST + threadIdx.x;
    uint32_t field = 0;
    if (v < n) {
#pragma unroll
        for (int k = 0; k < 3; k++) field = max(field, s3t::exponent_field(xyz[3 * (size_t)v + k]));
    }
    flag_warp(&state->bad, field == 0xffu);
    field = __reduce_max_sync(FULL, field);
    if ((threadIdx.x & 31) == 0 && field) atomicMax(&state->exp_field, field);
}

// one thread per face: its sides with distinct ends into the edge table; a face with an index outside [0, n) sets
// state->bad and adds nothing
__global__ void __launch_bounds__(ST) k_sm_sides(const int32_t* __restrict__ faces, uint32_t nf, uint32_t n,
                                                 SmoothBuffers b)
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
        if (s == VOXEL_NO_SLOT) {                       // the table holds 2 slots per side: not reached
            b.state->overflow = 1;
            continue;
        }
        atomicAdd(&b.sides[s], 1u);
    }
}

// one thread per slot: an edge adds one to the degree of both ends, and holds both when its count is not 2
__global__ void __launch_bounds__(ST) k_sm_edges(SmoothBuffers b)
{
    const uint32_t s = blockIdx.x * ST + threadIdx.x;
    const unsigned long long key = s < b.cap ? b.keys[s] : s3v::EMPTY_KEY;
    const bool edge = key != s3v::EMPTY_KEY;
    const uint32_t lo = edge ? (uint32_t)(key >> 32) : VOXEL_NO_SLOT, hi = edge ? (uint32_t)key : VOXEL_NO_SLOT;
    take_per_warp(b.degree, lo);                        // a hub's edges share one atomic per warp
    take_per_warp(b.degree, hi);
    if (edge && b.sides[s] != 2) {
        b.held[lo] = 1;
        b.held[hi] = 1;
    }
}

// block_counts[i] = the degree sum of block i of POINT_BLOCK vertices
__global__ void __launch_bounds__(POINT_BLOCK) k_sm_block_sums(const uint32_t* __restrict__ degree, uint32_t n,
                                                               uint32_t* __restrict__ block_counts)
{
    __shared__ uint32_t wsum[POINT_BLOCK / 32];
    const uint32_t v = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const uint32_t d = __reduce_add_sync(FULL, v < n ? degree[v] : 0u);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = d;
    __syncthreads();
    if (threadIdx.x < 32) {
        const uint32_t s = __reduce_add_sync(FULL, wsum[threadIdx.x]);
        if (threadIdx.x == 0) block_counts[blockIdx.x] = s;
    }
}

// per vertex: the row start (cursor), the fixed-point position, the held / isolated counts and the degree limit
__global__ void __launch_bounds__(POINT_BLOCK) k_sm_offsets(const float* __restrict__ xyz, SmoothBuffers b, uint32_t n)
{
    __shared__ uint32_t wsum[POINT_BLOCK / 32];
    const uint32_t v = blockIdx.x * POINT_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t d = v < n ? b.degree[v] : 0u;
    uint32_t s = d;                                     // inclusive scan within the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, s, o);
        if (lane >= o) s += t;
    }
    if (lane == 31) wsum[w] = s;
    __syncthreads();
    uint32_t before = 0;
    for (int k = 0; k < w; k++) before += wsum[k];
    const bool held = v < n && b.held[v];
    if (v < n) {
        b.cursor[v] = b.block_counts[blockIdx.x] + before + s - d;
        const int E = s3t::exponent(b.state->exp_field);
#pragma unroll
        for (int k = 0; k < 3; k++) b.q[0][3 * (size_t)v + k] = s3t::quantise(xyz[3 * (size_t)v + k], E);
    }
    count_warp(&b.state->held, held);
    count_warp(&b.state->isolated, v < n && d == 0);
    flag_warp(&b.state->overflow, !held && d > s3t::DEGREE_LIMIT);
}

// one thread per slot: each end of an edge gets the other in its row
__global__ void __launch_bounds__(ST) k_sm_scatter(SmoothBuffers b)
{
    const uint32_t s = blockIdx.x * ST + threadIdx.x;
    const unsigned long long key = s < b.cap ? b.keys[s] : s3v::EMPTY_KEY;
    const bool edge = key != s3v::EMPTY_KEY;
    const uint32_t lo = edge ? (uint32_t)(key >> 32) : VOXEL_NO_SLOT, hi = edge ? (uint32_t)key : VOXEL_NO_SLOT;
    const uint32_t at_lo = take_per_warp(b.cursor, lo);
    const uint32_t at_hi = take_per_warp(b.cursor, hi);
    if (edge) {
        b.rows[at_lo] = hi;
        b.rows[at_hi] = lo;
    }
}

// one pass: qout = qin moved by k towards (k > 0) or away from (k < 0) the mean of the neighbours, for free vertices
__global__ void __launch_bounds__(ST) k_sm_pass(const long long* __restrict__ qin, long long* __restrict__ qout,
                                                const uint32_t* __restrict__ degree, const uint8_t* __restrict__ held,
                                                const uint32_t* __restrict__ row_end,
                                                const uint32_t* __restrict__ rows, uint32_t n, double k,
                                                SmoothState* state)
{
    const uint32_t v = blockIdx.x * ST + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool hub = false, over = false;
    uint32_t d = 0;
    if (v < n) {
        d = degree[v];
        const bool free = d != 0 && !held[v];
        long long q[3] = {qin[3 * (size_t)v], qin[3 * (size_t)v + 1], qin[3 * (size_t)v + 2]};
        if (free && d <= HUB) {
            unsigned long long sum[3] = {0, 0, 0};     // modulo 2^64: exact below the limits, defined above them
            const uint32_t end = row_end[v];
            for (uint32_t i = end - d; i < end; i++) {
                const uint32_t u = rows[i];
#pragma unroll
                for (int a = 0; a < 3; a++) sum[a] += (unsigned long long)qin[3 * (size_t)u + a];
            }
#pragma unroll
            for (int a = 0; a < 3; a++) {
                q[a] = s3t::update(q[a], (long long)sum[a], d, k);
                over |= s3t::over_limit(q[a]);
            }
        }
        hub = free && d > HUB;
        if (!hub) {
#pragma unroll
            for (int a = 0; a < 3; a++) qout[3 * (size_t)v + a] = q[a];
        }
    }
    // the warp sums each long row together, 32 neighbours at a time
    for (unsigned hubs = __ballot_sync(FULL, hub); hubs; hubs &= hubs - 1) {
        const int owner = __ffs(hubs) - 1;
        const uint32_t u = __shfl_sync(FULL, v, owner), du = __shfl_sync(FULL, d, owner);
        const uint32_t end = row_end[u];
        unsigned long long sum[3] = {0, 0, 0};
        for (uint32_t i = end - du + lane; i < end; i += 32) {
            const uint32_t w = rows[i];
#pragma unroll
            for (int a = 0; a < 3; a++) sum[a] += (unsigned long long)qin[3 * (size_t)w + a];
        }
#pragma unroll
        for (int a = 0; a < 3; a++)
            for (int o = 16; o; o >>= 1) sum[a] += __shfl_xor_sync(FULL, sum[a], o);
        if (lane == owner) {
#pragma unroll
            for (int a = 0; a < 3; a++) {
                const long long q = s3t::update(qin[3 * (size_t)u + a], (long long)sum[a], du, k);
                over |= s3t::over_limit(q);
                qout[3 * (size_t)u + a] = q;
            }
        }
    }
    flag_warp(&state->overflow, over);
}

// one thread per face: its fixed-point unit normal into the sums of its three vertices (faces with three distinct
// valid indices); a free corner whose final coordinate is not finite sets state->overflow
__global__ void __launch_bounds__(ST) k_sm_face_normals(const int32_t* __restrict__ faces, uint32_t nf, uint32_t n,
                                                        const float* __restrict__ xyz, const long long* __restrict__ q,
                                                        SmoothBuffers b)
{
    const uint32_t f = blockIdx.x * ST + threadIdx.x;
    const int lane = threadIdx.x & 31;
    uint32_t v[3] = {VOXEL_NO_SLOT, VOXEL_NO_SLOT, VOXEL_NO_SLOT};
    long long m[3] = {0, 0, 0};
    bool has = false, over = false;
    if (f < nf) {
        bool valid = true;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            v[k] = (uint32_t)faces[3 * (size_t)f + k];
            valid = valid && v[k] < n;
        }
        if (valid) {
            const int E = s3t::exponent(b.state->exp_field);
            float p[3][3];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const bool free = is_free(b.degree, b.held, v[k]);
                final_position(xyz, q, free, E, v[k], p[k]);
                over |= free && !(p[k][0] - p[k][0] == 0.0f && p[k][1] - p[k][1] == 0.0f &&
                                  p[k][2] - p[k][2] == 0.0f);
            }
            has = v[0] != v[1] && v[1] != v[2] && v[0] != v[2] && s3t::face_normal(p[0], p[1], p[2], m);
        }
    }
    flag_warp(&b.state->overflow, over);
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const uint32_t key = has ? v[k] : VOXEL_NO_SLOT;
        const unsigned grp = __match_any_sync(FULL, key);
        const bool leader = lane == __ffs(grp) - 1;
#pragma unroll
        for (int a = 0; a < 3; a++) {
            // at most 32 terms of |m| <= 2^24: the 32-bit sum is exact
            const int sum = (int)__reduce_add_sync(grp, (uint32_t)(int)m[a]);
            if (has && leader) atomicAdd(&b.nsum[3 * (size_t)key + a], (unsigned long long)(long long)sum);
        }
    }
}

// per vertex: the output position and normal, and the largest displacement; nothing is written after an error
__global__ void __launch_bounds__(ST) k_sm_write(const float* xyz, const float* nrm, uint32_t n,
                                                 const long long* __restrict__ q, SmoothBuffers b, float* xyz_out,
                                                 float* nrm_out)
{
    if (b.state->bad || b.state->overflow) return;
    const uint32_t v = blockIdx.x * ST + threadIdx.x;
    double move = 0.0;
    if (v < n) {
        const bool free = is_free(b.degree, b.held, v);
        const float old[3] = {xyz[3 * (size_t)v], xyz[3 * (size_t)v + 1], xyz[3 * (size_t)v + 2]};
        float p[3];
        final_position(xyz, q, free, s3t::exponent(b.state->exp_field), v, p);
        if (free) move = s3t::displacement(old, p);
        const long long s[3] = {(long long)b.nsum[3 * (size_t)v], (long long)b.nsum[3 * (size_t)v + 1],
                                (long long)b.nsum[3 * (size_t)v + 2]};
        float nn[3];
        const bool keep = s[0] == 0 && s[1] == 0 && s[2] == 0;
        if (nrm_out) {
            if (keep) {
#pragma unroll
                for (int k = 0; k < 3; k++) nn[k] = nrm[3 * (size_t)v + k];
            } else {
                s3v::normal_out(s[0], s[1], s[2], nn);
            }
        }
#pragma unroll
        for (int k = 0; k < 3; k++) {
            xyz_out[3 * (size_t)v + k] = p[k];
            if (nrm_out) nrm_out[3 * (size_t)v + k] = nn[k];
        }
    }
    unsigned long long bits = (unsigned long long)__double_as_longlong(move);
    for (int o = 16; o; o >>= 1) bits = max(bits, __shfl_xor_sync(FULL, bits, o));
    if ((threadIdx.x & 31) == 0 && bits) atomicMax(&b.state->max_move, bits);
}

cudaError_t SmoothWorkspace::run(const float* xyz, const float* nrm, const int32_t* faces, uint32_t n, uint32_t nf,
                                 int passes, double lambda, double mu, float* xyz_out, float* nrm_out, cudaStream_t st,
                                 int64_t* launches)
{
    const size_t av = n ? n : 1;
    const uint32_t cap = 6ull * nf > 64 ? (uint32_t)(6ull * nf) : 64u;   // two slots per side: at most half are taken
    cudaError_t e = grow_group(Grow(keys, cap), Grow(sides, cap), Grow(rows, cap));
    if (e == cudaSuccess)
        e = grow_group(Grow(degree, av), Grow(held, av), Grow(block_counts, (av + POINT_BLOCK - 1) / POINT_BLOCK + 1),
                       Grow(cursor, av), Grow(q[0], 3 * av), Grow(q[1], 3 * av));
    if (e == cudaSuccess) e = nsum.ensure(3 * av);
    if (e == cudaSuccess) e = state.ensure(1);
    if (e != cudaSuccess) return e;
    const SmoothBuffers b{keys, sides, cap, degree, held, block_counts, cursor, rows, {q[0], q[1]}, nsum, state};
    e = cudaMemsetAsync(b.keys, 0xff, (size_t)cap * sizeof(*b.keys), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.sides, 0, (size_t)cap * sizeof(*b.sides), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.degree, 0, av * sizeof(*b.degree), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.held, 0, av * sizeof(*b.held), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.nsum, 0, 3 * av * sizeof(*b.nsum), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b.state, 0, sizeof(*b.state), st);
    if (e != cudaSuccess) return e;
    const int nb = (int)grid(n, POINT_BLOCK);
    k_sm_exponent<<<grid(n, ST), ST, 0, st>>>(xyz, n, b.state);
    k_sm_sides<<<grid(nf, ST), ST, 0, st>>>(faces, nf, n, b);
    k_sm_edges<<<grid(b.cap, ST), ST, 0, st>>>(b);
    k_sm_block_sums<<<nb, POINT_BLOCK, 0, st>>>(b.degree, n, b.block_counts);
    e = launch_block_scan(b.block_counts, nb, &b.state->entries, st);
    if (e != cudaSuccess) return e;
    k_sm_offsets<<<nb, POINT_BLOCK, 0, st>>>(xyz, b, n);
    k_sm_scatter<<<grid(b.cap, ST), ST, 0, st>>>(b);
    for (int p = 0; p < passes; p++) {
        const double k = mu == 0.0 || p % 2 == 0 ? lambda : mu;
        k_sm_pass<<<grid(n, ST), ST, 0, st>>>(b.q[p & 1], b.q[(p + 1) & 1], b.degree, b.held, b.cursor, b.rows, n, k,
                                              b.state);
    }
    const long long* qf = b.q[passes & 1];
    k_sm_face_normals<<<grid(nf, ST), ST, 0, st>>>(faces, nf, n, xyz, qf, b);
    k_sm_write<<<grid(n, ST), ST, 0, st>>>(xyz, nrm, n, qf, b, xyz_out, nrm_out);
    *launches += 7 + passes + 2;
    return cudaGetLastError();
}

}  // namespace s3d
