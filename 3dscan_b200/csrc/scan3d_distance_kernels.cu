// scan3d_distance_kernels.cu -- the distances of samples from the nearest face of a triangle mesh within R
// (scan3d_voxel_surface_distance, scan3d_voxel_surface_distance_dev, scan3d_mesh_distance_dev).  The closest point, the
// sign, the cell box of a face and the order of the sums are in common/scan3d_distance_math.h, shared with the host
// test; this file owns the face index, the query and the reduction.
//
// Count (2 launches): per face the index and finiteness checks, its cell box and its entry count, summed per block of
// POINT_BLOCK faces and over the mesh; k_scan turns the block sums into offsets.  The host reads the total.
// Index (3 launches): each face's entries (face, cell) take consecutive places from its block's offset; the cells go
// into the open-addressing table of scan3d_hash.cuh with a face count per cell; each cell reserves its range of the id
// array (one atomic per warp of slots, as k_align_ranges); one thread per entry scatters the face id into its cell's
// range.  The order inside a range varies from run to run; the selection cannot, because it is by (d2, face).
// Query (2 launches): one sample per thread probes the 27 cells around its cell and keeps the exact (d2, face) minimum,
// writes its outputs and adds to its block's statistics in a fixed tree; one block sums the block partials in a fixed
// order.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "../common/scan3d_distance_math.h"

namespace s3d {

namespace {

constexpr int QT = s3p::BLOCK;            // threads per query block: one sample each
constexpr int IT = 256;                   // threads per block of the range and scatter kernels
constexpr unsigned FULL = 0xffffffffu;
constexpr int CELLS_PER_ENTRY = 2;        // table slots per entry: at most half of them are taken

unsigned grid(uint64_t n, int threads) { return n ? (unsigned)((n + threads - 1) / threads) : 1u; }

// the kernels' view of the index
struct DistanceIndex {
    unsigned long long* keys;             // [cap] s3v::pack_key of the cell, s3v::EMPTY_KEY = free
    uint2* cells;                         // [cap] (faces in the cell, end of its range in ids)
    uint32_t* entry_slot;                 // [entries]
    uint32_t* entry_face;                 // [entries]
    uint32_t* ids;                        // [entries]
    uint32_t* cursor;
    uint32_t cap;
};

__device__ __forceinline__ bool finite3(const float* v)
{
    return v[0] - v[0] == 0.0f && v[1] - v[1] == 0.0f && v[2] - v[2] == 0.0f;
}

// the corners of face f into c [3][3]; false when an index is outside [0, n)
__device__ __forceinline__ bool load_corners(const float* __restrict__ xyz, const int32_t* __restrict__ faces,
                                             uint32_t n, uint32_t f, uint32_t v[3], float c[3][3])
{
#pragma unroll
    for (int k = 0; k < 3; k++) v[k] = (uint32_t)faces[3 * (size_t)f + k];
    if (v[0] >= n || v[1] >= n || v[2] >= n) return false;
#pragma unroll
    for (int k = 0; k < 3; k++)
#pragma unroll
        for (int j = 0; j < 3; j++) c[k][j] = xyz[3 * (size_t)v[k] + j];
    return true;
}

__device__ __forceinline__ bool degenerate(const uint32_t v[3]) { return v[0] == v[1] || v[1] == v[2] || v[0] == v[2]; }

// exclusive prefix sum of v over the POINT_BLOCK threads of the block (every thread calls it)
__device__ __forceinline__ uint32_t block_exclusive(uint32_t v)
{
    __shared__ uint32_t ws[POINT_BLOCK / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t s = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, s, o);
        if (lane >= o) s += t;
    }
    if (lane == 31) ws[w] = s;
    __syncthreads();
    if (w == 0) {
        uint32_t x = ws[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(FULL, x, o);
            if (lane >= o) x += t;
        }
        ws[lane] = x;
    }
    __syncthreads();
    return (w ? ws[w - 1] : 0u) + s - v;
}

__device__ __forceinline__ bool has_normal(const float* nrm, uint32_t i)
{
    return nrm[3 * (size_t)i] != 0.0f || nrm[3 * (size_t)i + 1] != 0.0f || nrm[3 * (size_t)i + 2] != 0.0f;
}

// (d, i) beats (bd, bi): the larger distance, a tie the smaller sample
__device__ __forceinline__ bool farther(double d, long long i, double bd, long long bi)
{
    return d > bd || (d == bd && i < bi);
}

}  // namespace

// one thread per face and per vertex: the finiteness and face-index checks, the cell box of a face and its entry
// count; counts[block] = the entries of the block's faces, state->entries their sum over the mesh
__global__ void __launch_bounds__(POINT_BLOCK) k_di_count(const float* __restrict__ xyz,
                                                          const int32_t* __restrict__ faces, uint32_t n, uint32_t nf,
                                                          double S, uint32_t* __restrict__ counts,
                                                          DistanceState* __restrict__ st)
{
    __shared__ unsigned long long ws[POINT_BLOCK / 32];
    const uint32_t i = blockIdx.x * POINT_BLOCK + threadIdx.x;
    bool bad = i < n && !finite3(xyz + 3 * (size_t)i), range = false;
    unsigned long long cnt = 0;
    if (i < nf) {
        uint32_t v[3];
        float c[3][3];
        if (!load_corners(xyz, faces, n, i, v, c)) {
            bad = true;
        } else if (finite3(c[0]) && finite3(c[1]) && finite3(c[2])) {
            long long lo[3], hi[3];
            if (!s3p::face_cells(c[0], c[1], c[2], S, lo, hi)) range = true;
            else if (!degenerate(v)) cnt = s3p::face_entries(lo, hi);
        }
    }
    unsigned long long s = cnt;
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    const bool any_bad = __syncthreads_or(bad), any_range = __syncthreads_or(range);
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int k = 0; k < POINT_BLOCK / 32; k++) t += ws[k];
        if ((uint64_t)blockIdx.x * POINT_BLOCK < (nf ? nf : 1)) counts[blockIdx.x] = (uint32_t)t;
        if (t) atomicAdd(&st->entries, t);
        if (any_bad) st->bad = 1;
        if (any_range) st->range = 1;
    }
}

// one thread per face (entries < 2^32, no error): each entry (face, cell) at its place, its cell into the table with
// the cell's count
__global__ void __launch_bounds__(POINT_BLOCK) k_di_insert(const float* __restrict__ xyz,
                                                           const int32_t* __restrict__ faces, uint32_t nf, double S,
                                                           const uint32_t* __restrict__ offsets, DistanceIndex ix)
{
    const uint32_t f = blockIdx.x * POINT_BLOCK + threadIdx.x;
    long long lo[3] = {0, 0, 0}, hi[3] = {-1, -1, -1};
    uint32_t cnt = 0;
    if (f < nf) {
        uint32_t v[3];
        float c[3][3];
        load_corners(xyz, faces, 0xffffffffu, f, v, c);
        if (!degenerate(v) && s3p::face_cells(c[0], c[1], c[2], S, lo, hi)) cnt = (uint32_t)s3p::face_entries(lo, hi);
    }
    uint32_t e = offsets[blockIdx.x] + block_exclusive(cnt);
    if (!cnt) return;
    for (long long z = lo[2]; z <= hi[2]; z++)
        for (long long y = lo[1]; y <= hi[1]; y++)
            for (long long x = lo[0]; x <= hi[0]; x++, e++) {
                bool claimed;
                const uint32_t s = find_or_insert(ix.keys, ix.cap, s3v::pack_key(x, y, z), &claimed);
                if (s != VOXEL_NO_SLOT) atomicAdd(&ix.cells[s].x, 1u);
                ix.entry_slot[e] = s;
                ix.entry_face[e] = f;
            }
}

// each occupied cell reserves its range: cells[s].y = its first id (the scatter advances it to the end)
__global__ void __launch_bounds__(IT) k_di_ranges(DistanceIndex ix)
{
    const int lane = threadIdx.x & 31;
    const uint32_t stride = gridDim.x * IT;
    for (uint32_t base = blockIdx.x * IT + (threadIdx.x & ~31u); base < ix.cap; base += stride) {
        const uint32_t s = base + lane;
        const uint32_t n = s < ix.cap ? ix.cells[s].x : 0u;
        uint32_t before = n;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL, before, off);
            if (lane >= off) before += v;
        }
        uint32_t first = 0;
        if (lane == 31 && before) first = atomicAdd(ix.cursor, before);
        first = __shfl_sync(FULL, first, 31);
        if (n) ix.cells[s].y = first + before - n;
    }
}

// one thread per entry: its face id into its cell's range
__global__ void __launch_bounds__(IT) k_di_scatter(DistanceIndex ix, uint32_t entries)
{
    const uint32_t e = blockIdx.x * IT + threadIdx.x;
    if (e >= entries) return;
    const uint32_t s = ix.entry_slot[e];
    if (s == VOXEL_NO_SLOT) return;
    ix.ids[atomicAdd(&ix.cells[s].y, 1u)] = ix.entry_face[e];
}

// one thread per sample: the nearest face within R, the outputs and the block's statistics (partials[block])
__global__ void __launch_bounds__(QT) k_di_query(DistanceIndex ix, const float* __restrict__ xyz,
                                                 const int32_t* __restrict__ faces, double S, double r2,
                                                 const float* __restrict__ smp, const float* __restrict__ nrm,
                                                 uint32_t ns, float* __restrict__ dist, int32_t* __restrict__ face_out,
                                                 DistancePartial* __restrict__ partials)
{
    __shared__ double red[QT / 32][3];
    __shared__ long long red_i[QT / 32];
    __shared__ float red_f[QT / 32][2];
    const uint32_t i = blockIdx.x * QT + threadIdx.x;
    bool sample = false, invalid = false, matched = false, inside = false;
    double best = 0.0, side = 0.0;
    uint32_t best_f = VOXEL_NO_SLOT;
    if (i < ns) {
        sample = !nrm || has_normal(nrm, i);
        if (sample) {
            const double p[3] = {smp[3 * (size_t)i], smp[3 * (size_t)i + 1], smp[3 * (size_t)i + 2]};
            long long c[3];
            invalid = !(p[0] - p[0] == 0.0 && p[1] - p[1] == 0.0 && p[2] - p[2] == 0.0);
            if (!invalid && s3l::cell_of(p, S, c)) {
                for (int dz = -1; dz <= 1; dz++)
                    for (int dy = -1; dy <= 1; dy++)
                        for (int dx = -1; dx <= 1; dx++) {
                            const long long a = c[0] + dx, b = c[1] + dy, e = c[2] + dz;
                            if (a < s3v::I_MIN || a >= s3v::I_MAX || b < s3v::I_MIN || b >= s3v::I_MAX ||
                                e < s3v::I_MIN || e >= s3v::I_MAX)
                                continue;
                            const uint32_t slot = find_slot(ix.keys, ix.cap, s3v::pack_key(a, b, e));
                            if (slot == VOXEL_NO_SLOT) continue;
                            const uint2 cell = ix.cells[slot];
                            for (uint32_t u = cell.y - cell.x; u < cell.y; u++) {
                                const uint32_t f = ix.ids[u];
                                if (f == best_f) continue;   // a face in several of the cells
                                uint32_t v[3];
                                float q[3][3];
                                load_corners(xyz, faces, 0xffffffffu, f, v, q);
                                double s;
                                const double d2 = s3p::face_distance(p, q[0], q[1], q[2], &s);
                                if (d2 <= r2 && (best_f == VOXEL_NO_SLOT || s3p::closer(d2, f, best, best_f))) {
                                    best = d2;
                                    best_f = f;
                                    side = s;
                                }
                            }
                        }
            }
        }
        matched = best_f != VOXEL_NO_SLOT;
        inside = matched && side < 0.0;
        if (dist) dist[i] = matched ? s3p::signed_distance(best, side) : __int_as_float(0x7fc00000);
        if (face_out) face_out[i] = matched ? (int32_t)best_f : -1;
    }
    const double d = matched ? s3p::root(best) : 0.0, d2 = matched ? best : 0.0;
    const float sd = matched ? s3p::signed_distance(best, side) : 0.0f;
    double x[3] = {d, d2, matched ? d : -1.0};
    long long xi = matched ? (long long)i : -1;
    float mn = matched ? sd : __int_as_float(0x7f800000), mx = matched ? sd : __int_as_float(0xff800000);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        x[0] = __dadd_rn(x[0], __shfl_down_sync(FULL, x[0], off));
        x[1] = __dadd_rn(x[1], __shfl_down_sync(FULL, x[1], off));
        const double od = __shfl_down_sync(FULL, x[2], off);
        const long long oi = __shfl_down_sync(FULL, xi, off);
        if (oi >= 0 && (xi < 0 || farther(od, oi, x[2], xi))) x[2] = od, xi = oi;
        mn = fminf(mn, __shfl_down_sync(FULL, mn, off));
        mx = fmaxf(mx, __shfl_down_sync(FULL, mx, off));
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) {
        red[w][0] = x[0], red[w][1] = x[1], red[w][2] = x[2];
        red_i[w] = xi;
        red_f[w][0] = mn, red_f[w][1] = mx;
    }
    const uint32_t n_sample = __syncthreads_count(sample), n_matched = __syncthreads_count(matched);
    const uint32_t n_invalid = __syncthreads_count(invalid), n_inside = __syncthreads_count(inside);
    if (threadIdx.x != 0) return;
    DistancePartial r;
    r.sum_d = red[0][0], r.sum_d2 = red[0][1], r.max_d = red[0][2], r.max_sample = red_i[0];
    r.min_signed = red_f[0][0], r.max_signed = red_f[0][1];
    for (int k = 1; k < QT / 32; k++) {
        r.sum_d = __dadd_rn(r.sum_d, red[k][0]);
        r.sum_d2 = __dadd_rn(r.sum_d2, red[k][1]);
        if (red_i[k] >= 0 && (r.max_sample < 0 || farther(red[k][2], red_i[k], r.max_d, r.max_sample)))
            r.max_d = red[k][2], r.max_sample = red_i[k];
        r.min_signed = fminf(r.min_signed, red_f[k][0]);
        r.max_signed = fmaxf(r.max_signed, red_f[k][1]);
    }
    r.samples = n_sample, r.matched = n_matched, r.invalid = n_invalid, r.inside = n_inside;
    partials[blockIdx.x] = r;
}

// one block: the partials of all query blocks, summed in the order of common/scan3d_distance_math.h
__global__ void __launch_bounds__(QT) k_di_stats(const DistancePartial* __restrict__ partials, uint32_t blocks,
                                                 DistanceState* __restrict__ st)
{
    __shared__ double buf[2][QT];
    __shared__ DistancePartial best[QT];
    __shared__ unsigned long long cnt[4][QT];
    double a = 0.0, b = 0.0;
    DistancePartial m;
    m.max_d = -1.0, m.max_sample = -1;
    m.min_signed = __int_as_float(0x7f800000), m.max_signed = __int_as_float(0xff800000);
    unsigned long long c[4] = {0, 0, 0, 0};
    for (uint32_t k = threadIdx.x; k < blocks; k += QT) {
        const DistancePartial& p = partials[k];
        a = __dadd_rn(a, p.sum_d);
        b = __dadd_rn(b, p.sum_d2);
        if (p.max_sample >= 0 && (m.max_sample < 0 || farther(p.max_d, p.max_sample, m.max_d, m.max_sample)))
            m.max_d = p.max_d, m.max_sample = p.max_sample;
        m.min_signed = fminf(m.min_signed, p.min_signed);
        m.max_signed = fmaxf(m.max_signed, p.max_signed);
        c[0] += p.samples, c[1] += p.matched, c[2] += p.invalid, c[3] += p.inside;
    }
    buf[0][threadIdx.x] = a;
    buf[1][threadIdx.x] = b;
    best[threadIdx.x] = m;
    for (int k = 0; k < 4; k++) cnt[k][threadIdx.x] = c[k];
    __syncthreads();
    for (int h = QT / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) {
            const int o = threadIdx.x + h;
            buf[0][threadIdx.x] = __dadd_rn(buf[0][threadIdx.x], buf[0][o]);
            buf[1][threadIdx.x] = __dadd_rn(buf[1][threadIdx.x], buf[1][o]);
            DistancePartial& x = best[threadIdx.x];
            const DistancePartial& y = best[o];
            if (y.max_sample >= 0 && (x.max_sample < 0 || farther(y.max_d, y.max_sample, x.max_d, x.max_sample)))
                x.max_d = y.max_d, x.max_sample = y.max_sample;
            x.min_signed = fminf(x.min_signed, y.min_signed);
            x.max_signed = fmaxf(x.max_signed, y.max_signed);
            for (int k = 0; k < 4; k++) cnt[k][threadIdx.x] += cnt[k][o];
        }
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    const bool any = cnt[1][0] != 0;
    st->sum_d = buf[0][0];
    st->sum_d2 = buf[1][0];
    st->max_d = any ? best[0].max_d : 0.0;
    st->max_sample = any ? best[0].max_sample : -1;
    st->min_signed = any ? best[0].min_signed : 0.0f;
    st->max_signed = any ? best[0].max_signed : 0.0f;
    st->samples = cnt[0][0], st->matched = cnt[1][0], st->invalid = cnt[2][0], st->inside = cnt[3][0];
}

cudaError_t DistanceWorkspace::count(const float* xyz, const int32_t* faces, uint32_t n, uint32_t nf, double S,
                                     cudaStream_t st, int64_t* launches)
{
    const unsigned nbf = grid(nf, POINT_BLOCK), nbv = grid(n, POINT_BLOCK);
    cudaError_t e = face_counts.ensure(nbf);
    if (e == cudaSuccess) e = state.ensure(1);
    if (e == cudaSuccess) e = cudaMemsetAsync(state, 0, sizeof(DistanceState), st);
    if (e != cudaSuccess) return e;
    k_di_count<<<nbf > nbv ? nbf : nbv, POINT_BLOCK, 0, st>>>(xyz, faces, n, nf, S, face_counts, state);
    e = launch_block_scan(face_counts, (int)nbf, &state.get()->entries32, st);
    *launches += 2;
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t DistanceWorkspace::query(const float* xyz, const int32_t* faces, uint32_t nf, uint32_t entries, double S,
                                     double r2, const float* samples, const float* nrm, uint32_t ns, float* dist,
                                     int32_t* face, cudaStream_t st, int64_t* launches)
{
    const unsigned long long want = (unsigned long long)CELLS_PER_ENTRY * entries;
    const uint32_t cap = want < 64 ? 64u : want > 0xffffffffull ? 0xffffffffu : (uint32_t)want;
    const unsigned nbq = grid(ns, QT);
    table = cap;
    cudaError_t e = grow_group(Grow(keys, cap), Grow(cells, cap));
    if (e == cudaSuccess) e = grow_group(Grow(entry_slot, entries ? entries : 1), Grow(entry_face, entries ? entries : 1),
                                         Grow(ids, entries ? entries : 1));
    if (e == cudaSuccess) e = partials.ensure(nbq);
    if (e == cudaSuccess) e = cursor.ensure(1);
    if (e != cudaSuccess) return e;
    const DistanceIndex ix{keys, cells, entry_slot, entry_face, ids, cursor, cap};
    e = cudaMemsetAsync(ix.keys, 0xff, (size_t)cap * sizeof(*ix.keys), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ix.cells, 0, (size_t)cap * sizeof(*ix.cells), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ix.cursor, 0, sizeof(*ix.cursor), st);
    if (e != cudaSuccess) return e;
    k_di_insert<<<grid(nf, POINT_BLOCK), POINT_BLOCK, 0, st>>>(xyz, faces, nf, S, face_counts, ix);
    k_di_ranges<<<grid(cap, IT) < 1024u ? grid(cap, IT) : 1024u, IT, 0, st>>>(ix);
    k_di_scatter<<<grid(entries, IT), IT, 0, st>>>(ix, entries);
    k_di_query<<<nbq, QT, 0, st>>>(ix, xyz, faces, S, r2, samples, nrm, ns, dist, face, partials);
    k_di_stats<<<1, QT, 0, st>>>(partials, nbq, state);
    *launches += 5;
    return cudaGetLastError();
}

}  // namespace s3d
