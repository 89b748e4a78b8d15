// scan3d_align_kernels.cu -- point-to-plane ICP of a source cloud against the merged voxel cloud
// (scan3d_align_to_voxels*).  The arithmetic is in common/scan3d_align_math.h, shared with the host test; this file
// owns the model's cell index, the reduction order and the device-side iteration state.
//
// Index (3 launches): the model points (voxel outputs with a non-zero normal) are hashed by their cell of edge
// S = max_distance (1 + 2^-20) into an open-addressing table (scan3d_hash.cuh) with a point count per cell; the cells
// then reserve their ranges of the entry array through a cursor (one atomic per warp of slots), and the points are
// scattered into their ranges with their coordinates and normals beside the ordinal.  The order inside a range varies from run to run; the
// selection cannot, because it is by (distance, ordinal).
//
// Iteration (2 launches): k_align_match gives each thread SPT samples (sample j = point j * stride, block b takes
// samples [b SPB, (b + 1) SPB)), probes the 27 cells around each transformed sample, keeps the nearest model point
// within max_distance and adds the pair's 28 products to per-thread sums; the block reduces them in a fixed tree
// (warp shuffles, then the 8 warps in order) to one partial per block.  k_align_solve (one block) sums the partials in
// a fixed order -- thread t adds blocks t, t + 256, ... in turn, then a shared-memory tree -- solves, updates T and
// decides whether the run is over.  The grid depends only on the sample bound, and blocks past the last sample
// contribute exact zeros, so the result does not depend on the SM count or on scheduling, and a bound larger than the
// sample count (the ctx route reads its count on the device) gives the same bits.  After the run ends both kernels
// return at once, so the launch count is fixed.
#include "scan3d_internal.h"
#include "scan3d_hash.cuh"
#include "../common/scan3d_align_math.h"

namespace s3d {

namespace {

constexpr int IT = 256;                  // threads per block of the index kernels
constexpr int MT = 256;                  // threads per match block
constexpr int SPT = 8;                   // samples per match thread
constexpr long long SPB = (long long)MT * SPT;
constexpr int NV = s3l::NSUM + 1;        // the sums and the pair count
constexpr unsigned FULL = 0xffffffffu;
constexpr uint32_t CELLS_PER_VOXEL = 2;  // index slots per model voxel: at most half of them are taken

__device__ __forceinline__ uint32_t model_count(const VoxelTable& t, int par)
{
    return min(t.state->total[par], t.max_voxels);
}

__device__ __forceinline__ bool has_normal(const float* nrm, uint32_t o)
{
    return nrm[3 * (size_t)o] != 0.0f || nrm[3 * (size_t)o + 1] != 0.0f || nrm[3 * (size_t)o + 2] != 0.0f;
}

}  // namespace

// the cell of every model point, and the point count per cell; block 0 also initialises the run's state
__global__ void __launch_bounds__(IT) k_align_cells(AlignIndex ix, VoxelTable t, int par, const float* __restrict__ xyz,
                                                    const float* __restrict__ nrm, double S, AlignState* __restrict__ st,
                                                    AlignRun run, const uint32_t* __restrict__ n_dev)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (int k = 0; k < 12; k++) st->T[k] = run.T0[k];
        st->rms_first = st->rms_last = 0.0;
        st->pairs_first = st->pairs_last = 0;
        st->iterations = st->status = st->done = st->rounds = 0;
        st->overflow = t.state->overflow || t.state->occupied > t.max_voxels;
        st->n_src = n_dev ? *n_dev : 0u;
    }
    const uint32_t m = model_count(t, par);
    for (uint32_t o = blockIdx.x * IT + threadIdx.x; o < m; o += gridDim.x * IT) {
        uint32_t slot = VOXEL_NO_SLOT;
        const double p[3] = {xyz[3 * (size_t)o], xyz[3 * (size_t)o + 1], xyz[3 * (size_t)o + 2]};
        long long c[3];
        if (has_normal(nrm, o) && s3l::cell_of(p, S, c)) {
            bool claimed;
            slot = find_or_insert(ix.keys, ix.cap, s3v::pack_key(c[0], c[1], c[2]), &claimed);
            if (slot != VOXEL_NO_SLOT) atomicAdd(&ix.cells[slot].x, 1u);
        }
        ix.model_slot[o] = slot;
    }
}

// each occupied cell reserves its range: cells[s].y = its first entry (the scatter advances it to the end).  A warp
// reserves the ranges of its 32 slots with one atomic on the cursor (one per cell serialised on a single address).
__global__ void __launch_bounds__(IT) k_align_ranges(AlignIndex ix)
{
    const int lane = threadIdx.x & 31;
    const uint32_t stride = gridDim.x * IT;
    for (uint32_t base = blockIdx.x * IT + (threadIdx.x & ~31u); base < ix.cap; base += stride) {
        const uint32_t s = base + lane;
        const uint32_t n = s < ix.cap ? ix.cells[s].x : 0u;
        uint32_t before = n;                               // inclusive prefix sum over the warp
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

__global__ void __launch_bounds__(IT) k_align_scatter(AlignIndex ix, VoxelTable t, int par, const float* __restrict__ xyz,
                                                      const float* __restrict__ nrm)
{
    const uint32_t m = model_count(t, par);
    for (uint32_t o = blockIdx.x * IT + threadIdx.x; o < m; o += gridDim.x * IT) {
        const uint32_t s = ix.model_slot[o];
        if (s == VOXEL_NO_SLOT) continue;
        const size_t e = atomicAdd(&ix.cells[s].y, 1u);
        ix.entries[2 * e] = make_float4(xyz[3 * (size_t)o], xyz[3 * (size_t)o + 1], xyz[3 * (size_t)o + 2],
                                        __uint_as_float(o));
        ix.entries[2 * e + 1] = make_float4(nrm[3 * (size_t)o], nrm[3 * (size_t)o + 1], nrm[3 * (size_t)o + 2], 0.0f);
    }
}

// one partial of the sums per block; partials[v * gridDim.x + block]
__global__ void __launch_bounds__(MT) k_align_match(AlignIndex ix, const AlignState* __restrict__ st, AlignRun run,
                                                    const float* __restrict__ xyz, const uint32_t* __restrict__ n_dev,
                                                    long long n_max, int stride, double* __restrict__ partials)
{
    __shared__ double T[12];
    __shared__ double red[MT / 32][NV];
    if (*(volatile const int*)&st->done) return;
    if (threadIdx.x < 12) T[threadIdx.x] = st->T[threadIdx.x];
    __syncthreads();
    const long long n = n_dev ? min((long long)*n_dev, n_max) : n_max;
    const long long samples = (n + stride - 1) / stride;
    double s[s3l::NSUM];
#pragma unroll
    for (int k = 0; k < s3l::NSUM; k++) s[k] = 0.0;
    double pairs = 0.0;
    for (int k = 0; k < SPT; k++) {
        const long long j = (long long)blockIdx.x * SPB + (long long)k * MT + threadIdx.x;
        if (j >= samples) break;
        const size_t i = (size_t)j * (size_t)stride;
        double p[3];
        s3l::transform(T, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], p);
        uint32_t best_e;
        if (align_nearest(ix, p, run.S, run.r2, &best_e) == VOXEL_NO_SLOT) continue;
        const float4 q = ix.entries[2 * (size_t)best_e], nq = ix.entries[2 * (size_t)best_e + 1];
        double J[6], r;
        s3l::row(p, q.x, q.y, q.z, nq.x, nq.y, nq.z, J, &r);
        s3l::accumulate(J, r, s);
        pairs = __dadd_rn(pairs, 1.0);
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int v = 0; v < NV; v++) {
        double x = v < s3l::NSUM ? s[v] : pairs;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) x = __dadd_rn(x, __shfl_down_sync(FULL, x, off));
        if (lane == 0) red[w][v] = x;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double a = red[0][threadIdx.x];
        for (int k = 1; k < MT / 32; k++) a = __dadd_rn(a, red[k][threadIdx.x]);
        partials[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = a;
    }
}

// the sums of all blocks, the solve and the update of T
__global__ void __launch_bounds__(MT) k_align_solve(AlignState* __restrict__ st, AlignRun run,
                                                    const double* __restrict__ partials, uint32_t blocks)
{
    __shared__ double buf[MT];
    __shared__ double tot[NV];
    if (*(volatile const int*)&st->done) return;
    for (int v = 0; v < NV; v++) {
        double a = 0.0;
        for (uint32_t b = threadIdx.x; b < blocks; b += MT) a = __dadd_rn(a, partials[(size_t)v * blocks + b]);
        buf[threadIdx.x] = a;
        __syncthreads();
        for (int h = MT / 2; h > 0; h >>= 1) {
            if (threadIdx.x < h) buf[threadIdx.x] = __dadd_rn(buf[threadIdx.x], buf[threadIdx.x + h]);
            __syncthreads();
        }
        if (threadIdx.x == 0) tot[v] = buf[0];
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    const long long pairs = (long long)tot[s3l::NSUM];
    const double rms = s3l::rms(tot[27], pairs);
    if (st->rounds == 0) {
        st->pairs_first = pairs;
        st->rms_first = rms;
    }
    st->pairs_last = pairs;
    st->rms_last = rms;
    st->rounds++;
    double x[6], dR[9], th;
    if (pairs < 6 || !s3l::solve6(tot, x) || !s3l::rodrigues(x, dR, &th)) {
        st->status = 2;
        st->done = 1;
        return;
    }
    double T[12];
    for (int k = 0; k < 12; k++) T[k] = st->T[k];
    s3l::compose(dR, x + 3, T);
    for (int k = 0; k < 12; k++) st->T[k] = T[k];
    st->iterations++;
    if (s3l::converged(th, x + 3, run.stop_rotation, run.stop_translation)) {
        st->status = 0;
        st->done = 1;
    } else if (st->iterations >= run.max_iterations) {
        st->status = 1;
        st->done = 1;
    }
}

static unsigned index_grid(unsigned long long n, int sm_count)
{
    unsigned long long b = (n + IT - 1) / IT;
    const unsigned long long cap = 8ull * (unsigned)sm_count;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

static uint32_t match_blocks(long long n_max, int stride)
{
    const long long samples = (n_max + stride - 1) / stride;
    const long long b = (samples + SPB - 1) / SPB;
    return (uint32_t)(b < 1 ? 1 : b);
}

cudaError_t AlignWorkspace::index(const VoxelTable& t, int par, const float* xyz, const float* nrm, const AlignRun& run,
                                  const uint32_t* n_dev, int sm_count, cudaStream_t st, int64_t* launches)
{
    const uint32_t maxv = t.max_voxels, cap = CELLS_PER_VOXEL * maxv;
    cudaError_t e =
        grow_group(Grow(keys, cap), Grow(cells, cap), Grow(model_slot, maxv), Grow(entries, 2 * (size_t)maxv));
    if (e == cudaSuccess) e = state.ensure(1);
    if (e == cudaSuccess) e = cursor.ensure(1);
    if (e != cudaSuccess) return e;
    view = AlignIndex{keys, cells, model_slot, entries, cursor, cap};
    e = cudaMemsetAsync(keys, 0xff, (size_t)cap * sizeof(*view.keys), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(cells, 0, (size_t)cap * sizeof(*view.cells), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(cursor, 0, sizeof(*view.cursor), st);
    if (e != cudaSuccess) return e;
    const unsigned gm = index_grid(maxv, sm_count);
    k_align_cells<<<gm, IT, 0, st>>>(view, t, par, xyz, nrm, run.S, state, run, n_dev);
    k_align_ranges<<<index_grid(cap, sm_count), IT, 0, st>>>(view);
    k_align_scatter<<<gm, IT, 0, st>>>(view, t, par, xyz, nrm);
    *launches += 3;
    return cudaGetLastError();
}

cudaError_t AlignWorkspace::align(const VoxelTable& t, int par, const float* xyz, const float* nrm, const AlignRun& run,
                                  const float* src, const uint32_t* n_dev, long long n_max, int stride, int sm_count,
                                  cudaStream_t st, int64_t* launches)
{
    const uint32_t blocks = match_blocks(n_max, stride);
    cudaError_t e = partials.ensure((size_t)NV * blocks);
    if (e == cudaSuccess) e = index(t, par, xyz, nrm, run, n_dev, sm_count, st, launches);
    for (int it = 0; it < run.max_iterations && e == cudaSuccess; it++) {
        k_align_match<<<blocks, MT, 0, st>>>(view, state, run, src, n_dev, n_max, stride, partials);
        k_align_solve<<<1, MT, 0, st>>>(state, run, partials, blocks);
        *launches += 2;
        e = cudaGetLastError();
    }
    return e;
}

}  // namespace s3d
