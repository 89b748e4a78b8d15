// scan3d_mesh_kernels.cu -- the camera-grid mesh of the compacted points (scan3d_build_mesh): triangle faces
// between neighbouring valid pixels and area-weighted per-vertex normals.  A bandwidth-bound post-pass: the
// arithmetic is in common/scan3d_mesh_math.h, shared with the host test.
//
// Every kernel works on the blocks of POINT_BLOCK consecutive raster pixels that k_count / k_scan use for the
// point offsets, 4 pixels per thread.  Faces are numbered in raster order of their cells (T1 before
// T2), so a block's faces and its points are both contiguous ranges of the outputs: the emit kernel stages them
// in shared memory and writes each range with 16-byte stores.
#include "scan3d_internal.h"
#include "../common/scan3d_mesh_math.h"

namespace s3d {

namespace {

constexpr int MT = 256;                 // threads per block
constexpr int MPT = POINT_BLOCK / MT;   // pixels per thread
static_assert(MPT == 4, "k_mesh_index: 4 consecutive pixels per thread (one 16-byte index vector)");

// Exclusive prefix of v[k] over the block in phase-major order (phase k of every thread before phase k + 1, threads
// in order within a phase); *total = the block's sum.  One barrier.
__device__ __forceinline__ void block_phase_scan(const uint32_t (&v)[MPT], uint32_t (&ex)[MPT], uint32_t* total)
{
    __shared__ uint32_t wsum[MPT][MT / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t s[MPT];
#pragma unroll
    for (int k = 0; k < MPT; k++) {
        s[k] = v[k];
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, s[k], o);
            if (lane >= o) s[k] += t;
        }
        if (lane == 31) wsum[k][w] = s[k];
    }
    __syncthreads();
    uint32_t base = 0;
#pragma unroll
    for (int k = 0; k < MPT; k++) {
        uint32_t before = 0, all = 0;
#pragma unroll
        for (int i = 0; i < MT / 32; i++) {
            const uint32_t x = wsum[k][i];
            before += i < w ? x : 0;
            all += x;
        }
        ex[k] = base + before + s[k] - v[k];
        base += all;
    }
    *total = base;
}

// pixel (r, c) as a mesh vertex: outside the grid or invalid -> ok = false
__device__ __forceinline__ s3m::MeshPt fetch(const int32_t* __restrict__ idx, const float* __restrict__ pts, int W,
                                              int H, int r, int c, int32_t* i_out = nullptr)
{
    s3m::MeshPt q{0.0f, 0.0f, 0.0f, false};
    int32_t i = -1;
    if (r >= 0 && r < H && c >= 0 && c < W) i = __ldg(idx + (size_t)r * W + c);
    if (i >= 0) {
        q.x = __ldg(pts + 3 * (size_t)i);
        q.y = __ldg(pts + 3 * (size_t)i + 1);
        q.z = __ldg(pts + 3 * (size_t)i + 2);
        q.ok = true;
    }
    if (i_out) *i_out = i;
    return q;
}

// n 32-bit words from shared memory to g (4-byte aligned): scalar head and tail, 16-byte stores between
__device__ __forceinline__ void store_range(const uint32_t* s, uint32_t* __restrict__ g, int n)
{
    int head = (int)(((16 - ((uintptr_t)g & 15)) & 15) >> 2);
    head = head < n ? head : n;
    const int nv = (n - head) >> 2;
    for (int k = threadIdx.x; k < head; k += MT) g[k] = s[k];
    uint4* gv = reinterpret_cast<uint4*>(g + head);
    for (int k = threadIdx.x; k < nv; k += MT) {
        const uint32_t* q = s + head + 4 * k;
        gv[k] = make_uint4(q[0], q[1], q[2], q[3]);
    }
    for (int k = head + 4 * nv + threadIdx.x; k < n; k += MT) g[k] = s[k];
}

}  // namespace

// idx[p] = point index of pixel p (its rank among the valid pixels in raster order), -1 if invalid
__global__ void __launch_bounds__(MT) k_mesh_index(const uint8_t* __restrict__ valid, const uint32_t* __restrict__ offsets,
                                                   int32_t* __restrict__ idx, size_t plane)
{
    const size_t p0 = (size_t)blockIdx.x * POINT_BLOCK + (size_t)MPT * threadIdx.x;
    bool v[MPT];
    if (p0 + MPT <= plane) {
        const uchar4 q = *reinterpret_cast<const uchar4*>(valid + p0);
        v[0] = q.x != 0; v[1] = q.y != 0; v[2] = q.z != 0; v[3] = q.w != 0;
    } else {
        for (int j = 0; j < MPT; j++) v[j] = p0 + j < plane && valid[p0 + j] != 0;
    }
    const uint32_t n[MPT] = {(uint32_t)v[0] + v[1] + v[2] + v[3], 0, 0, 0};
    uint32_t ex[MPT], total;
    block_phase_scan(n, ex, &total);
    uint32_t rank = offsets[blockIdx.x] + ex[0];
    int32_t out[MPT];
    for (int j = 0; j < MPT; j++) out[j] = v[j] ? (int32_t)rank++ : -1;
    if (p0 + MPT <= plane) {
        *reinterpret_cast<int4*>(idx + p0) = make_int4(out[0], out[1], out[2], out[3]);
    } else {
        for (int j = 0; j < MPT; j++)
            if (p0 + j < plane) idx[p0 + j] = out[j];
    }
}

// faces of the cells whose top-left corner lies in the block (pixel base + k MT + thread of phase k: every load of a
// warp covers consecutive pixels)
__global__ void __launch_bounds__(MT) k_mesh_count(const int32_t* __restrict__ idx, const float* __restrict__ pts, int W,
                                                   int H, float t2, uint32_t* __restrict__ face_counts)
{
    const size_t plane = (size_t)W * H;
    uint32_t n[MPT], ex[MPT], total;
#pragma unroll
    for (int k = 0; k < MPT; k++) {
        const size_t p = (size_t)blockIdx.x * POINT_BLOCK + (size_t)k * MT + threadIdx.x;
        const int r = (int)(p / (size_t)W), c = (int)(p - (size_t)r * W);
        n[k] = 0;
        if (p < plane && r < H - 1 && c < W - 1) {
            const s3m::MeshPt a = fetch(idx, pts, W, H, r, c), b = fetch(idx, pts, W, H, r, c + 1);
            const s3m::MeshPt d = fetch(idx, pts, W, H, r + 1, c), e = fetch(idx, pts, W, H, r + 1, c + 1);
            n[k] = __popc(s3m::cell_faces(a, b, d, e, t2));
        }
    }
    block_phase_scan(n, ex, &total);
    if (threadIdx.x == 0) face_counts[blockIdx.x] = total;
}

// faces at the block's face offset, normals at the block's point offset
__global__ void __launch_bounds__(MT) k_mesh_emit(const int32_t* __restrict__ idx, const float* __restrict__ pts, int W,
                                                  int H, float t2, const uint32_t* __restrict__ point_offsets,
                                                  const uint32_t* __restrict__ face_offsets, int32_t* __restrict__ faces,
                                                  float* __restrict__ normals)
{
    __shared__ uint32_t s_faces[2 * POINT_BLOCK * 3];
    __shared__ uint32_t s_normals[POINT_BLOCK * 3];
    const size_t plane = (size_t)W * H;
    int32_t corner[MPT][4];   // point indices of a, b, d, e of the pixel's cell
    int bits[MPT];
    float nrm[MPT][3];
    uint32_t cnt[MPT];
#pragma unroll
    for (int j = 0; j < MPT; j++) {
        const size_t p = (size_t)blockIdx.x * POINT_BLOCK + (size_t)j * MT + threadIdx.x;
        const int r = (int)(p / (size_t)W), c = (int)(p - (size_t)r * W);
        bits[j] = 0;
        corner[j][0] = -1;
        cnt[j] = 0;
        if (p < plane) {
            s3m::MeshPt nb[3][3];
            nb[0][0].ok = false;
            nb[0][1] = fetch(idx, pts, W, H, r - 1, c);
            nb[0][2] = fetch(idx, pts, W, H, r - 1, c + 1);
            nb[1][0] = fetch(idx, pts, W, H, r, c - 1);
            nb[1][1] = fetch(idx, pts, W, H, r, c, &corner[j][0]);
            nb[1][2] = fetch(idx, pts, W, H, r, c + 1, &corner[j][1]);
            nb[2][0] = fetch(idx, pts, W, H, r + 1, c - 1);
            nb[2][1] = fetch(idx, pts, W, H, r + 1, c, &corner[j][2]);
            const s3m::MeshPt e = fetch(idx, pts, W, H, r + 1, c + 1, &corner[j][3]);
            if (r < H - 1 && c < W - 1) bits[j] = s3m::cell_faces(nb[1][1], nb[1][2], nb[2][1], e, t2);
            s3m::vertex_normal(nb, t2, nrm[j]);
            // one scan for both counts: faces (<= 2 POINT_BLOCK a block) in the high half, points in the low half
            cnt[j] = ((uint32_t)__popc(bits[j]) << 16) | (nb[1][1].ok ? 1u : 0u);
        }
    }
    uint32_t ex[MPT], total;
    block_phase_scan(cnt, ex, &total);
#pragma unroll
    for (int j = 0; j < MPT; j++) {
        uint32_t f = ex[j] >> 16;
        const uint32_t q = ex[j] & 0xffffu;
        const int32_t ia = corner[j][0], ib = corner[j][1], id = corner[j][2], ie = corner[j][3];
        if (bits[j] & 1) {
            s_faces[3 * f] = ia; s_faces[3 * f + 1] = id; s_faces[3 * f + 2] = ib;
            f++;
        }
        if (bits[j] & 2) {
            s_faces[3 * f] = ib; s_faces[3 * f + 1] = id; s_faces[3 * f + 2] = ie;
            f++;
        }
        if (ia >= 0) {
            s_normals[3 * q] = __float_as_uint(nrm[j][0]);
            s_normals[3 * q + 1] = __float_as_uint(nrm[j][1]);
            s_normals[3 * q + 2] = __float_as_uint(nrm[j][2]);
        }
    }
    __syncthreads();
    store_range(s_faces, reinterpret_cast<uint32_t*>(faces) + 3 * (size_t)face_offsets[blockIdx.x], 3 * (int)(total >> 16));
    store_range(s_normals, reinterpret_cast<uint32_t*>(normals) + 3 * (size_t)point_offsets[blockIdx.x],
                3 * (int)(total & 0xffffu));
}

cudaError_t launch_mesh(const uint8_t* valid, const float* pts, int W, int H, float max_edge, int32_t* idx,
                        uint32_t* block_counts, uint32_t* face_counts, uint32_t* totals, int32_t* faces, float* normals,
                        cudaStream_t st, int64_t* launches)
{
    const size_t plane = (size_t)W * H;
    const int nb = (int)((plane + POINT_BLOCK - 1) / POINT_BLOCK);
    const float t2 = s3m::edge_t2(max_edge);
    cudaError_t e = launch_point_offsets(valid, plane, block_counts, totals, st);
    if (e != cudaSuccess) return e;
    k_mesh_index<<<nb, MT, 0, st>>>(valid, block_counts, idx, plane);
    k_mesh_count<<<nb, MT, 0, st>>>(idx, pts, W, H, t2, face_counts);
    e = launch_block_scan(face_counts, nb, totals + 1, st);
    if (e != cudaSuccess) return e;
    k_mesh_emit<<<nb, MT, 0, st>>>(idx, pts, W, H, t2, block_counts, face_counts, faces, normals);
    *launches += 6;
    return cudaGetLastError();
}

}  // namespace s3d
