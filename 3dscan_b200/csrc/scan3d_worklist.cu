// scan3d_worklist.cu -- work list of the single-pass kernel: the tiles that hold at least one ROI pixel.
// Tiles without any selected pixel never enter the persistent kernel: their outputs (phase 0, fringe order -1,
// valid 0, c_p_map 0) are written right here and their frame segments are never read.
#include "scan3d_fused_common.cuh"

namespace s3d {

int fused_num_tiles(const scan3d_config& c)
{
    // upper bound of the single-pass kernel's tile count (its tiles hold at least 128 pixels)
    return (int)(((size_t)c.W * c.H + 127) / 128) + 1;
}

// ---- work list: tiles that contain at least one ROI pixel ---------------------------------------
// One warp per tile looks at the tile's ROI bytes.  Tiles without any selected pixel never enter
// the main kernel: their outputs (phase 0, fringe order -1, valid 0, c_p_map 0) are written right
// here and their 56 input frame segments are never read.  The flags are then compacted, in raster
// order, into the work list the persistent kernel walks in phase-aligned rounds.
__global__ void k_tile_flags(const uint8_t* __restrict__ roi, int T, int plane, int n_tiles, size_t roi_off,
                             uint8_t* __restrict__ flags, float* __restrict__ unw_v, float* __restrict__ unw_h,
                             int16_t* __restrict__ code_v, int16_t* __restrict__ code_h, uint8_t* __restrict__ valid,
                             int2* __restrict__ cpmap, int dirs)
{
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t >= n_tiles) return;
    const int p0 = t * T, wt = min(T, plane - p0);
    const uint4* r = reinterpret_cast<const uint4*>(roi + roi_off + p0);
    bool any = false;
    for (int i = lane; i < wt / 16; i += 32) {
        const uint4 v = r[i];
        any |= (v.x | v.y | v.z | v.w) != 0;
    }
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) flags[t] = any ? 1 : 0;
    if (any) return;
    const uint4 z = make_uint4(0, 0, 0, 0), m1 = make_uint4(~0u, ~0u, ~0u, ~0u);
    for (int i = lane; i < wt / 4; i += 32) {       // 4 floats
        reinterpret_cast<uint4*>(unw_v + p0)[i] = z;
        if (dirs == 2) reinterpret_cast<uint4*>(unw_h + p0)[i] = z;
    }
    for (int i = lane; i < wt / 8; i += 32) {       // 8 int16 = -1
        reinterpret_cast<uint4*>(code_v + p0)[i] = m1;
        if (dirs == 2) reinterpret_cast<uint4*>(code_h + p0)[i] = m1;
    }
    for (int i = lane; i < wt / 16; i += 32) reinterpret_cast<uint4*>(valid + p0)[i] = z;
    if (dirs == 2)
        for (int i = lane; i < wt / 2; i += 32) reinterpret_cast<uint4*>(cpmap + p0)[i] = z;
}

// exclusive scan of the flags by one CTA -> list of non-empty tile ids (raster order) + its length.
// Each thread owns a contiguous chunk of flags, so one block-wide scan suffices.
__global__ void k_tile_list(const uint8_t* __restrict__ flags, int n_tiles, int* __restrict__ list,
                            int* __restrict__ n_list, uint32_t* __restrict__ d_count)
{
    __shared__ int wsum[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int per = (n_tiles + 1023) / 1024;
    const int i0 = threadIdx.x * per, i1 = min(n_tiles, i0 + per);
    int cnt = 0;
    for (int i = i0; i < i1; i++) cnt += flags[i] != 0;
    int incl = cnt;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    if (w == 0) {
        int v = wsum[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += t;
        }
        wsum[lane] = v;   // inclusive over warps
    }
    __syncthreads();
    int pos = (w ? wsum[w - 1] : 0) + incl - cnt;
    for (int i = i0; i < i1; i++)
        if (flags[i]) list[pos++] = i;
    if (threadIdx.x == 0) {
        *n_list = wsum[31];
        n_list[n_tiles + 8] = 0;   // the fused kernel's counter: next work-list position
        *d_count = 0;   // overwritten by the fused kernel's last tile when there is any work
    }
}

cudaError_t launch_worklist(const FusedArgs& a, int T, int dirs, cudaStream_t st)
{
    k_tile_flags<<<(a.n_tiles + 7) / 8, 256, 0, st>>>(a.roi_list ? a.roi_list : a.roi, T, a.W * a.H, a.n_tiles, (size_t)a.row0 * a.W, a.tile_flags,
                                                      a.unw_v, a.unw_h, a.code_v, a.code_h, a.valid, a.cpmap, dirs);
    k_tile_list<<<1, 1024, 0, st>>>(a.tile_flags, a.n_tiles, a.tile_list, a.n_list, a.d_count);
    return cudaGetLastError();
}

}  // namespace s3d
