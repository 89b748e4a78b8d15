// scan3d_internal.h -- context layout and kernel launcher declarations (not part of the ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/scan3d.h"
#include "scan3d_math.cuh"

#define S3D_PLANE_MASK_H 10   // internal: valid_map_horizontal when the stage API is used

namespace s3d {
// tensor maps of the last few capture stacks (a map depends on the stack's address and the tile size only)
struct TensorMapCache {
    static constexpr int SLOTS = 8;
    const uint8_t* stack[SLOTS] = {};
    int box[SLOTS] = {};
    alignas(64) CUtensorMap map[SLOTS];
    int next = 0;
};

// the voxel-grid merge's hash table (scan3d_voxel_kernels.cu)
constexpr uint32_t VOXEL_NO_SLOT = 0xffffffffu;   // no slot / no ordinal yet
// the integer sums of one voxel (zero-initialised); first_inv = ~(index of the first point within the current add)
struct VoxelSlot {
    unsigned long long q[3];   // positions inside the voxel, Q steps
    unsigned long long m[3];   // normals, Q steps, two's complement
    unsigned long long c[3];   // colours
    uint32_t n, first_inv;
};
struct VoxelState {
    unsigned long long dropped;
    uint32_t occupied;         // slots taken = distinct voxels inserted
    uint32_t overflow;         // an ordinal >= max_voxels was assigned
    uint32_t total[2];         // voxels with an ordinal, after an even / odd number of adds (chunks)
    uint32_t chunk_new;        // new voxels of the current add (chunk)
    uint32_t pad;
};
struct VoxelTable {
    unsigned long long* keys;  // [cap], s3v::EMPTY_KEY = free
    VoxelSlot* acc;            // [cap]
    uint32_t* ordinal;         // [cap], VOXEL_NO_SLOT until assigned
    uint32_t* ord2slot;        // [max_voxels]
    VoxelState* state;
    uint32_t cap, max_voxels;
    double S;                  // (double)voxel_size
};

// the alignment's cell index of the model (scan3d_align_kernels.cu)
struct AlignIndex {
    unsigned long long* keys;  // [cap], s3v::EMPTY_KEY = free; key = s3v::pack_key of the cell
    uint2* cells;              // [cap] (points in the cell, end of its range in entries)
    uint32_t* model_slot;      // [max_voxels] cell slot of each voxel, VOXEL_NO_SLOT = not in the model
    float4* entries;           // [2 max_voxels] per model point: (x, y, z, ordinal bits), (nx, ny, nz, 0)
    uint32_t* cursor;          // [1]
    uint32_t cap;
};
// the device state of one alignment run
struct AlignState {
    double T[12];              // current estimate [R | t], row-major
    double rms_first, rms_last;
    long long pairs_first, pairs_last;
    int iterations, status, done, rounds;   // updates applied, scan3d_align_result.status, run ended, solves run
    int overflow;              // the voxel accumulator overflowed (read when the index is built)
    uint32_t n_src;            // the ctx route's point count (read when the index is built)
};
struct AlignRun {
    double T0[12];             // T_init
    double S;                  // cell edge
    double r2;                 // max_distance^2
    double stop_rotation, stop_translation;
    int max_iterations;
};
}  // namespace s3d

struct scan3d_ctx {
    scan3d_config cfg{};
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    std::string err;
    int64_t launches = 0;

    // calibration
    bool has_calib = false;
    bool fast_div_ok = false;      // see scan3d_math.cuh div_const
    scan3d_calib hcal{};
    s3d::DeviceCalib dcal{};
    double2* cam_lut = nullptr;    // [H][W] (u',v') of the local rows, only if the camera is distorted
    double2* proj_lut = nullptr;   // [PH][PW], only if the projector is distorted
    double* atan_tab = nullptr;    // hi[33] then lo[33]
    float* pts_ext = nullptr;      // scan3d_set_points_buffer: caller-owned (possibly peer) destination of the points
    uint8_t* pattern_profiles = nullptr;   // scan3d_generate_patterns: 1-D profiles of both directions' patterns
    bool have_profiles[2] = {false, false};
    uint8_t* roi_eff = nullptr;    // SCAN3D_FLAG_MODULATION_MASK: ROI && modulation criterion of the current direction
    uint8_t* roi_eff_h = nullptr;  // ... single-pass entry: the horizontal direction's plane (roi_eff = the vertical one's)
    uint8_t* roi_strict = nullptr; // SCAN3D_FLAG_STRICT_REFERENCE: (ROI == 1) && N in {3, 4}, whole frame
    double* nstep_w = nullptr;     // sin[64] then cos[64] (generic-N extension)
    short2* undist_xy[2] = {nullptr, nullptr};     // cv::undistort's fixed-point map of the camera [0] / projector [1]
    uint16_t* undist_frac[2] = {nullptr, nullptr}; // (scan3d_undistort_frames; built on first use per calibration)

    // planes (row-major [H][W])
    float* wrapped[2] = {nullptr, nullptr};
    float* unwrapped[2] = {nullptr, nullptr};
    int16_t* code[2] = {nullptr, nullptr};
    uint8_t* mask[2] = {nullptr, nullptr};
    uint8_t* valid = nullptr;
    int2* cpmap = nullptr;
    double* xyz = nullptr;         // lazily allocated by scan3d_triangulate

    // compacted points
    float* pts = nullptr;          // [H*W][3]
    uint32_t* pix = nullptr;       // [H*W]   (only with SCAN3D_FLAG_POINT_PIXELS / stage API)
    uint8_t* rgb = nullptr;        // [H*W][3] (only when a texture is set)
    uint8_t* texture = nullptr;    // [H][W][3] BGR
    uint32_t* d_count = nullptr;   // [1]
    uint32_t* block_counts = nullptr;  // stage-API compaction scratch
    unsigned long long* tile_state = nullptr;  // fused kernel decoupled look-back
    uint8_t* tile_flags = nullptr;             // fused kernel work list (see k_tile_flags)
    int* tile_list = nullptr;
    unsigned long long* trace = nullptr;       // SCAN3D_TRACE=1: per-CTA pipeline timeline
    uint32_t epoch = 0;
    s3d::TensorMapCache tmaps;

    // staging for the host-buffer entries
    uint8_t* d_stack = nullptr;
    uint8_t* d_roi = nullptr;
    uint8_t* d_undist = nullptr;   // scan3d_reconstruct_raw: the undistorted stack

    // scan3d_build_mesh (allocated on the first build)
    int32_t* mesh_idx = nullptr;          // [H*W] point index of each pixel, -1 = invalid
    uint32_t* mesh_counts = nullptr;      // face counts / offsets per block of POINT_BLOCK pixels
    uint32_t* mesh_totals = nullptr;      // [2] points, faces
    int32_t* mesh_faces = nullptr;        // [2(W-1)(H-1)][3]
    float* mesh_normals = nullptr;        // [H*W][3]

    // scan3d_voxel_begin: the merge accumulator (independent of the points; reallocated when a begin asks for more)
    s3d::VoxelTable vox{};
    bool vox_begun = false;        // a begin has run
    bool vox_fresh = false;        // the outputs are those of the adds since begin (a finish ran after the last add)
    uint64_t vox_bound = 0;        // upper bound of the points added since begin (W*H per ctx add, n per dev add)
    uint32_t vox_chunks = 0;       // adds (chunks of <= W*H points) since begin
    uint32_t vox_alloc_cap = 0, vox_alloc_max = 0;   // what the buffers hold
    uint32_t* vox_point_slot = nullptr;   // [H*W] per-point scratch of an add
    uint8_t* vox_flags = nullptr;         // [H*W]
    float* vox_xyz = nullptr;             // [max_voxels][3] outputs of scan3d_voxel_finish
    float* vox_nrm = nullptr;             // [max_voxels][3]
    uint8_t* vox_rgb = nullptr;           // [max_voxels][3]
    uint32_t* vox_cnt = nullptr;          // [max_voxels]

    // scan3d_align_to_voxels (allocated by the first align, grown with max_voxels and the sample count)
    s3d::AlignIndex aln{};
    uint32_t aln_alloc_max = 0;           // max_voxels the index buffers hold
    uint32_t aln_alloc_blocks = 0;        // blocks of match partials the partial buffer holds
    double* aln_partials = nullptr;       // [ALIGN_NSUM + 1][blocks]
    s3d::AlignState* aln_state = nullptr;

    int cta_limit = 0;             // scan3d_set_cta_limit

    // scan3d_set_registration
    bool reg_on = false;
    float reg_R[16] = {}, reg_t[3] = {};

    // stage bookkeeping
    bool have_wrapped[2] = {false, false};
    bool have_unwrapped[2] = {false, false};
    bool have_cpmap = false, have_valid = false, have_xyz = false, have_points = false;
    bool have_mesh = false;        // built from the current points; every entry that rewrites or drops them clears it
    bool in_reconstruct = false;   // stage entries called from scan3d_reconstruct_dev's stage chain
};

namespace s3d {

struct Shape {
    int W, H;         // local frame
    int row0, H_total;
    int PW, PH;
};

inline Shape shape_of(const scan3d_config& c)
{
    Shape s;
    s.W = c.W; s.H = c.H; s.row0 = c.row0;
    s.H_total = c.H_total > 0 ? c.H_total : c.H;
    s.PW = c.PW; s.PH = c.PH;
    return s;
}

// ---- stage-wise kernels (any W, H) ----
cudaError_t launch_mask(const Shape& s, const uint8_t* roi_full, uint8_t* mask, cudaStream_t st);
cudaError_t launch_expand_patterns(const uint8_t* profiles, int profile_len, int n_patterns, uint8_t* out, int PW, int PH,
                                   int dir, cudaStream_t st);
cudaError_t launch_strict_roi(const uint8_t* roi, uint8_t* roi_eff, size_t n, int N, cudaStream_t st);
cudaError_t launch_modulation_roi(const Shape& s, const uint8_t* fringe, const uint8_t* roi, uint8_t* roi_eff, cudaStream_t st);
cudaError_t launch_wrapped(const Shape& s, int N, const uint8_t* fringe, const uint8_t* roi_full,
                           float* wrapped, const double* atan_tab, const double* nstep_w,
                           bool libdevice, cudaStream_t st);
cudaError_t launch_unwrap(const Shape& s, int dir, int M, const uint8_t* gray, const uint8_t* inv,
                          float* wrapped, const uint8_t* mask, int16_t* code, float* unwrapped,
                          cudaStream_t st);
cudaError_t launch_cpmap(const Shape& s, int fw_v, int fw_h, const float* unw_v, const float* unw_h,
                         const uint8_t* mask_v, const uint8_t* mask_h, int2* cpmap, uint8_t* valid,
                         cudaStream_t st);
cudaError_t launch_triangulate(const Shape& s, const DeviceCalib& cal, const double2* cam_lut,
                               const double2* proj_lut, const int2* cpmap, const uint8_t* valid,
                               double* xyz, cudaStream_t st);
cudaError_t launch_undistort_lut(const double* K9_k5_dev_unused, const DeviceCalib& cal, bool projector,
                                 int W, int H, int row0, double2* lut, cudaStream_t st);
// Raster-order point offsets of the valid plane, 2 launches (k_count, k_scan): block_counts[b] = number of valid
// pixels before block b of POINT_BLOCK pixels, *total = all of them.
constexpr int POINT_BLOCK = 1024;
cudaError_t launch_point_offsets(const uint8_t* valid, size_t plane, uint32_t* block_counts, uint32_t* total,
                                 cudaStream_t st);
// exclusive scan of counts[n] in place by one CTA (k_scan), *total = the sum; 1 launch
cudaError_t launch_block_scan(uint32_t* counts, int n, uint32_t* total, cudaStream_t st);
// 3 launches: count, scan, scatter.  pix / rgb / texture may be null.
cudaError_t launch_compact(const Shape& s, const double* xyz, const uint8_t* valid,
                           const uint8_t* texture, uint32_t* block_counts, float* pts, uint32_t* pix,
                           uint8_t* rgb, uint32_t* d_count, cudaStream_t st, int* n_launches);

// ---- fused single-pass kernel (W % 16 == 0, N in {3,4,5,8}) ----
struct FusedArgs {
    const uint8_t* stack;   // [NF][H][W]
    const uint8_t* roi;     // [H_total][W]
    const uint8_t* roi2;    // modulation criterion: the horizontal direction's effective ROI (roi = the vertical one's)
    const uint8_t* roi_list;   // ... and the caller's ROI, a superset of both: the work list is built from it
    float* unw_v; float* unw_h;
    int16_t* code_v; int16_t* code_h;
    uint8_t* valid;         // final valid (dirs==2) or mask (dirs==1)
    int2* cpmap;
    float* pts; uint32_t* pix; uint8_t* rgb; const uint8_t* texture;
    uint32_t* d_count;
    unsigned long long* tile_state;
    uint8_t* tile_flags;          // [n_tiles] tile holds at least one ROI pixel
    int* tile_list;               // [n_tiles] ids of those tiles, raster order
    int* n_list;                  // [1]; n_list[n_tiles + 8] is the counter the CTAs draw work-list positions from
    int reg_on;                   // fold register_point_clouds' transform into the point store (scan3d_set_registration)
    float reg_R[16], reg_t[3];
    int ctas_per_sm;              // 0 = all the kernel can have; else the launch takes at most this many CTA slots per SM
    TensorMapCache* tmap_cache;   // host pointer (the launcher's cache of tensor maps; unused on the device)
    unsigned long long* trace;    // optional timeline buffer (SCAN3D_TRACE), else null
    const double2* cam_lut; const double2* proj_lut;
    const double* atan_tab;
    uint32_t epoch;
    int W, H, row0, H_total, PW, PH;
    int N, M_v, M_h, fw_v, fw_h;
    double fw_v_d, fw_h_d;        // the fringe widths as doubles (5/compute_correspondance.cpp:648: fw * (Phi / 2Pi) in double)
    int n_tiles;
};
int fused_num_tiles(const scan3d_config& c);

// the single-pass kernel (scan3d_fused_kernel7.cu)
bool fused7_supported(const scan3d_config& c);
bool fused7_folds_registration(const scan3d_config& c);
cudaError_t launch_fused7(const scan3d_config& c, const FusedArgs& a, const DeviceCalib& cal,
                          int sm_count, cudaStream_t st);

// ---- either side of the path (scan3d_aux_kernels.cu) ----
cudaError_t launch_undistort_map(const double K[9], const double d[5], int W, int H, short2* map_xy, uint16_t* map_frac,
                                 cudaStream_t st);
cudaError_t launch_remap_frames(const uint8_t* src, uint8_t* dst, const short2* map_xy, const uint16_t* map_frac, int W,
                                int H, int n_frames, int sm_count, cudaStream_t st);
cudaError_t launch_roi_fill(const uint8_t* outline, int W, int H, uint8_t* roi, uint8_t* filled, cudaStream_t st);
cudaError_t launch_register_points(const float* src, float* dst, long long n, const float R[16], float tx, float ty,
                                   float tz, int sm_count, cudaStream_t st);

// ---- camera-grid mesh (scan3d_mesh_kernels.cu) ----
// MESH_LAUNCHES launches: point offsets (k_count, k_scan), pixel -> point index plane, face counts per block, their
// scan, faces + normals.  idx [W*H], block_counts [cdiv(W*H, POINT_BLOCK)], face_counts [same], totals [2]
// (points, faces); faces [2(W-1)(H-1)][3], normals [W*H][3].
constexpr int MESH_LAUNCHES = 6;
cudaError_t launch_mesh(const uint8_t* valid, const float* pts, int W, int H, float max_edge, int32_t* idx,
                        uint32_t* block_counts, uint32_t* face_counts, uint32_t* totals, int32_t* faces, float* normals,
                        cudaStream_t st);

// ---- voxel-grid merge (scan3d_voxel_kernels.cu; common/scan3d_voxel_math.h has the arithmetic) ----
// VOXEL_ADD_LAUNCHES launches for `plane` points (the ctx add reads the point count from n_dev, <= plane): insert,
// flag, k_count + k_scan over the flags, assign.  point_slot and flags [plane], block_counts [cdiv(plane,
// POINT_BLOCK)]; par = number of adds (chunks) since begin, mod 2.  nrm / rgb may be null (zeros).
constexpr int VOXEL_ADD_LAUNCHES = 5;
cudaError_t launch_voxel_add(const VoxelTable& t, const float* xyz, const float* nrm, const uint8_t* rgb,
                             const uint32_t* n_dev, uint32_t plane, uint32_t* point_slot, uint8_t* flags,
                             uint32_t* block_counts, int par, cudaStream_t st);
// slots of the table for max_voxels: at most half of them are ever taken (scan3d_voxel_kernels.cu)
uint32_t voxel_table_capacity(uint32_t max_voxels, int sm_count);
// 1 launch: the merged voxels in first-point order into xyz / nrm [max_voxels][3], rgb [max_voxels][3], cnt
cudaError_t launch_voxel_finish(const VoxelTable& t, int par, float* xyz, float* nrm, uint8_t* rgb, uint32_t* cnt,
                                int sm_count, cudaStream_t st);

// ---- scan-to-model alignment (scan3d_align_kernels.cu; common/scan3d_align_math.h has the arithmetic) ----
// ALIGN_INDEX_LAUNCHES launches: cell keys and counts (which also initialises *state from run, the voxel overflow
// flag and, when n_dev is set, the source count), cell ranges, scatter of the model points.  The model is the first
// min(total, max_voxels) voxel outputs of t (total = t.state->total[par]); xyz / nrm [max_voxels][3].  The index holds
// ALIGN_CELLS_PER_VOXEL * max_voxels slots (at most half of them taken) and must be reset before (keys 0xff, cells and
// cursor 0).
constexpr int ALIGN_INDEX_LAUNCHES = 3;
constexpr uint32_t ALIGN_CELLS_PER_VOXEL = 2;
cudaError_t launch_align_index(const AlignIndex& ix, const VoxelTable& t, int par, const float* xyz, const float* nrm,
                               double S, AlignState* state, const AlignRun& run, const uint32_t* n_dev, int sm_count,
                               cudaStream_t st);
// One match + one solve launch per iteration.  The source is xyz[i * stride] for i * stride < n, n = min(*n_dev, n_max)
// when n_dev is set, else n_max; the grid depends on n_max and stride only (align_match_blocks).  partials
// [ALIGN_NSUM + 1][blocks].
constexpr int ALIGN_NSUM = 28;
uint32_t align_match_blocks(long long n_max, int stride);
cudaError_t launch_align_iteration(const AlignIndex& ix, AlignState* state, const AlignRun& run, const float* xyz,
                                   const uint32_t* n_dev, long long n_max, int stride, double* partials, cudaStream_t st);

// ---- debug / self-test ----
cudaError_t launch_debug_atan2(const double* y, const double* x, float* out, int n, int mode,
                               const double* atan_tab, cudaStream_t st);

cudaError_t launch_debug_divcheck(unsigned long long* bad, cudaStream_t st);


}  // namespace s3d
