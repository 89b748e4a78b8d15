// scan3d_internal.h -- context layout and kernel launcher declarations (not part of the ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/scan3d.h"
#include "scan3d_device_buffer.h"
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

// the surface extraction's lattice table (scan3d_surface_kernels.cu), one slot per distinct lattice point
struct SurfaceState {
    unsigned long long undefined;  // lattice points without a model point within max_distance
    uint32_t occupied;             // slots taken = distinct lattice points
    uint32_t overflow;             // an insert found no free slot, or a vertex ordinal reached max_points
    uint32_t vertices, faces;
};
struct SurfaceTable {
    unsigned long long* keys;      // [cap] s3v::pack_key of the lattice point, s3v::EMPTY_KEY = free
    unsigned long long* owner;     // [cap] min(27 o + k) of a candidate cell, ~0 = not a candidate
    double* f;                     // [cap] corner value
    uint32_t* nearest;             // [cap] ordinal of the nearest model point, VOXEL_NO_SLOT = f undefined
    uint32_t* vert;                // [cap] VOXEL_NO_SLOT = not an active cell, else its vertex ordinal
    SurfaceState* state;
    uint32_t cap, max_points;
    double S;                      // (double)voxel_size
};

// the connected components of a triangle mesh (scan3d_components_kernels.cu)
struct ComponentsState {
    unsigned long long threshold;  // K of the keep rule: component c is kept when eligible and its key is >= K
    uint32_t components;           // of the mesh
    uint32_t kept, largest;        // components kept; the most faces of one component
    uint32_t vertices, faces;      // kept
    uint32_t bad;                  // a face index outside [0, vertices)
    uint32_t pad;
};

// the surface simplification (scan3d_decimate_kernels.cu); the clusters are a second VoxelTable
struct DecimateState {
    uint32_t collapsed;            // faces with two corners in one cluster
    uint32_t fallbacks;            // clusters placed at their mean after a failed solve
    uint32_t faces;                // kept faces
    uint32_t zero;                 // stays 0: the vertex count of an empty surface's voxel add
};
struct DecimateBuffers {
    uint32_t* point_slot;          // [vertices] cluster slot of each vertex
    uint8_t* vert_flags;           // [vertices]
    uint32_t* vert_counts;         // [cdiv(vertices, POINT_BLOCK) + 1]
    unsigned long long* quad;      // [vertices][10] quadric sums per cluster ordinal (int64 two's complement), zeroed
    int32_t* ctri;                 // [faces][3] cluster ordinals of the corners
    uint32_t* table;               // [table_cap] face indices, VOXEL_NO_SLOT = free
    uint32_t table_cap;
    uint32_t* slot_of;             // [faces] table slot of each face, VOXEL_NO_SLOT = collapsed
    uint8_t* keep;                 // [faces]
    uint32_t* face_counts;         // [cdiv(faces, POINT_BLOCK) + 1]
    DecimateState* state;          // zeroed
};

// the surface smoothing (scan3d_smooth_kernels.cu); the undirected edges are a hash of (min << 32 | max) keys
struct SmoothState {
    unsigned long long max_move;   // bits of the largest displacement (a non-negative double, so the bits order it)
    uint32_t exp_field;            // the largest biased float exponent field of the coordinates
    uint32_t bad;                  // a coordinate not finite or a face index outside [0, vertices): SCAN3D_ERR_ARG
    uint32_t overflow;             // a free vertex over a limit of common/scan3d_smooth_math.h: SCAN3D_ERR_CONFIG
    uint32_t held, isolated;       // vertices on an edge whose count is not 2; vertices without a neighbour
    uint32_t entries;              // neighbour row entries (the sum of the degrees)
};
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
}  // namespace s3d

// Every device buffer the context owns is a DeviceBuffer: scan3d_destroy frees them all by deleting the context.
struct scan3d_ctx {
    template <class T>
    using Buf = s3d::DeviceBuffer<T>;

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
    Buf<double2> cam_lut;          // [H][W] (u',v') of the local rows, only if the camera is distorted
    Buf<double2> proj_lut;         // [PH][PW], only if the projector is distorted
    Buf<double> atan_tab;          // hi[33] then lo[33]
    Buf<double> code_term;         // [2^max(M_v, M_h)] the unwrap term of every fringe order
    float* pts_ext = nullptr;      // scan3d_set_points_buffer: caller-owned (possibly peer) destination of the points
    Buf<uint8_t> pattern_profiles; // scan3d_generate_patterns: 1-D profiles of both directions' patterns
    bool have_profiles[2] = {false, false};
    Buf<uint8_t> roi_eff;          // SCAN3D_FLAG_MODULATION_MASK: ROI && modulation criterion of the current direction
    Buf<uint8_t> roi_eff_h;        // ... single-pass entry: the horizontal direction's plane (roi_eff = the vertical one's)
    Buf<uint8_t> roi_strict;       // SCAN3D_FLAG_STRICT_REFERENCE: (ROI == 1) && N in {3, 4}, whole frame
    Buf<double> nstep_w;           // sin[64] then cos[64] (generic-N extension)
    Buf<short2> undist_xy[2];      // cv::undistort's fixed-point map of the camera [0] / projector [1]
    Buf<uint16_t> undist_frac[2];  // (scan3d_undistort_frames; built on first use per calibration)

    // planes (row-major [H][W])
    Buf<float> wrapped[2];
    Buf<float> unwrapped[2];
    Buf<int16_t> code[2];
    Buf<uint8_t> mask[2];
    Buf<uint8_t> valid;
    Buf<int2> cpmap;
    Buf<double> xyz;               // lazily allocated by scan3d_triangulate

    // compacted points
    Buf<float> pts;                // [H*W][3]
    Buf<uint32_t> pix;             // [H*W]   (only with SCAN3D_FLAG_POINT_PIXELS / stage API)
    Buf<uint8_t> rgb;              // [H*W][3] (only when a texture is set)
    Buf<uint8_t> texture;          // [H][W][3] BGR
    Buf<uint32_t> d_count;         // [1]
    Buf<uint32_t> block_counts;    // stage-API compaction scratch
    Buf<unsigned long long> tile_state;  // fused kernel decoupled look-back
    Buf<uint8_t> tile_flags;             // fused kernel work list (see k_tile_flags)
    Buf<int> tile_list;
    Buf<unsigned long long> trace;       // SCAN3D_TRACE=1: per-CTA pipeline timeline
    uint32_t epoch = 0;
    s3d::TensorMapCache tmaps;

    // staging for the host-buffer entries
    Buf<uint8_t> d_stack;
    Buf<uint8_t> d_roi;
    Buf<uint8_t> d_undist;         // scan3d_reconstruct_raw: the undistorted stack

    // scan3d_build_mesh (allocated on the first build)
    Buf<int32_t> mesh_idx;         // [H*W] point index of each pixel, -1 = invalid
    Buf<uint32_t> mesh_counts;     // face counts / offsets per block of POINT_BLOCK pixels
    Buf<uint32_t> mesh_totals;     // [2] points, faces
    Buf<int32_t> mesh_faces;       // [2(W-1)(H-1)][3]
    Buf<float> mesh_normals;       // [H*W][3]

    // scan3d_voxel_begin: the merge accumulator (independent of the points; reallocated when a begin asks for more).
    // vox is the kernels' view of the vox_* buffers below.
    s3d::VoxelTable vox{};
    bool vox_begun = false;        // a begin has run
    bool vox_fresh = false;        // the outputs are those of the adds since begin (a finish ran after the last add)
    uint64_t vox_bound = 0;        // upper bound of the points added since begin (W*H per ctx add, n per dev add)
    uint32_t vox_chunks = 0;       // adds (chunks of <= W*H points) since begin
    Buf<unsigned long long> vox_keys;     // [cap] the table
    Buf<s3d::VoxelSlot> vox_acc;          // [cap]
    Buf<uint32_t> vox_ordinal;            // [cap]
    Buf<uint32_t> vox_ord2slot;           // [max_voxels]
    Buf<s3d::VoxelState> vox_state;
    Buf<uint32_t> vox_point_slot;         // [H*W] per-point scratch of an add
    Buf<uint8_t> vox_flags;               // [H*W]
    Buf<float> vox_xyz;                   // [max_voxels][3] outputs of scan3d_voxel_finish
    Buf<float> vox_nrm;                   // [max_voxels][3]
    Buf<uint8_t> vox_rgb;                 // [max_voxels][3]
    Buf<uint32_t> vox_cnt;                // [max_voxels]

    // scan3d_align_to_voxels (allocated by the first align, grown with max_voxels and the sample count); aln is the
    // kernels' view of the aln_* index buffers
    s3d::AlignIndex aln{};
    Buf<unsigned long long> aln_keys;     // [2 max_voxels]
    Buf<uint2> aln_cells;                 // [2 max_voxels]
    Buf<uint32_t> aln_model_slot;         // [max_voxels]
    Buf<float4> aln_entries;              // [2 max_voxels]
    Buf<uint32_t> aln_cursor;             // [1]
    Buf<double> aln_partials;             // [ALIGN_NSUM + 1][blocks]
    Buf<s3d::AlignState> aln_state;

    // scan3d_voxel_surface (allocated by the first extraction, grown on demand); srf is the kernels' view of the
    // lattice table srf_keys ... srf_state
    s3d::SurfaceTable srf{};
    bool srf_ready = false;               // the surface of the current voxel outputs is held
    Buf<unsigned long long> srf_keys;     // [cap]
    Buf<unsigned long long> srf_owner;    // [cap]
    Buf<double> srf_f;                    // [cap]
    Buf<uint32_t> srf_nearest;            // [cap]
    Buf<uint32_t> srf_vert;               // [cap]
    Buf<s3d::SurfaceState> srf_state;
    Buf<uint8_t> srf_flags;               // [27 max_voxels] (o, k) owns an active cell
    Buf<uint32_t> srf_flag_counts;        // [cdiv(27 max_voxels, POINT_BLOCK) + 1]
    Buf<uint32_t> srf_vert_slot;          // [max_points] lattice slot of each vertex
    Buf<uint32_t> srf_face_counts;        // [cdiv(max_points, SURFACE_VB) + 1] faces per block of vertices, then offsets
    int64_t srf_vertices = 0, srf_faces = 0;
    Buf<float> srf_xyz;                   // [vertices][3]
    Buf<float> srf_nrm;                   // [vertices][3]
    Buf<uint8_t> srf_rgb;                 // [vertices][3]
    Buf<int32_t> srf_tri;                 // [faces][3]

    // scan3d_voxel_surface_components / scan3d_mesh_components_dev (allocated on first use, grown on demand)
    bool cc_ready = false;                // the component table of the last scan3d_voxel_surface_components is held
    int64_t cc_components = 0;
    Buf<uint32_t> cc_parent;              // [vertices] union-find forest, then each vertex's root
    Buf<uint8_t> cc_flags;                // [vertices] root flags, then the vertices' keep flags
    Buf<uint32_t> cc_vert_counts;         // [cdiv(vertices, POINT_BLOCK) + 1] block offsets of the flags
    Buf<int32_t> cc_label;                // [vertices] component ids, then the kept vertices' new indices
    Buf<uint32_t> cc_comp_v;              // [vertices] per component: vertices, faces, kept flag
    Buf<uint32_t> cc_comp_f;
    Buf<uint8_t> cc_kept;
    Buf<uint8_t> cc_keep_f;               // [faces]
    Buf<uint32_t> cc_face_counts;         // [cdiv(faces, POINT_BLOCK) + 1]
    Buf<s3d::ComponentsState> cc_state;
    Buf<float> cc_xyz;                    // the second surface set, swapped with srf_* after a compaction
    Buf<float> cc_nrm;
    Buf<uint8_t> cc_rgb;
    Buf<int32_t> cc_tri;

    // scan3d_voxel_surface_decimate (allocated on first use, grown on demand); dec is the kernels' view of the cluster
    // table dec_keys ... dec_state, never the merge's ctx->vox.  The emission writes the components' second set.
    bool srf_decimated = false;           // the held surface is a simplification (it is not simplified again)
    s3d::VoxelTable dec{};
    Buf<unsigned long long> dec_keys;     // [cap] the cluster table
    Buf<s3d::VoxelSlot> dec_acc;          // [cap]
    Buf<uint32_t> dec_ordinal;            // [cap]
    Buf<uint32_t> dec_ord2slot;           // [vertices]
    Buf<s3d::VoxelState> dec_vstate;
    Buf<uint32_t> dec_point_slot;         // [vertices]
    Buf<uint8_t> dec_vert_flags;          // [vertices]
    Buf<uint32_t> dec_vert_counts;        // [cdiv(vertices, POINT_BLOCK) + 1]
    Buf<unsigned long long> dec_quad;     // [vertices][10]
    Buf<int32_t> dec_ctri;                // [faces][3]
    Buf<uint32_t> dec_table;              // [2 faces]
    Buf<uint32_t> dec_slot_of;            // [faces]
    Buf<uint8_t> dec_keep;                // [faces]
    Buf<uint32_t> dec_face_counts;        // [cdiv(faces, POINT_BLOCK) + 1]
    Buf<s3d::DecimateState> dec_state;

    // scan3d_voxel_surface_smooth / scan3d_mesh_smooth_dev (allocated on first use, grown on demand).  The surface
    // route writes the components' second set's xyz and normals.
    bool srf_smoothed = false;            // the held surface is smoothed (scan3d_voxel_surface_decimate refuses it)
    Buf<unsigned long long> sm_keys;      // [6 faces] the edge table
    Buf<uint32_t> sm_sides;               // [6 faces]
    Buf<uint32_t> sm_rows;                // [6 faces]
    Buf<uint32_t> sm_degree;              // [vertices]
    Buf<uint8_t> sm_held;                 // [vertices]
    Buf<uint32_t> sm_block_counts;        // [cdiv(vertices, POINT_BLOCK) + 1]
    Buf<uint32_t> sm_cursor;              // [vertices]
    Buf<long long> sm_q[2];               // [vertices][3]
    Buf<unsigned long long> sm_nsum;      // [vertices][3]
    Buf<s3d::SmoothState> sm_state;

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

// the C entries' error returns: a failed CUDA call names itself in ctx->err
#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                \
            return SCAN3D_ERR_CUDA;                                                       \
        }                                                                                 \
    } while (0)

namespace s3d {

inline int fail(scan3d_ctx* ctx, int code, const char* msg)
{
    if (ctx) ctx->err = msg;
    return code;
}

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
// pixels before block b of POINT_BLOCK pixels, *total = all of them.  An empty plane takes one block (total 0).
constexpr int POINT_BLOCK = 1024;
cudaError_t launch_point_offsets(const uint8_t* valid, size_t plane, uint32_t* block_counts, uint32_t* total,
                                 cudaStream_t st);
// exclusive scan of counts[n] in place by one CTA (k_scan), *total = the sum; 1 launch
cudaError_t launch_block_scan(uint32_t* counts, int n, uint32_t* total, cudaStream_t st);

// rank of this thread's flag among the flags of its POINT_BLOCK block (every thread of the block calls it); with the
// block offsets of launch_point_offsets this places a flagged item at its compacted position
__device__ __forceinline__ uint32_t block_rank(bool flag)
{
    __shared__ uint32_t wsum[POINT_BLOCK / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) wsum[w] = __popc(b);
    __syncthreads();
    uint32_t before = 0;
    for (int k = 0; k < w; k++) before += wsum[k];
    return before + __popc(b & ((1u << lane) - 1));
}
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
    const double* code_term;      // [2^max(M_v, M_h)] code*2.0*Pi per fringe order (fill_code_term_table)
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

// ---- surface extraction (scan3d_surface_kernels.cu; common/scan3d_surface_math.h has the arithmetic) ----
// launch_surface_counts: SURFACE_COUNT_LAUNCHES launches after launch_align_index built the model's index (cell edge
// s3l::cell_edge(max_distance)): candidate cells (27 per model voxel, with their order key), their other 7 corners,
// the corner values, the (o, k) flags of active cells, k_count + k_scan over them (the vertex ordinals), vertex
// assignment with the faces per block of SURFACE_VB vertices, and the scan of those.  The table must be reset before
// (keys 0xff, owner 0xff, vert 0xff, state 0).  flags [27 max_voxels], flag_counts [cdiv(27 max_voxels, POINT_BLOCK)],
// vert_slot [max_points], face_counts [cdiv(max_points, SURFACE_VB)].
// launch_surface_emit: 1 launch, the vertices (xyz, normals, rgb) and faces once the counts are known.
constexpr int SURFACE_COUNT_LAUNCHES = 8;
constexpr int SURFACE_VB = 256;
cudaError_t launch_surface_counts(const SurfaceTable& s, const AlignIndex& ix, const VoxelTable& t, int par,
                                  const float* vox_nrm, float max_distance, uint8_t* flags, uint32_t* flag_counts,
                                  uint32_t* vert_slot, uint32_t* face_counts, cudaStream_t st);
cudaError_t launch_surface_emit(const SurfaceTable& s, const uint8_t* vox_rgb, const uint32_t* vert_slot,
                                const uint32_t* face_counts, uint32_t vertices, float* xyz, float* nrm, uint8_t* rgb,
                                int32_t* faces, cudaStream_t st);
// slots of the lattice table for max_points: at most half of them are ever taken
uint32_t surface_table_capacity(uint32_t max_points, int sm_count);

// ---- connected components of a triangle mesh (scan3d_components_kernels.cu) ----
// launch_cc_labels: COMPONENT_LABEL_LAUNCHES launches for n vertices and n_faces faces [n_faces][3]: parent = v,
// union per face, find per vertex with the root flags, k_count + k_scan over them (state->components), the roots' ids,
// every vertex's id into label [n].  state must be zeroed before; parent and flags [n], block_counts [cdiv(n,
// POINT_BLOCK) + 1].  Any n below 2^31 and n_faces below 2^32, 0 included.
// launch_cc_select: COMPONENT_SELECT_LAUNCHES launches after it: vertices and faces per component (comp_v, comp_f [n],
// zeroed before), the selection (state->threshold, kept, largest), the keep flags (keep_v [n], keep_f [n_faces], kept
// [components]), k_count + k_scan over each of keep_v (state->vertices) and keep_f (state->faces).
// launch_cc_emit: COMPONENT_EMIT_LAUNCHES launches: the kept vertices into xyz2 / nrm2 / rgb2 (their new indices into
// new_index [n]), then the kept faces, remapped, into faces2.
constexpr int COMPONENT_LABEL_LAUNCHES = 7;
constexpr int COMPONENT_SELECT_LAUNCHES = 7;
constexpr int COMPONENT_EMIT_LAUNCHES = 2;
cudaError_t launch_cc_labels(const int32_t* faces, uint32_t n_faces, uint32_t n, uint32_t* parent, uint8_t* flags,
                             uint32_t* block_counts, int32_t* label, ComponentsState* state, cudaStream_t st);
cudaError_t launch_cc_select(const int32_t* faces, uint32_t n_faces, uint32_t n, const int32_t* label,
                             unsigned long long min_faces, unsigned long long max_components, uint32_t* comp_v,
                             uint32_t* comp_f, uint8_t* kept, uint8_t* keep_v, uint8_t* keep_f, uint32_t* vert_counts,
                             uint32_t* face_counts, ComponentsState* state, cudaStream_t st);
cudaError_t launch_cc_emit(const uint8_t* keep_v, const uint32_t* vert_counts, uint32_t n, const float* xyz,
                           const float* nrm, const uint8_t* rgb, const uint8_t* keep_f, const uint32_t* face_counts,
                           uint32_t n_faces, const int32_t* faces, int32_t* new_index, float* xyz2, float* nrm2,
                           uint8_t* rgb2, int32_t* faces2, cudaStream_t st);

// ---- surface simplification (scan3d_decimate_kernels.cu; common/scan3d_decimate_math.h has the arithmetic) ----
// DECIMATE_LAUNCHES launches for a surface of n_vertices (xyz, nrm, rgb) and n_faces (tri): launch_voxel_add over the
// vertices into t (the clusters, edge t.S = H; t must be reset as scan3d_voxel_begin resets the merge's table, with
// max_voxels >= max(n_vertices, 1)), the face quadrics with the cluster triples, the duplicate-face table, the keep
// flags, k_count + k_scan over them (b.state->faces), then the vertices of the clusters into xyz2 / nrm2 / rgb2 [n_vertices]
// and the kept faces into faces2 [n_faces].  b.quad, b.state zeroed and b.table set to 0xff before.
constexpr int DECIMATE_LAUNCHES = VOXEL_ADD_LAUNCHES + 7;
cudaError_t launch_decimate(const VoxelTable& t, const DecimateBuffers& b, const float* xyz, const float* nrm,
                            const uint8_t* rgb, const int32_t* tri, uint32_t n_vertices, uint32_t n_faces, double H,
                            float* xyz2, float* nrm2, uint8_t* rgb2, int32_t* faces2, int sm_count, cudaStream_t st);

// ---- surface smoothing (scan3d_smooth_kernels.cu; common/scan3d_smooth_math.h has the arithmetic) ----
// SMOOTH_BUILD_LAUNCHES + passes + SMOOTH_END_LAUNCHES launches for n vertices (xyz, nrm may be null) and nf faces
// [nf][3]: the exponent max and the finiteness check over the vertices, the sides into the edge table, the degrees and
// held flags per edge, the degree sums per POINT_BLOCK vertices, their k_scan, the row starts with the fixed-point
// positions, the neighbour rows; then one gather per pass (k = lambda, or lambda and mu alternating when mu != 0);
// then the face normals and the write of xyz_out / nrm_out (nrm_out may be null), which writes nothing when the state
// holds an error.  xyz_out may be xyz and nrm_out nrm.  b.keys 0xff; b.sides, b.degree, b.held, b.nsum, b.state zeroed
// before; b.cap >= 2 * 3 nf.
constexpr int SMOOTH_BUILD_LAUNCHES = 7;
constexpr int SMOOTH_END_LAUNCHES = 2;
cudaError_t launch_smooth(const SmoothBuffers& b, const float* xyz, const float* nrm, const int32_t* faces, uint32_t n,
                          uint32_t nf, int passes, double lambda, double mu, float* xyz_out, float* nrm_out,
                          cudaStream_t st);

// ---- debug / self-test ----
cudaError_t launch_debug_atan2(const double* y, const double* x, float* out, int n, int mode,
                               const double* atan_tab, cudaStream_t st);

cudaError_t launch_debug_divcheck(unsigned long long* bad, cudaStream_t st);


}  // namespace s3d
