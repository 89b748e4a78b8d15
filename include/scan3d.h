/*
 * scan3d.h -- C ABI of the B200-native reconstruction hot path of pranavkantgaur/3dscan.
 *
 * This is the drop-in boundary: one entry point per stage function that the reference's
 * main() calls between capture and PLY (PROJECT_GLOBAL/intermodule_dependencies.h:10-25,
 * called at M_tech_project_console/m_tech_project_console.cpp:372-401), plus one fused entry
 * that runs the whole path in a single pass over the captured pattern stack.
 *
 *   reference (C++ linkage, globals)                this library (extern "C", explicit ctx)
 *   ---------------------------------------------   ------------------------------------------
 *   void compute_wrapped_phase(int pattern_type)    scan3d_compute_wrapped_phase[_dev]
 *        3/wrapped_phase.cpp:402
 *   void unwrap_phase(int pattern_type)             scan3d_unwrap_phase[_dev]
 *        4/phase_unwrap.cpp:367
 *   void compute_c_p_map()                          scan3d_compute_c_p_map
 *        5/compute_correspondance.cpp:630
 *   void triangulate()                              scan3d_triangulate
 *        7/triangulation.cpp:1444
 *   void save_point_cloud(unsigned)                 scan3d_compact_points + scan3d_write_ply
 *        8/save_point_cloud.cpp:26
 *   load_matrices() / read_parameters()             scan3d_set_calibration
 *        6/system_calibration.cpp:1526, 7/triangulation.cpp:149
 *   (all five calls above, one scan)                scan3d_reconstruct[_dev]
 *   either side of the path:
 *   cvUndistort2 in the capture loop                scan3d_undistort_frames[_dev]
 *        2/project_pattern.cpp:220,234,372-427
 *   image_scissor()'s region fill                   scan3d_roi_fill[_dev]
 *        M_tech_project_console/m_tech_project_console.cpp:186-229
 *   void register_point_clouds(...)                 scan3d_register_points[_dev]
 *        9/register_point_clouds.cpp:22
 *   void generate_pattern()                         scan3d_generate_patterns[_dev]
 *        1/pattern_generator.cpp:513
 *
 * Data contract
 *   - Every image-sized plane is ROW-MAJOR [H][W] (the reference's globals are [col][row];
 *     INTEGRATION.md shows the transposing shim).  pattern_type / dir: 0 = vertical stripes
 *     (encodes projector x), 1 = horizontal (encodes projector y).
 *   - The reference passes data between stages through extern globals
 *     (PROJECT_GLOBAL/common_variables.h:12-62); here the ctx owns the same planes in HBM and
 *     the getters below copy them out.  The caller owns all host buffers.
 *   - Pointers named *_host are host memory, *_dev are device memory on the ctx's GPU.
 *   - All work is ordered on the ctx's stream; entries taking host buffers synchronise before
 *     they return, *_dev entries are asynchronous (use scan3d_sync).
 *   - Per-pixel failures are expressed only through the valid planes, as in the reference.
 *   - Return value: 0 on success, negative scan3d_status otherwise; scan3d_last_error() gives
 *     a message.  There is no CPU fallback: without a usable CUDA device every compute entry
 *     fails with SCAN3D_ERR_CUDA.
 */
#ifndef SCAN3D_H
#define SCAN3D_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCAN3D_VERSION 100

typedef struct scan3d_ctx scan3d_ctx;

typedef enum {
    SCAN3D_OK = 0,
    SCAN3D_ERR_CONFIG = -1,      /* bad sizes / unsupported N, M */
    SCAN3D_ERR_CUDA = -2,        /* CUDA runtime error (message has the detail) */
    SCAN3D_ERR_STATE = -3,       /* stage called out of order / calibration missing */
    SCAN3D_ERR_ARG = -4,         /* null pointer, bad enum */
    SCAN3D_ERR_IO = -5           /* file could not be written */
} scan3d_status;

/* Compile-time sizes and initialised globals of the reference
 * (PROJECT_GLOBAL/global_cv.h:49-53, common_variables.h:6-10,23-24) as a runtime struct. */
typedef struct {
    int32_t W, H;          /* camera frame held by this ctx (H = local rows when row-sharded) */
    int32_t PW, PH;        /* projector resolution */
    int32_t N;             /* number_of_patterns_fringe: 3,4,5 (reference) or 8 / 6..16 (extension) */
    int32_t M_v, M_h;      /* number_of_patterns_binary_{vertical,horizontal}: 1..15 */
    int32_t fw_v, fw_h;    /* fringe_width_pixels_{vertical,horizontal} */
    int32_t dirs;          /* 1 = vertical only (stages 3+4), 2 = both directions (full path) */
    int32_t row0;          /* row-sharding: global row of local row 0 (0 when not sharded) */
    int32_t H_total;       /* row-sharding: full frame height (0 or H when not sharded) */
    uint32_t flags;        /* SCAN3D_FLAG_* */
} scan3d_config;

#define SCAN3D_FLAG_NONE 0u
#define SCAN3D_FLAG_POINT_PIXELS 1u  /* also emit pix[count] = global row*W+col of every point */
/* Fused entry only: solve the per-pixel normal equations with fused multiply-adds and the
 * right-hand side reduced first (~90 instead of ~220 FP64 operations).  Same solution as the
 * reference's cvTranspose/cvMatMul/cvInvert chain (7/triangulation.cpp:1202-1206) up to rounding:
 * <= 1e-10 relative in double, i.e. the float points differ only in rare last-bit ties.  Without
 * this flag the operation order is the reference's and the points are bit-identical to it. */
#define SCAN3D_FLAG_FAST_TRIANGULATION 2u
/* check_I_mod_criteria's second, commented-out validity criterion (3/wrapped_phase.cpp:84-104):
 * a pixel of the selected region is kept only when its fringe modulation
 * sqrtf(3 (I0-I2)^2 + (2 I1-I0-I2)^2) / (float)(I0+I1+I2) exceeds 0.01 (per direction, from that
 * direction's three fringe images).  OFF by default: the reference's live path is ROI-only.
 * 3-step configurations without row sharding only; with the flag scan3d_reconstruct runs the
 * stage kernels in sequence instead of the single-pass kernel (the mask recurrence then needs
 * the modulation of pixels two rows up, which a linear tile does not hold). */
#define SCAN3D_FLAG_MODULATION_MASK 4u
/* check_I_mod_criteria exactly as committed (3/wrapped_phase.cpp:78-127): a pixel is selected only where the ROI
 * byte == 1, and only when N is 3 or 4 -- the reference's 5-step block (:117-127) is commented out, so its own
 * 5-step run ends with an all-zero valid map and an empty cloud.  OFF by default: by default every non-zero ROI
 * byte selects its pixel for every N (documented extension; image_scissor only writes 0 and 1). */
#define SCAN3D_FLAG_STRICT_REFERENCE 8u

/* The 8 matrices load_matrices() reads (6/system_calibration.cpp:1526-1554): intrinsics (3x3
 * row-major), distortion (k1,k2,p1,p2,k3), world->device rotation vectors and translations. */
typedef struct {
    double Kc[9], dc[5], Kp[9], dp[5];
    double rc[3], tc[3], rp[3], tp[3];
} scan3d_calib;

typedef enum {
    SCAN3D_PLANE_WRAPPED_V = 0,   /* f32  wrapped_phi_vertical   (stage entries only)        */
    SCAN3D_PLANE_WRAPPED_H = 1,   /* f32  wrapped_phi_horizontal (stage entries only)        */
    SCAN3D_PLANE_UNWRAPPED_V = 2, /* f32  unwrapped_phi_vertical                              */
    SCAN3D_PLANE_UNWRAPPED_H = 3, /* f32  unwrapped_phi_horizontal                            */
    SCAN3D_PLANE_CODE_V = 4,      /* i16  code_vertical (-1 = invalid)                        */
    SCAN3D_PLANE_CODE_H = 5,      /* i16  code_horizontal                                     */
    SCAN3D_PLANE_MASK = 6,        /* u8   valid_map_vertical == valid_map_horizontal          */
    SCAN3D_PLANE_VALID = 7,       /* u8   valid_map (merged, after the projector-bounds test) */
    SCAN3D_PLANE_CPMAP = 8,       /* i32[2] c_p_map[row*W+col] = (proj x, proj y)             */
    SCAN3D_PLANE_XYZ = 9,         /* f64[3] intersection_points (scan3d_triangulate only)     */
    SCAN3D_PLANE_COUNT_
} scan3d_plane;

/* ---- lifecycle ------------------------------------------------------------------------ */
int scan3d_version(void);
int scan3d_create(const scan3d_config *cfg, int device, scan3d_ctx **out);
void scan3d_destroy(scan3d_ctx *ctx);
const char *scan3d_last_error(const scan3d_ctx *ctx); /* ctx may be NULL: last create error */
/* Use an existing cudaStream_t (e.g. the caller's framework stream); NULL = ctx-owned stream. */
int scan3d_set_stream(scan3d_ctx *ctx, void *cuda_stream);
int scan3d_sync(scan3d_ctx *ctx);

/* load_matrices / read_parameters / compute_A / assign_3d_coordinates: uploads the calibration,
 * builds A = K[R|t] for both devices and the undistorted-pixel tables on the GPU (once per
 * calibration instead of once per triangulate() call, 7/triangulation.cpp:228-439,1061-1126). */
int scan3d_set_calibration(scan3d_ctx *ctx, const scan3d_calib *cal);
/* 3x4 row-major A matrices computed above (for diffing against the reference's A_cam/A_proj). */
int scan3d_get_projection_matrices(scan3d_ctx *ctx, double A_cam[12], double A_proj[12]);

/* Optional texture ("Point_cloud/texture.bmp", 8/save_point_cloud.cpp:59-66): BGR u8 [H][W][3].
 * NULL clears it (points then carry rgb = 0). */
int scan3d_set_texture(scan3d_ctx *ctx, const uint8_t *bgr_host);

/* ---- stage entries (mirror the reference's call sequence) ------------------------------ */
/* compute_wrapped_phase(pattern_type): fringe = [N][H][W] u8 captured phase-shift frames,
 * roi = selected_region as u8 [H_total][W] (non-zero = selected; row-sharded ctxs pass the FULL
 * frame's ROI).  Produces WRAPPED_{V,H} and MASK (ROI after the raster mask recurrence). */
int scan3d_compute_wrapped_phase(scan3d_ctx *ctx, int dir, const uint8_t *fringe_host,
                                 const uint8_t *roi_host);
int scan3d_compute_wrapped_phase_dev(scan3d_ctx *ctx, int dir, const uint8_t *fringe_dev,
                                     const uint8_t *roi_dev);
/* unwrap_phase(pattern_type): gray / inv = [M][H][W] u8 captured Gray-code frames and their
 * inverses.  Produces CODE_{V,H}, UNWRAPPED_{V,H}; adds Pi to WRAPPED_{V,H} in place. */
int scan3d_unwrap_phase(scan3d_ctx *ctx, int dir, const uint8_t *gray_host,
                        const uint8_t *inv_host);
int scan3d_unwrap_phase_dev(scan3d_ctx *ctx, int dir, const uint8_t *gray_dev,
                            const uint8_t *inv_dev);
/* compute_c_p_map(): produces CPMAP and VALID from UNWRAPPED_{V,H} and MASK. */
int scan3d_compute_c_p_map(scan3d_ctx *ctx);
/* triangulate(): produces XYZ (dense f64, allocated on first use) from CPMAP and VALID. */
int scan3d_triangulate(scan3d_ctx *ctx);
/* save_point_cloud()'s count + raster-order gather: compacts XYZ/VALID (+texture) into the
 * ctx's point buffers; *count_out receives the number of points. */
int scan3d_compact_points(scan3d_ctx *ctx, int64_t *count_out);

/* ---- fused entry: the whole path in one pass ------------------------------------------- */
/* stack = the captured pattern stack, planes [H][W] u8 in this order:
 *   fringe_v[N], gray_v[M_v], inv_v[M_v]   (and, when dirs == 2)   fringe_h[N], gray_h[M_h], inv_h[M_h]
 * Produces UNWRAPPED_*, CODE_*, VALID (MASK when dirs == 1), CPMAP and the compacted points. */
int64_t scan3d_stack_bytes(const scan3d_config *cfg);
int scan3d_reconstruct(scan3d_ctx *ctx, const uint8_t *stack_host, const uint8_t *roi_host,
                       int64_t *count_out);
int scan3d_reconstruct_dev(scan3d_ctx *ctx, const uint8_t *stack_dev, const uint8_t *roi_dev);

/* ---- results -------------------------------------------------------------------------- */
int64_t scan3d_plane_bytes(const scan3d_ctx *ctx, int plane);
int scan3d_get_plane(scan3d_ctx *ctx, int plane, void *dst_host);     /* synchronous D2H */
void *scan3d_device_plane(scan3d_ctx *ctx, int plane);                /* NULL if not allocated */
/* code plane widened to the reference's int (common_variables.h:12-13) */
int scan3d_get_code_i32(scan3d_ctx *ctx, int dir, int32_t *dst_host);
/* c_p_map widened to the reference's long int [W*H][2] (common_variables.h:15) */
int scan3d_get_cpmap_i64(scan3d_ctx *ctx, int64_t *dst_host);

int scan3d_point_count(scan3d_ctx *ctx, int64_t *count_out);          /* syncs the stream */
/* Raster-ordered points: xyz f32[count][3], pix u32[count] (global row*W+col), rgb u8[count][3].
 * Any destination may be NULL.  max_points bounds the copy. */
int scan3d_get_points(scan3d_ctx *ctx, float *xyz_host, uint32_t *pix_host, uint8_t *rgb_host,
                      int64_t max_points);
void *scan3d_device_points(scan3d_ctx *ctx);        /* f32[capacity][3] */
/* Let the reconstruction write its compacted points into a caller-provided device buffer of at
 * least capacity_points*12 bytes (capacity_points >= W*H) instead of the ctx-owned one; NULL
 * restores the ctx-owned buffer.  The pointer may be PEER memory (another GPU's allocation
 * mapped into this process, e.g. through CUDA IPC): the kernel's point stream then goes straight
 * over NVLink while the decode is still running -- how the row-sharded mode delivers every
 * rank's points to one GPU without a separate exchange (3dscan_b200/sharding.py, PeerPointSink).
 * No reference counterpart (the reference is single-process, 8/save_point_cloud.cpp:85-136). */
int scan3d_set_points_buffer(scan3d_ctx *ctx, void *points_dev, int64_t capacity_points);
/* Helpers for that mode (one process per GPU): allocate a device block on `device` and export
 * its CUDA IPC handle (64 bytes); map another process's block for kernels running on `device`
 * (cudaIpcOpenMemHandle with lazy peer access).  close/free undo them. */
int scan3d_peer_alloc(int device, int64_t bytes, void **dev_ptr, uint8_t handle_out[64]);
int scan3d_peer_free(int device, void *dev_ptr);
int scan3d_peer_open(int device, const uint8_t handle[64], void **dev_ptr);
int scan3d_peer_close(int device, void *dev_ptr);
void *scan3d_device_point_pixels(scan3d_ctx *ctx);  /* u32[capacity]    */
void *scan3d_device_point_count(scan3d_ctx *ctx);   /* u32[1] on device (for collectives) */

/* generate_pattern() (1/pattern_generator.cpp:513): the projector patterns of one direction, in the
 * order the capture stack uses -- fringe[N] (:291-397), Gray[M] (:56-197), inverse Gray[M]
 * (:490-507) -- as u8 images [N + 2M][PH][PW], written by the GPU (PW % 16 == 0).  dir 0 =
 * vertical stripes (value depends on the column), 1 = horizontal.  N = 3, 4, 5 follow the
 * reference's expressions (bit-identical to its Generated_patterns images); other N use 2*pi*k/N. */
int64_t scan3d_pattern_bytes(const scan3d_config *cfg, int dir);
int scan3d_generate_patterns_dev(scan3d_ctx *ctx, int dir, uint8_t *patterns_dev);
int scan3d_generate_patterns(scan3d_ctx *ctx, int dir, uint8_t *patterns_host);

/* save_point_cloud()'s pcl::io::savePLYFile equivalent: "x y z red green blue" vertices,
 * ASCII (binary = 0, PCL's default) or binary_little_endian. */
int scan3d_write_ply(scan3d_ctx *ctx, const char *path, int binary);
/* save_point_cloud()'s pcl::io::savePCDFileASCII equivalent (8/save_point_cloud.cpp:212): PCD v0.7,
 * "x y z rgb" per point, 8 significant digits, rgb packed into a float as PCL 1.6 does. */
int scan3d_write_pcd(scan3d_ctx *ctx, const char *path);

/* ---- camera-grid mesh of the points (no reference counterpart: its users meshed the cloud elsewhere) -------------
 * The point index of a valid pixel is its rank among the valid pixels in raster order, so the camera grid is the
 * mesh.  Cell (r, c) (0 <= r < H-1, 0 <= c < W-1) has corners a = (r,c), b = (r,c+1), d = (r+1,c), e = (r+1,c+1)
 * and two candidate triangles, T1 = (a, d, b) then T2 = (b, d, e).  A triangle is emitted when its three pixels are
 * valid and each edge's squared length ((dx*dx + dy*dy) + dz*dz, separately rounded float operations) is finite and
 * <= max_edge*max_edge.  Faces are int32 point indices, ordered by cell in raster order, T1 before T2; the winding is
 * counter-clockwise seen from the camera (the right-hand face normal points toward it, also after registration).
 * The normal of a point is the sum of the unnormalised face normals (v1 - v0) x (v2 - v0) of its up-to-six emitted
 * triangles, divided by its length (IEEE sqrt and division); (0,0,0) when that length is 0 or not finite, e.g. for
 * an isolated point.  The exact arithmetic is in 3dscan_b200/common/scan3d_mesh_math.h.
 *
 * scan3d_build_mesh: after scan3d_reconstruct[_dev] / scan3d_compact_points, from the VALID plane and the points
 * where they currently are (scan3d_set_points_buffer included); asynchronous on the ctx stream, always 6 kernel
 * launches.  max_edge > 0, +inf = no length limit.  Errors: SCAN3D_ERR_ARG for a bad max_edge (NaN, <= 0);
 * SCAN3D_ERR_STATE without points or with dirs == 1; SCAN3D_ERR_CONFIG for a row-sharded ctx (a shard's last cell row
 * needs the next shard's first row) or W*H >= 2^31.  The face buffer (2(W-1)(H-1) faces) and the normal buffer (W*H)
 * are ctx-owned, allocated by the first build.  Every entry that rewrites or drops the points (a reconstruct,
 * scan3d_compact_points, scan3d_set_points_buffer, scan3d_align_to_voxels with apply) makes the mesh stale: the getters
 * below then return SCAN3D_ERR_STATE (the device pointers NULL) until scan3d_build_mesh runs again. */
int scan3d_build_mesh(scan3d_ctx *ctx, float max_edge);
int scan3d_mesh_face_count(scan3d_ctx *ctx, int64_t *count_out);             /* syncs */
/* faces int32[n][3], normals f32[point_count][3]; either may be NULL; max_faces bounds the face copy */
int scan3d_get_mesh(scan3d_ctx *ctx, int32_t *faces_host, float *normals_host, int64_t max_faces);
void *scan3d_device_mesh_faces(scan3d_ctx *ctx);       /* NULL until a mesh is built */
void *scan3d_device_point_normals(scan3d_ctx *ctx);
/* vertices "x y z nx ny nz red green blue" (colours as scan3d_write_ply) + "element face" with
 * "property list uchar int vertex_indices"; ascii (%.9g, faces "3 i j k") or binary_little_endian */
int scan3d_write_mesh_ply(scan3d_ctx *ctx, const char *path, int binary);

/* ---- voxel-grid merge of registered views (the reference concatenated them: 9/register_point_clouds.cpp) ---------
 * One output point per occupied voxel of edge s = voxel_size, averaged over every point that fell into it, from every
 * add since scan3d_voxel_begin.  Per point and axis t = (double)x / (double)s, i = floor(t), q = the position inside
 * the voxel in 2^24 steps; a point is dropped (counted, contributes nothing) when a coordinate is not finite or some
 * i is outside [-2^20, 2^20).  A normal with a non-finite component counts as (0,0,0); otherwise each component is
 * clamped to [-1, 1] and rounded to 2^24 steps.  The sums per voxel are integers, so the outputs do not depend on the
 * hash function, the table layout, thread scheduling or how a cloud is split into adds:
 *   coordinate (float)(((double)i + (double)sum_q / (2^24 (double)n)) * (double)s)
 *   normal     the sum of the fixed-point normals divided by its length (double), (0,0,0) if the sum is 0, so views
 *              without normals do not bias the direction
 *   colour     (sum + n/2) / n per channel (integer division), count n (uint32)
 * The exact arithmetic is in 3dscan_b200/common/scan3d_voxel_math.h.
 *
 * Output order: voxels come in order of their first point.  Points are numbered across all adds since begin, first by
 * add, then by position within the add; dropped points take no place.  Adding A then B gives the same per-voxel
 * values as B then A, only the order differs.
 *
 * scan3d_voxel_begin: resets the ctx's accumulator and sizes it for up to max_voxels distinct voxels (device memory of
 * about 190 B per voxel plus 31 B per voxel of outputs, reused by later begins that ask for no more).  The
 * accumulator is independent of the ctx's points: a later reconstruct does not touch it.  No kernel launch.
 * scan3d_voxel_add_points: the ctx's current points, wherever they are (scan3d_set_points_buffer included, row-sharded
 * contexts included); each brings its normal from the mesh when the mesh of the current points is fresh
 * (scan3d_build_mesh), else (0,0,0), and its colour when a texture is set, else (0,0,0), as scan3d_write_ply does.
 * Always 5 kernel launches.
 * scan3d_voxel_add_points_dev: n points from caller device memory on the ctx's GPU (xyz f32[n][3], normals f32[n][3]
 * or NULL, rgb u8[n][3] or NULL; NULL means zeros), ordered on the ctx stream.  Runs in chunks of W*H points, 5 kernel
 * launches per chunk (none for n = 0); the order rule holds across chunks.
 * Both adds are asynchronous and never synchronise.
 * scan3d_voxel_finish: computes the outputs, asynchronously, 1 kernel launch.  A begin or an add after it makes the
 * outputs stale: the getters below return SCAN3D_ERR_STATE before the first finish and while the outputs are stale.
 *
 * Errors: SCAN3D_ERR_ARG for voxel_size not finite or <= 0, max_voxels < 1 or >= 2^31, a null xyz_dev with n > 0,
 * n < 0, xyz_dev / normals_dev not 4-byte aligned, a null path.  SCAN3D_ERR_STATE for an add before begin, a ctx add
 * without points or with dirs == 1.  SCAN3D_ERR_CONFIG, before any launch, for an add whose upper bound (W*H for the
 * ctx add, n for the dev add) would push the points since begin past 2^32 - 1.
 * More distinct voxels than max_voxels is detected on the device; the adds stop inserting new voxels, so they neither
 * hang nor write outside their buffers.  The condition is sticky: scan3d_voxel_count, scan3d_get_voxels and
 * scan3d_write_voxel_ply return SCAN3D_ERR_CONFIG with a message until the next begin. */
int scan3d_voxel_begin(scan3d_ctx *ctx, float voxel_size, int64_t max_voxels);
int scan3d_voxel_add_points(scan3d_ctx *ctx);                       /* the ctx's current points */
int scan3d_voxel_add_points_dev(scan3d_ctx *ctx, const float *xyz_dev, const float *normals_dev,
                                const uint8_t *rgb_dev, int64_t n);
int scan3d_voxel_finish(scan3d_ctx *ctx);                           /* async */
/* syncs; either pointer may be NULL */
int scan3d_voxel_count(scan3d_ctx *ctx, int64_t *voxels_out, int64_t *dropped_out);
/* xyz f32[n][3], normals f32[n][3], rgb u8[n][3], counts u32[n] of the first n = min(voxels, max_voxels) voxels;
 * any pointer may be NULL */
int scan3d_get_voxels(scan3d_ctx *ctx, float *xyz_host, float *normals_host, uint8_t *rgb_host,
                      uint32_t *counts_host, int64_t max_voxels);
/* the vertex element of scan3d_write_mesh_ply ("x y z nx ny nz red green blue"), no face element; ascii (%.9g) or
 * binary_little_endian */
int scan3d_write_voxel_ply(scan3d_ctx *ctx, const char *path, int binary);

/* ---- scan-to-model alignment: point-to-plane ICP of a view against the merged voxel cloud (the reference's users ran
 * MeshLab's ICP on the exported clouds) -------------------------------------------------------------------------------
 * Refines a rigid estimate T (p_model = T p_source) of a roughly registered view before it is added to the merge, so
 * that an error of the turntable angle or pivot (register_point_clouds' Pi = 22/7 alone rotates by theta * 1.000402)
 * does not place one surface in the merge several times.
 *
 * Model: the outputs of the last scan3d_voxel_finish whose normal is not (0,0,0).  The align reads the accumulator and
 * never changes it: the voxel getters return the same bytes before and after.
 * Source: scan3d_align_to_voxels uses the ctx's current points, wherever they are (scan3d_set_points_buffer and
 * row-sharded contexts included); scan3d_align_to_voxels_dev uses n points xyz f32[n][3] in device memory of the ctx's
 * GPU, ordered on the ctx stream.  Sample j is point j * stride.  A point with a non-finite coordinate, or whose
 * transformed coordinate / max_distance (1 + 2^-20) has a cell outside [-2^20, 2^20) on some axis, is never paired.
 * Correspondence: for p' = T p (double), the model point q with the smallest ((dx*dx + dy*dy) + dz*dz) in double, a
 * tie going to the smaller voxel ordinal; the pair is kept when that is <= max_distance^2.  This is the exact nearest
 * neighbour within the radius: the search covers every model point that can qualify (a cell index of edge
 * max_distance (1 + 2^-20) and the 27 cells around the query's).
 * Update: each pair gives J = [p' x n_q, n_q] and r = (p' - q) . n_q; with A = sum J^T J and b = sum J^T r the update
 * solves (A + mu I) x = -b by an LDL^T factorisation, mu = 1e-6 * trace(A) / 6, which keeps a rank-deficient scene (a
 * plane alone; the synthetic plane + sphere, free to turn about the plane normal through the sphere centre) finite.
 * x = (omega, v); dR = Rodrigues(omega) exactly (sin and cos by a fixed polynomial, not the small-angle matrix);
 * T <- [dR | v] T.  The run ends converged (status 0) after an update with |omega| <= stop_rotation and |v| <=
 * stop_translation (stop_rotation = stop_translation = 0: never), at the iteration limit (status 1), or with fewer than
 * 6 pairs or a solve that fails its pivot test (every pivot > mu / 2, mu finite and > 0; status 2, T = the last good
 * estimate, T_init when no update succeeded).  rms_* = sqrt(sum r^2 / pairs) of an iteration's pairs before its
 * update (0 without pairs).  The exact arithmetic is in 3dscan_b200/common/scan3d_align_math.h; the sums are reduced
 * in a fixed order, so results are bit-reproducible and independent of the GPU's SM count.
 * apply = 1: the source is then transformed in place by the returned T rounded to float, by scan3d_register_points'
 * kernel with the translation in R's fourth column and a zero pivot (register_point's float operation order).  On the
 * ctx variant this rewrites the points, so the mesh becomes stale, as after every other rewriting entry.
 * Synchronisation: the iteration loop, the convergence test and the state live in device memory; the host does not
 * wait between iterations.  The entry synchronises the ctx stream once, at the end, to copy the result out (the
 * apply, if any, is queued after that and runs asynchronously).
 * Launches: always 3 (cell index of the model) + 2 per max_iterations (match, solve; those after the run ended return
 * at once) + 1 with apply when the source is not empty.  The index buffers (about 60 B per max_voxels) are ctx-owned,
 * allocated by the first align and grown with max_voxels.
 * Errors: SCAN3D_ERR_ARG for null pointers (xyz_dev may be NULL when n = 0), a max_distance not finite or <= 0,
 * max_iterations outside 1..64, stride < 1, a negative or NaN stop threshold, n < 0, xyz_dev not 4-byte aligned, or a
 * T_init that is not finite, whose last row is not (0, 0, 0, 1) or whose 3x3 block R is not a rotation within 1e-6
 * (every element of R^T R - I, and det R - 1, within 1e-6).  SCAN3D_ERR_STATE before scan3d_voxel_begin, before the
 * first scan3d_voxel_finish or after an add since it; for the ctx variant also without points or with dirs == 1.
 * SCAN3D_ERR_CONFIG when the accumulator overflowed (max_voxels too small), found on the device and reported after the
 * final synchronisation, without applying. */
typedef struct {
    double T_init[16];         /* row-major 4x4 rigid start estimate (identity when the nominal registration is already
                                  folded into the points) */
    float max_distance;        /* correspondence radius, finite, > 0 (model units) */
    int32_t max_iterations;    /* 1..64 */
    int32_t stride;            /* >= 1: source sample j is point j * stride */
    double stop_rotation;      /* radians, >= 0 */
    double stop_translation;   /* model units, >= 0; 0 and 0 = always run max_iterations */
    int32_t apply;             /* 1: transform the source cloud in place by the returned T */
} scan3d_align_params;

typedef struct {
    double T[16];              /* p_model = T p_source; T_init when no update succeeded */
    int32_t iterations;        /* updates applied */
    int32_t status;            /* 0 converged, 1 iteration limit, 2 too few pairs / singular system (T = last good) */
    int64_t pairs_first, pairs_last;   /* correspondences of the first / last iteration */
    double rms_first, rms_last;        /* point-to-plane RMS of those iterations, before their update */
} scan3d_align_result;

int scan3d_align_to_voxels(scan3d_ctx *ctx, const scan3d_align_params *p, scan3d_align_result *out);
int scan3d_align_to_voxels_dev(scan3d_ctx *ctx, float *xyz_dev, int64_t n, const scan3d_align_params *p,
                               scan3d_align_result *out);

/* ---- either side of the path (SURVEY.md 8 f2 / f4) --------------------------------------- */
/* cvUndistort2(cap, undist_cap, K, d) as the capture loop applies it to every captured camera frame
 * and every projected pattern (2/project_pattern.cpp:220,234,372-427): OpenCV 2.4's cv::undistort,
 * i.e. the 5-fractional-bit map of initUndistortRectifyMap (built in stripes of max(1, 4096/W) rows)
 * and cv::remap's fixed-point bilinear blend with a constant 0 border -- bit-identical to OpenCV.
 * device_kind 0 = camera (Kc, dc; frames [n][H][W]), 1 = projector (Kp, dp; frames [n][PH][PW]).
 * The map is built on the GPU once per calibration and reused for every frame (the reference
 * rebuilds it per image).  src and dst must not overlap.  Needs scan3d_set_calibration. */
int scan3d_undistort_frames(scan3d_ctx *ctx, int device_kind, const uint8_t *src_host, int n_frames,
                            uint8_t *dst_host);
int scan3d_undistort_frames_dev(scan3d_ctx *ctx, int device_kind, const uint8_t *src_dev, int n_frames,
                                uint8_t *dst_dev);
/* that map, for diffing against cv::initUndistortRectifyMap(CV_16SC2): xy = int16 [H][W][2] (source
 * column, row), frac = uint16 [H][W] (fy*32 + fx).  Either destination may be NULL. */
int scan3d_get_undistort_map(scan3d_ctx *ctx, int device_kind, int16_t *xy_host, uint16_t *frac_host);

/* image_scissor()'s scan-line fill (M_tech_project_console/m_tech_project_console.cpp:186-229): from
 * the lasso outline the user drew (internal_image, non-zero = outline, u8 [H_total][W]) to
 * selected_region (u8 [H_total][W], 1 = selected): every zero pixel strictly between the first and the
 * last outline pixel of its row.  filled (optional) receives the outline image after the reference's
 * in-place fill -- what it saves as i1.jpg; filled_dev may equal outline_dev. */
int scan3d_roi_fill(scan3d_ctx *ctx, const uint8_t *outline_host, uint8_t *roi_host, uint8_t *filled_host);
int scan3d_roi_fill_dev(scan3d_ctx *ctx, const uint8_t *outline_dev, uint8_t *roi_dev, uint8_t *filled_dev);

/* register_point_clouds()'s per-cloud transform (9/register_point_clouds.cpp:93-137): rotate the
 * cloud captured at turntable angle theta_deg about the Y axis through the pivot (tx,ty,tz), in the
 * reference's float arithmetic (its Pi = 22/7 included).  xyz = f32 [n][3]; dst may equal src. */
int scan3d_register_points(scan3d_ctx *ctx, const float *src_host, float *dst_host, int64_t n,
                           float theta_deg, float tx, float ty, float tz);
int scan3d_register_points_dev(scan3d_ctx *ctx, const float *src_dev, float *dst_dev, int64_t n,
                               float theta_deg, float tx, float ty, float tz);
/* the 4x4 float matrix R it uses (row-major), for diffing */
int scan3d_register_rotation(float theta_deg, float R[16]);

/* Both steps folded into the single-pass entry (SURVEY.md 8 f4):
 * scan3d_set_registration: the points scan3d_reconstruct[_dev] produces from now on are already rotated by
 * theta_deg about the Y axis through (tx,ty,tz) -- register_point_clouds' transform applied to each float point where
 * the kernel stores it, bit-identical to scan3d_register_points run afterwards, without another pass over the cloud.
 * enable = 0 switches it off.
 * scan3d_reconstruct_raw[_dev]: raw = the captured stack BEFORE the capture loop's cvUndistort2 (same plane order as
 * scan3d_reconstruct): undistorts every frame (camera calibration) into a ctx-owned stack and runs the single-pass
 * kernel on it, chained on the ctx's stream -- one call from raw captures to (registered) points, equal to
 * scan3d_undistort_frames + scan3d_reconstruct (+ scan3d_register_points).  Whole-frame contexts only. */
int scan3d_set_registration(scan3d_ctx *ctx, int enable, float theta_deg, float tx, float ty, float tz);
int scan3d_reconstruct_raw(scan3d_ctx *ctx, const uint8_t *raw_stack_host, const uint8_t *roi_host, int64_t *count_out);
int scan3d_reconstruct_raw_dev(scan3d_ctx *ctx, const uint8_t *raw_stack_dev, const uint8_t *roi_dev);

/* Several contexts on several streams of ONE GPU (a batch of scans, BASELINE configs[3]): limit the persistent kernel
 * of this context to ctas_per_sm of the SM's CTA slots (it can hold 2-4, depending on the frame stack), so that the
 * kernels of the other contexts are resident beside it and the pipeline fill and drain of one scan overlap the
 * steady state of the others.  0 = no limit (default: one context then uses the whole GPU). */
int scan3d_set_cta_limit(scan3d_ctx *ctx, int ctas_per_sm);

/* number of kernels this ctx has launched since creation (bench.py's gpu_launches) */
int64_t scan3d_launch_count(const scan3d_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* SCAN3D_H */
