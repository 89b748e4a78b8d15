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
 * NULL clears it.  Points carry colours only if a texture was set when they were computed (a reconstruct or
 * scan3d_compact_points) and scan3d_set_texture(NULL) has not run since; otherwise their colours are zeros. */
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
 * (scan3d_build_mesh), else (0,0,0), and its colour as scan3d_write_ply writes it: the texture's when a texture was
 * set when the points were computed and scan3d_set_texture(NULL) has not run since, else (0,0,0).
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

/* ---- triangle surface of the merged voxels: point-to-plane distance on the voxel lattice (Hoppe et al. 1992), meshed
 * by naive surface nets (Gibson 1998) --------------------------------------------------------------------------------
 * One closed, oriented triangle surface of the whole object from the merge, in place of the reconstruction the
 * reference's users ran in another tool.  A pure function of the merge outputs, their order and max_distance: the
 * result is bit-reproducible and does not depend on the hash, the scheduling or the GPU's SM count.
 *
 * s = the voxel_size of the last scan3d_voxel_begin, S = (double)s.  The model is the outputs of the last
 * scan3d_voxel_finish whose normal is not (0,0,0), with their ordinals o (the alignment's model).
 * Lattice point g = (i, j, k), integers in [-2^20, 2^20); x_g = ((double)i*S, (double)j*S, (double)k*S).  Cell g is the
 * cube with min corner g, corners g + (a, b, c), a, b, c in {0, 1}.  A model voxel sits in the cell of its own merge
 * index (not recomputed from its rounded output coordinate).
 * Candidate cell: some model voxel v has max(|g - v|) <= 1 on every axis.  A cell with a corner outside the key range is
 * never active and is not held.
 * Corner value f(g): q = the nearest model point to x_g by the alignment's rule (d = ((dx*dx + dy*dy) + dz*dz) in
 * double, dx = x_g - (double)q_x; q qualifies when d <= R*R, R = (double)max_distance; a tie goes to the smaller
 * ordinal); f(g) = (dx*n_x + dy*n_y) + dz*n_z with q's normal n (the alignment's residual).  Undefined when no model
 * point is within R.  g is inside when f < 0, outside when f >= 0.
 * Active cell: a candidate whose 8 corners are all defined and not all on one side.
 * Vertex of an active cell: its 12 edges in the order: the four x-edges at (b, c) = (0,0), (1,0), (0,1), (1,1), then the
 * four y-edges at (a, c) and the four z-edges at (a, b) in the same pattern.  On each edge whose lower end u and upper
 * end w lie on different sides, t = f_u / (f_u - f_w); the crossing takes ((double)g_u,axis + t)*S on the edge's axis
 * and x_u's other two coordinates.  Per axis the crossings are summed in edge order from +0, divided by their number
 * in double and rounded to float.
 * Vertex normal: the trilinear gradient g_x = ((f100 - f000) + (f110 - f010)) + ((f101 - f001) + (f111 - f011)), g_y,
 * g_z likewise over the (0,0), (1,0), (0,1), (1,1) pattern of the other two axes, divided by sqrt((g_x^2 + g_y^2) +
 * g_z^2) in double and rounded to float; (0,0,0) when that length is 0 or not finite.
 * Vertex colour: per channel (sum of the 8 corners' nearest model points' colours + 4) / 8, integer division.
 * Faces: for each active cell g and axis a = x, y, z, with (b, d) the next two axes in cyclic order ((y,z), (z,x),
 * (x,y)): lattice edge g -> g + e_a gives a quad when its ends are on different sides and cells g, g - e_b,
 * g - e_b - e_d and g - e_d are all active.  v0..v3 = the vertices of g - e_b - e_d, g - e_d, g, g - e_b; when
 * f(g) < 0 <= f(g + e_a) the triangles are (v0, v1, v2), (v0, v2, v3), else (v0, v2, v1), (v0, v3, v2): every face's
 * right-hand normal points from inside to outside, the direction of the model normals.
 * Order: vertices by their cell's key min(27*o + k) over the model voxels v_o that make it a candidate, k = ((dz+1)*3 +
 * (dy+1))*3 + (dx+1) for the offset g - v_o; faces by their v2, then the axis, then the two triangles.  Vertex indices
 * are int32.  The exact arithmetic is in 3dscan_b200/common/scan3d_surface_math.h.
 * Synchronisation: scan3d_voxel_surface synchronises the ctx stream once, after the counts are known; the vertex and
 * face buffers are then sized, *out is filled and the emission is queued asynchronously.
 * Launches: always 3 (the alignment's cell index of the model, cell edge max_distance (1 + 2^-20)) + 8 (candidate
 * cells, their corners, corner values, active-cell flags, their k_count + k_scan, vertex ordinals with face counts,
 * the scan of those) before the synchronisation, + 1 (the emission) when it succeeds.
 * Memory (ctx-owned, allocated by the first extraction, grown on demand): about 68 B per max_points, 27 B + the index's
 * ~60 B per max_voxels, and 27 B per vertex + 12 B per face.
 * The extraction never changes the accumulator: the voxel getters return the same bytes before and after.  A later
 * begin, add or finish makes the surface stale (the getters and the writer then return SCAN3D_ERR_STATE); an align,
 * with or without apply, does not.  A failed extraction leaves no surface behind.
 * Errors: SCAN3D_ERR_ARG for null pointers, a max_distance not finite or <= 0, max_points outside [1, 2^31), a null
 * path.  SCAN3D_ERR_STATE before scan3d_voxel_begin, before the first scan3d_voxel_finish or after an add since it.
 * SCAN3D_ERR_CONFIG when the accumulator overflowed (max_voxels too small), or when more than max_points distinct
 * lattice points were needed: both are found on the device (inserting stops, so nothing hangs or overruns) and reported
 * at the synchronisation.  A model without normals gives 0 vertices and 0 faces, with SCAN3D_OK. */
typedef struct {
    float max_distance;        /* R: finite, > 0 (model units) */
    int64_t max_points;        /* capacity in distinct lattice points (candidate cells and their corners), 1 .. 2^31 - 1 */
} scan3d_surface_params;

typedef struct {
    int64_t vertices, faces;
    int64_t lattice_points;    /* distinct lattice points held (to size max_points) */
    int64_t undefined_points;  /* of them, without a model point within R (to choose R) */
} scan3d_surface_result;

int scan3d_voxel_surface(scan3d_ctx *ctx, const scan3d_surface_params *p, scan3d_surface_result *out);
/* xyz f32[v][3], normals f32[v][3], rgb u8[v][3] of the first v = min(vertices, max_vertices) vertices, faces
 * int32[f][3] of the first f = min(faces, max_faces) faces; any pointer may be NULL; syncs */
int scan3d_get_voxel_surface(scan3d_ctx *ctx, float *xyz, float *normals, uint8_t *rgb, int32_t *faces,
                             int64_t max_vertices, int64_t max_faces);
/* the vertex element of scan3d_write_mesh_ply plus its face element; ascii (%.9g) or binary_little_endian */
int scan3d_write_voxel_surface_ply(scan3d_ctx *ctx, const char *path, int binary);

/* ---- connected components of a triangle mesh; removal of the small pieces of the surface ----------------
 * Component: two vertices are connected when some face contains both; a face connects its three vertices (a degenerate
 * face such as (a, a, b) is allowed).  A vertex that no face uses is a component by itself, with 0 faces.  A face
 * belongs to the component of its vertices.
 * Component id: components are ranked by their smallest vertex index (the component of vertex 0 has id 0).  The labels
 * are a pure function of the faces and the vertex count: they do not depend on scheduling or on the SM count.
 * Keep rule (min_faces >= 0, max_components >= 0, 0 = no limit): of the components with at least min_faces faces, the
 * first max_components ranked by faces in descending order, ties going to the smaller id.  (0, 0) keeps everything;
 * min_faces = 1 drops the vertices that no face uses.
 * Compaction: kept vertices keep their relative order and their xyz, normal and rgb bytes; kept faces keep their
 * relative order with their indices remapped to the new vertex positions: new = cumsum(keep_v) - 1,
 * faces = new[faces[keep_f]].
 * Method: a lock-free union-find (ECL-CC: atomicCAS links the larger root under the smaller, finds halve the path), so
 * every root is its component's smallest vertex; the roots ranked by k_count + k_scan give the ids.  Counts per
 * component are integer atomics and the selection is an integer radix select, so every result is bit-reproducible.
 * scan3d_voxel_surface_components labels the held voxel surface, then replaces it in place by its kept components:
 * scan3d_get_voxel_surface and scan3d_write_voxel_surface_ply then return the cleaned surface, and a second call with
 * the same parameters changes nothing.  It needs a held surface (SCAN3D_ERR_STATE otherwise).  A later
 * scan3d_voxel_surface, begin, add or finish makes the component table stale (scan3d_get_surface_components then
 * returns SCAN3D_ERR_STATE); the staleness of the surface itself is unchanged; an align changes neither the surface nor
 * the table; the accumulator is never touched.
 * scan3d_mesh_components_dev labels any triangle mesh in device memory of the ctx's GPU (faces int32 [n_faces][3],
 * labels int32 [n_vertices]), ordered on the ctx stream; it leaves the held surface and the table alone.
 * Synchronisation: one per entry.  scan3d_voxel_surface_components synchronises once the counts, the selection and
 * the kept totals are known; *out is then filled and the compaction is queued asynchronously.
 * Launches: scan3d_mesh_components_dev always 7 (parent = v, one union per face, find per vertex with the root flags,
 * their k_count + k_scan, the roots' ids, every vertex's id).  scan3d_voxel_surface_components always 16, even for
 * (0, 0): those 7, then the counts per component, the selection, the keep flags, k_count + k_scan over the vertex
 * flags and over the face flags before the synchronisation, and 2 after it (kept vertices, kept faces).  With (0, 0)
 * the surface's bytes are unchanged.
 * Memory (ctx-owned, allocated on first use, grown on demand): 18 B per vertex and 1 B per face of scratch and
 * component table, plus the spare surface set of 27 B per kept vertex and 12 B per kept face that is swapped with the
 * held one.
 * Errors: SCAN3D_ERR_ARG for a null ctx, params, result or components_out; faces_dev NULL with n_faces > 0 or
 * label_dev NULL with n_vertices > 0; a negative min_faces or max_components; n_faces or n_vertices outside
 * [0, 2^31); device pointers not 4-byte aligned; and in scan3d_mesh_components_dev a face index outside
 * [0, n_vertices), which is found on the device and reported at the synchronisation (the labels are then
 * unspecified).  An argument or state error launches nothing and leaves the surface as it was. */
typedef struct {
    int64_t min_faces;       /* >= 0 */
    int64_t max_components;  /* >= 0, 0 = no limit */
} scan3d_components_params;

typedef struct {
    int64_t components;      /* of the surface as it was when the call began */
    int64_t kept;            /* components kept */
    int64_t vertices, faces; /* of the surface after the call */
    int64_t largest_faces;   /* faces of the component with the most, 0 for an empty surface */
} scan3d_components_result;

/* labels the held voxel surface, then replaces it in place by its kept components */
int scan3d_voxel_surface_components(scan3d_ctx *ctx, const scan3d_components_params *p, scan3d_components_result *out);
/* per component of the last call, in id order: vertex count, face count, kept flag of the first
 * min(components, max_components); any pointer may be NULL; syncs */
int scan3d_get_surface_components(scan3d_ctx *ctx, int64_t *vertices, int64_t *faces, uint8_t *kept,
                                  int64_t max_components);
/* labels of any triangle mesh in device memory of the ctx's GPU, ordered on the ctx stream; syncs once */
int scan3d_mesh_components_dev(scan3d_ctx *ctx, const int32_t *faces_dev, int64_t n_faces, int64_t n_vertices,
                               int32_t *label_dev, int64_t *components_out);

/* ---- simplification of the voxel surface: vertex clustering on a coarser grid with quadric placement (Rossignac &
 * Borrel 1993; Lindstrom 2000) ---------------------------------------------------------------------------------------
 * scan3d_voxel_surface_decimate replaces the held voxel surface in place by its simplification: scan3d_get_voxel_surface,
 * scan3d_write_voxel_surface_ply and scan3d_voxel_surface_components then work on the simplified surface.  The result
 * is a pure function of the held surface and cell_size: bit-reproducible, independent of scheduling and SM count.
 *
 * s = the voxel_size of the last scan3d_voxel_begin, H = (double)cell_size, r = H / s in [1, 256].
 * Cluster: a vertex's voxel of edge H in the merge's sense (per axis t = (double)x / H, i = floor(t), fraction
 * f = t - i in [0, 1]; the merge's key range).  Clusters are numbered in order of their first vertex (the merge's order
 * rule).  Each cluster becomes one output vertex, at the cluster's ordinal: its normal and colour are the merge's rules
 * over the cluster's vertices (the vertex normals as the points' normals, the vertex colours as their colours); its
 * position is the placement below.  Every cluster is output, including clusters that no kept face uses: a later
 * scan3d_voxel_surface_components with min_faces = 1 removes those.
 * Face quadric: for a face (a, b, c), d1 = p_b - p_a, d2 = p_c - p_a per axis in double; n = (d1y d2z - d1z d2y,
 * d1z d2x - d1x d2z, d1x d2y - d1y d2x); l2 = (nx nx + ny ny) + nz nz.  l2 == 0: the face adds no quadric (it still
 * counts for the faces below).  Else u = n / sqrt(l2) and w = (sqrt(l2) * 0.5) / (H * H), the face's area in cell units.
 * Each corner k, with its fractions f_k in its own cluster, has e = (u_x f_x + u_y f_y) + u_z f_z and adds the 10
 * coefficients (w * c_j) for c = (u_x u_x, u_x u_y, u_x u_z, u_y u_y, u_y u_z, u_z u_z, u_x e, u_y e, u_z e, e e), each
 * rounded to the int64 rint((w * c_j) * 2^40), half to even, to its cluster's sums (int64, two's complement; the bound
 * that keeps them below 2^63 for r in [1, 256] is derived in 3dscan_b200/common/scan3d_decimate_math.h).
 * Placement: A = the symmetric 3x3 matrix of the first 6 sums * 2^-40 (A00, A01, A02, A11, A12, A22), b = the next 3
 * * 2^-40; ybar = the cluster's mean in cell units from the merge's sums, sum q_a / (2^24 n).  tr = (A00 + A11) + A22;
 * tr == 0: y = ybar.  Else mu = 1e-3 * (tr / 3) and (A + mu I) y = b + mu ybar is solved by the alignment's LDL^T
 * (pivot test: mu finite and > 0, every pivot > mu / 2).  When the pivot test fails, or some y_a is not finite or not
 * in [0, 1], y = ybar and the cluster counts in mean_fallbacks.  The output coordinate is (float)(((double)i_a + y_a)
 * * H).  The exact operation order is in 3dscan_b200/common/scan3d_decimate_math.h.
 * Faces: face (a, b, c) maps to (C(a), C(b), C(c)), the cluster ordinals.  A face with two of them equal is dropped
 * (collapsed_faces).  The canonical triple is the cyclic rotation that puts the smallest ordinal first, which keeps
 * the winding; of the faces with the same canonical triple the first by face index is kept, the others are dropped
 * (duplicate_faces).  Opposite windings are different triples, so both are kept.  Kept faces keep their relative
 * order and their rotation.  The output can be non-manifold where a cluster joins two sheets of the surface.
 * State: needs a held surface (SCAN3D_ERR_STATE otherwise).  A surface is simplified once: a second call returns
 * SCAN3D_ERR_STATE until a new scan3d_voxel_surface (the overflow bound rests on surface-nets faces).  Components
 * before and after are allowed; the call makes the component table stale.  A later begin, add or finish makes the
 * surface stale as before; an align touches neither; the accumulator is never changed.
 * Synchronisation: one, after every launch, when the counts are known; *out is then filled and the simplified set
 * swapped in.
 * Launches: always 12, an empty surface included: 5 (the merge's add over the vertices), the face quadrics, the
 * duplicate-face table, the keep flags, k_count + k_scan over them, the vertices (placement), the faces.
 * Memory (ctx-owned, allocated on first use, grown on demand): about 275 B per vertex (the cluster table at ~184 B, the
 * quadric sums indexed by cluster ordinal at 80 B, 9 B of scratch) and 25 B per face (cluster triples, duplicate
 * table, slots and flags), plus the spare surface set, grown to 27 B per vertex and 12 B per face of the
 * input, which is swapped with the held one.
 * Errors: SCAN3D_ERR_ARG for a null ctx or out, a cell_size that is not finite, and (with a held surface) cell_size <
 * voxel_size or > 256 voxel_size; SCAN3D_ERR_CONFIG for a surface of 2^31 faces or more.  An argument, state or
 * size error launches nothing and leaves the surface as it was.  An empty surface gives 0 vertices and 0 faces,
 * with SCAN3D_OK. */
typedef struct {
    int64_t vertices, faces;     /* of the surface after the call */
    int64_t collapsed_faces;     /* dropped: two corners in one cluster */
    int64_t duplicate_faces;     /* dropped: same oriented cluster triple as an earlier face */
    int64_t mean_fallbacks;      /* clusters placed at their mean instead of the quadric minimum */
} scan3d_decimate_result;

int scan3d_voxel_surface_decimate(scan3d_ctx *ctx, float cell_size, scan3d_decimate_result *out);

/* ---- smoothing of the voxel surface and of device meshes: Taubin lambda|mu fairing with the uniform umbrella
 * operator (Taubin 1995), boundaries held ------------------------------------------------------------------------------
 * The result is a pure function of the mesh and the parameters: bit-reproducible, independent of scheduling, of the
 * hash and of the SM count.  The exact operation order is in 3dscan_b200/common/scan3d_smooth_math.h.
 *
 * Neighbours: each face (a, b, c) contributes its sides (a, b), (b, c), (c, a); a side with equal ends is skipped.
 * Two vertices are neighbours when some side joins them; the count of an undirected edge is the number of sides on it.
 * A vertex on an edge whose count is not 2 is held: open boundaries (count 1) and non-manifold edges (3 or more).
 * Held vertices and vertices without a neighbour (isolated) keep their xyz bytes exactly; the others are free.
 * Fixed point: 2^E is the smallest power of two above every |coordinate| of the mesh (E = the largest biased float
 * exponent field - 126, an exact max on the device); every vertex's position is the int64 Q = rint((double)x *
 * 2^(40 - E)), half to even, so coordinates down to 2^(E - 17) are held exactly.
 * Pass: every free vertex with d distinct neighbours, per axis, S = sum of the neighbours' Q (exact integers, so the
 * order of the neighbours does not matter), m = (double)S / (double)d, Q' = Q + rint(k * (m - (double)Q)), with
 * separately rounded IEEE operations (no FMA) and k = (double)lambda or (double)mu.  An iteration is a lambda pass then
 * a mu pass; mu = 0 gives plain Laplacian smoothing with one pass per iteration.  At the end a free vertex takes
 * (float)((double)Q * 2^(E - 40)).  iterations = 0 only quantises the free vertices and recomputes the normals.
 * Normals, recomputed from the final float positions: for each face with three distinct indices, the unit normal of
 * (p_b - p_a) x (p_c - p_a) in double, as a float, in the merge's fixed point (clamped to [-1, 1], rint(v * 2^24)), is
 * added to each of its three vertices (a face with a zero or non-finite cross product adds nothing); a vertex's normal
 * is then the merge's normalisation of its integer sums, and a vertex whose sums are all zero keeps its normal bytes.
 * Equal-weight face normals keep the sums of any hub below 2^55.
 * Limits (derived in the math header; each fails the whole call with SCAN3D_ERR_CONFIG and nothing is written): a free
 * vertex with more than 2^20 neighbours; a free vertex with some |Q| > 2^42 after a pass (a mu pass moves vertices away
 * from their neighbours' mean); a free vertex whose output coordinate rounds to +-inf; 6 * n_faces >= 2^32.
 *
 * scan3d_voxel_surface_smooth smooths the held voxel surface in place: scan3d_get_voxel_surface and
 * scan3d_write_voxel_surface_ply then return it.  Faces, colours and the vertex order do not change, so a component
 * table of scan3d_voxel_surface_components stays valid.  It needs a held surface (SCAN3D_ERR_STATE otherwise).
 * Smoothing after components or decimation is allowed, and so is smoothing again.  scan3d_voxel_surface_decimate
 * refuses a smoothed surface with SCAN3D_ERR_STATE until a new scan3d_voxel_surface (its overflow bound rests on
 * surface-nets geometry, which smoothing does not keep).  A later begin, add or finish makes the surface stale as
 * before; the accumulator is never touched.  The result is computed into the spare surface set and
 * swapped with the held one after the synchronisation, so on any error the surface is untouched.
 * scan3d_mesh_smooth_dev smooths any triangle mesh in device memory of the ctx's GPU in place: xyz_dev float
 * [n_vertices][3], normals_dev float [n_vertices][3] or NULL (no normals), faces_dev int32 [n_faces][3]; ordered on the
 * ctx stream.  It leaves the held surface and the component table alone, and on any error leaves the buffers as they
 * were.  The ctx's own camera-grid mesh is a valid target: scan3d_device_points, scan3d_device_point_normals and
 * scan3d_device_mesh_faces with the counts of scan3d_point_count and scan3d_mesh_face_count; the mesh stays valid, and
 * scan3d_write_mesh_ply then writes the smoothed single view.  The next reconstruct overwrites the points.
 * Synchronisation: one per call, after every launch.
 * Launches: 7 + passes + 2, with passes = iterations * 2 (mu != 0) or iterations (mu = 0), an empty mesh included:
 * the exponent max, the sides into the edge table, the degrees and held flags, the degree sums per block, their scan,
 * the row starts with the fixed-point positions, the neighbour rows; one gather per pass; the face normals; the write.
 * Memory (ctx-owned, allocated on first use, grown on demand): 81 B per vertex (two fixed-point position sets at 24 B,
 * the normal sums at 24 B, degree, row start and held flag) and 96 B per face (the edge table of 6 slots of 12 B, and
 * 6 row entries of 4 B); the surface route also grows the spare surface set's xyz and normals to 24 B per vertex.
 * Errors: SCAN3D_ERR_ARG for a null ctx, params or result; iterations outside [0, 4096]; lambda not in (0, 1] or mu not
 * in [-1, 0] (NaN and infinities included); and in scan3d_mesh_smooth_dev n_vertices or n_faces outside [0, 2^31), a
 * NULL xyz_dev or faces_dev with a non-zero count, a buffer not 4-byte aligned, and, found on the device, a coordinate
 * that is not finite or a face index outside [0, n_vertices).  An argument or state error launches nothing; an error
 * found on the device is reported at the synchronisation and nothing is written. */
#define SCAN3D_SMOOTH_MAX_ITERATIONS 4096
typedef struct {
    int32_t iterations;          /* [0, 4096]; MeshLab's default is 10 */
    float lambda;                /* (0, 1]; MeshLab's default is 0.5 */
    float mu;                    /* [-1, 0]; MeshLab's default is -0.53; 0 = Laplacian smoothing */
} scan3d_smooth_params;

typedef struct {
    int64_t vertices, faces;     /* of the mesh */
    int64_t held_vertices;       /* on an edge whose count is not 2 */
    int64_t isolated_vertices;   /* without a neighbour */
    int64_t passes;              /* gathers run */
    double max_displacement;     /* the largest Euclidean move of a vertex, model units */
} scan3d_smooth_result;

int scan3d_voxel_surface_smooth(scan3d_ctx *ctx, const scan3d_smooth_params *p, scan3d_smooth_result *out);
int scan3d_mesh_smooth_dev(scan3d_ctx *ctx, float *xyz_dev, float *normals_dev, int64_t n_vertices,
                           const int32_t *faces_dev, int64_t n_faces, const scan3d_smooth_params *p,
                           scan3d_smooth_result *out);

/* ---- hole filling of the voxel surface and of device meshes: minimum-weight triangulation of boundary loops with
 * Liepa's weight (Liepa 2003; Klincsek 1980; Barequet & Sharir 1995) ------------------------------------------------
 * The result is a pure function of the mesh and max_edges: bit-reproducible, independent of scheduling, of the hash and
 * of the SM count.  The exact operation order is in 3dscan_b200/common/scan3d_fill_math.h.
 *
 * Hole edges: each face (a, b, c) contributes its sides (a, b), (b, c), (c, a); a side with equal ends is skipped.  An
 * undirected edge whose side count is 1 is a boundary edge; its hole edge is the reversed side b -> a, and its rim
 * face is the one face that holds it.  A vertex is regular when exactly one hole edge leaves it and exactly one enters
 * it.  The successor of a hole edge is the hole edge that leaves its head.
 * Holes: a hole is a cycle of n hole edges, 3 <= n <= max_edges, through regular vertices only; v_0 is its smallest
 * vertex index, v_{t+1} the head of the hole edge that leaves v_t, F_t the rim face of hole edge t (v_t -> v_{t+1}).
 * Every loop of at most max_edges edges is a hole, the rim of a small open piece included.  Two kinds of boundary stay
 * open and count in open_edges: chains through vertices that are not regular (non-manifold boundary, two holes sharing
 * a vertex), and loops longer than max_edges.
 * Triangle terms, in double from the float coordinates, each operation correctly rounded: cross = (p_b - p_a) x (p_c -
 * p_a), l2 = (cx cx + cy cy) + cz cz, area = sqrt(l2) * 0.5, unit normal u = cross / sqrt(l2) when l2 > 0 (else none);
 * cos(T1, T2) = (u1x u2x + u1y u2y) + u1z u2z, and -1 when either has no normal.
 * Triangulation: for 0 <= i < j <= n - 1, cell (i, j) is the best triangulation of v_i ... v_j closed by v_j -> v_i.
 * j - i = 1 is hole edge i: feasible with weight (+inf, 0) and the normal of F_i.  A cell with j - i >= 2 is infeasible
 * when (i, j) != (0, n - 1) and {v_i, v_j} is already an edge of the mesh (so the output stays edge-manifold), or when
 * it has no feasible candidate.  Candidates k = i + 1 ... j - 1 with both cells (i, k) and (k, j) feasible give T_k =
 * (v_i, v_k, v_j), c_k = min(cos(T_k, N(i, k)), cos(T_k, N(k, j))) with N the triangle chosen for a cell (F_a for a hole
 * edge), and for cell (0, n - 1) also min with cos(T_k, F_{n-1}); cmin = min(cmin(i, k), cmin(k, j), c_k), area =
 * (area(i, k) + area(k, j)) + area(T_k).  The larger cmin wins, then the smaller area, then the smaller k.  When cell
 * (0, n - 1) is infeasible the hole is unfillable and stays open.
 * Output: a filled hole gets n - 2 faces (v_i, v_k, v_j) in preorder from cell (0, n - 1) (the cell's face, then cell
 * (i, k), then cell (k, j)), wound like the rim faces, so a flat continuation has cos = +1.  Holes are emitted in
 * ascending v_0, after the existing faces; vertices, their bytes and the existing faces do not change.  The patch has
 * no interior vertices (Liepa's refinement and fairing are not done).
 *
 * scan3d_voxel_surface_fill_holes fills the held voxel surface in place: scan3d_get_voxel_surface,
 * scan3d_write_voxel_surface_ply, components, smoothing and decimation then see the filled surface.  It needs a held
 * surface (SCAN3D_ERR_STATE otherwise), makes the component table stale and changes no other state: a filled surface
 * that was neither simplified nor smoothed can still be simplified.  For that, max_edges is capped at
 * SCAN3D_FILL_NETS_MAX_EDGES on such a surface (the decimation's quadric bound, extended to the fill faces of holes of
 * at most 22 surface-nets edges, is derived in the math header); on a simplified or smoothed surface, which decimation
 * refuses anyway, the cap is SCAN3D_FILL_MAX_EDGES.  Recommended order: extract, components, then smooth or decimate,
 * then fill; small pinholes can be filled right after extraction.  Smoothing after a fill is allowed, but a rim vertex
 * is then free and its umbrella reaches across the patch, which has no interior vertices.  A second fill adds nothing
 * unless max_edges grows.  A later begin, add or finish makes the surface stale as before.
 * scan3d_mesh_fill_holes_dev fills any triangle mesh in device memory of the ctx's GPU (xyz_dev float [n_vertices][3],
 * faces_dev int32 [n_faces][3]), capped at SCAN3D_FILL_MAX_EDGES: it writes only the added faces, int32 [faces_added][3],
 * to faces_out_dev, ordered on the ctx stream, and leaves the mesh, the held surface and the component table alone.
 * When more than max_faces_out faces are needed it writes nothing and returns SCAN3D_ERR_CONFIG with *out filled
 * (faces_added the faces needed, faces = n_faces, open_edges = boundary_edges).  The ctx's camera-grid mesh
 * (scan3d_device_points, scan3d_device_mesh_faces) is a valid input.
 * Synchronisation: two per call: once the holes are known (to size the scratch and, in the surface route, the spare
 * face set, into which the held faces are copied), and once after every launch.
 * Launches: 10, an empty mesh included: the sides into the edge table, the hole edges, the loop walks with the per-block
 * sums, k_scan over the holes, their edges and their DP cells; after the first synchronisation the holes and their
 * vertices, the DP (one block per hole), k_scan over the faces added, and the emission.  6 when the first
 * synchronisation finds an error.
 * Memory (ctx-owned, allocated on first use, grown on demand): 20 B per vertex, 96 B per face (the edge table of 6 slots
 * of 16 B), 8 B per hole edge of a hole, 20 B per hole, and 48 B per DP cell, n (n - 1) / 2 + 1 per hole of n edges
 * (25 MB for a hole of 1024); the surface route also grows the spare face set to 12 B per face after the fill.
 * Errors: SCAN3D_ERR_ARG for a null ctx or out; max_edges outside [3, cap]; in scan3d_mesh_fill_holes_dev n_vertices,
 * n_faces or max_faces_out outside [0, 2^31), a NULL xyz_dev, faces_dev or faces_out_dev with a non-zero count, a pointer
 * not 4-byte aligned, and, found on the device, a face index outside [0, n_vertices) or a coordinate that is not
 * finite.  SCAN3D_ERR_CONFIG when 6 n_faces >= 2^32, when n_faces plus the n - 2 faces of every hole reaches 2^31, or
 * when the holes' DP cells reach 2^32.
 * An argument or state error launches nothing; on any error nothing is written and the held surface is unchanged. */
#define SCAN3D_FILL_NETS_MAX_EDGES 22
#define SCAN3D_FILL_MAX_EDGES 1024
typedef struct {
    int64_t vertices, faces;     /* of the mesh after the call */
    int64_t boundary_edges;      /* hole edges before the call */
    int64_t holes;               /* loops of 3 to max_edges edges through regular vertices */
    int64_t filled;              /* holes closed; the others were unfillable */
    int64_t faces_added;
    int64_t open_edges;          /* hole edges after the call */
} scan3d_fill_result;

int scan3d_voxel_surface_fill_holes(scan3d_ctx *ctx, int32_t max_edges, scan3d_fill_result *out);
int scan3d_mesh_fill_holes_dev(scan3d_ctx *ctx, const float *xyz_dev, int64_t n_vertices, const int32_t *faces_dev,
                               int64_t n_faces, int32_t max_edges, int32_t *faces_out_dev, int64_t max_faces_out,
                               scan3d_fill_result *out);

/* ---- repair of the non-manifold edges and vertices of the voxel surface and of device meshes: MeshLab's "Repair non
 * Manifold Edges" and "Repair non Manifold Vertices by splitting" (vcglib tri::Clean; Gueziec, Taubin, Lazarus & Horn
 * 2001) ------------------------------------------------------------------------------------------------------------
 * The result is a pure function of the mesh and the flags: bit-reproducible, independent of scheduling, of the hash and
 * of the SM count.  The face key and the edge rule are in 3dscan_b200/common/scan3d_repair_math.h.
 * Flags: any non-empty combination of SCAN3D_REPAIR_FACES and SCAN3D_REPAIR_VERTICES; 0 and unknown bits are
 * SCAN3D_ERR_ARG.
 *
 * 1. Degenerate faces (always): a face with a repeated index is dropped (degenerate_faces).
 * 2. Duplicate faces (FACES): of the faces with the same set of three vertices, in either winding, the one with the
 *    smallest face index is kept and the others are dropped (duplicate_faces).  Unlike the simplification, opposite
 *    windings are duplicates too: the aim is a manifold.
 * 3. Non-manifold edges: the faces that survive steps 1-2 are counted on each undirected edge; an edge with more than 2
 *    counts in nonmanifold_edges, with or without FACES.  With FACES: each face has the key K(f) =
 *    (float_bits((float)area_f) << 32) | (0xFFFFFFFF - f), area_f the hole filling's triangle area (double, from the
 *    float coordinates).  On such an edge, f1 is the face with the largest K; f2 the face with the largest K among the
 *    faces whose side on the edge runs opposite to f1's, or, when none does, among the faces other than f1.  Every other
 *    face on the edge is dropped by it, and a face is removed when any of its edges drops it (nonmanifold_faces).  Every
 *    edge then has at most 2 faces.
 * 4. Non-manifold vertices (VERTICES): a corner (f, k) is numbered 3 f + k with the input face index.  The corners of
 *    vertex v in kept faces f and g are joined when f and g share an edge {v, w} that lies in exactly 2 kept faces; a
 *    fan is a class of joined corners.  The fan that holds v's smallest corner keeps index v; every other fan gets a
 *    new vertex, appended after the existing ones in ascending order of its smallest corner, with v's xyz, normal and
 *    rgb bytes (a copy sits exactly on its source: no vertex moves).  split_vertices counts the vertices with more than
 *    one fan, vertices_added the new vertices.
 * 5. Kept faces keep their relative order and their rotation, their corners remapped to their fans' vertices.  The
 *    input's vertices keep their index and bytes, those that no kept face uses included (components with min_faces = 1
 *    removes them).
 * With both flags no edge is in more than 2 faces and no vertex's faces form more than one fan; orientation is not
 * changed.  boundary_edges (edges in 1 kept face) and inconsistent_edges (edges in 2 kept faces whose sides run the same
 * way) are counted over the kept faces before the split; with FACES they equal the counts after the call.  A second
 * repair with the same flags changes nothing.
 *
 * scan3d_voxel_surface_repair repairs the held voxel surface in place: scan3d_get_voxel_surface,
 * scan3d_write_voxel_surface_ply and the later stages see the repaired surface.  It needs a held surface
 * (SCAN3D_ERR_STATE otherwise) and makes the component table stale (the vertex count changes); whether the surface is
 * simplified or smoothed does not change.  It is allowed before or after components, simplification, smoothing and
 * filling, and again.  Recommended order: extract, components, repair, then smooth or decimate (repair again after
 * decimating), then fill.  A repair never adds a face or moves a vertex, so a surface that could be simplified before
 * it still can.  But after a repair that dropped a face or split a vertex, a cell of the lattice can hold more than
 * one hole, which breaks the simplification's overflow bound for filled holes (derived in
 * 3dscan_b200/common/scan3d_repair_math.h): a fill that adds faces to such a surface makes scan3d_voxel_surface_decimate
 * return SCAN3D_ERR_STATE until the next scan3d_voxel_surface.  Repair before a fill of an unrefined surface only when
 * it will not be simplified, or simplify first.  A later begin, add or finish makes the surface stale as before.
 * scan3d_mesh_repair_dev repairs any triangle mesh in device memory of the ctx's GPU (xyz_dev float [n_vertices][3],
 * faces_dev int32 [n_faces][3]): it writes the kept, remapped faces, int32 [faces][3], to faces_out_dev (n_faces rows
 * always suffice; it must not be faces_dev), and the source vertex of each added vertex, int32 [vertices_added], to
 * source_out_dev (3 n_faces entries always suffice), ordered on the ctx stream; the caller extends its own attribute arrays with a gather.  It leaves the
 * inputs, the held surface and the component table alone.  When more than max_source_out vertices are needed it
 * writes nothing and returns SCAN3D_ERR_CONFIG with *out filled.  The ctx's camera-grid mesh (scan3d_device_points,
 * scan3d_device_mesh_faces) is a valid input.
 * Synchronisation: two per call, once the counts are known (to size, in the surface route, the spare surface set, into
 * which the held vertices are copied) and once after every launch.  On any error the held surface is unchanged.
 * Launches: 12, an empty mesh included: the finiteness and face-index checks with the degenerate faces and the
 * duplicate table, the keys and sides into the edge table, the largest key other than f1 per edge, the drop flags
 * with the kept faces' sides, the edge counts with the unions of the corners, the fans' roots, k_count + k_scan over
 * the new vertices and over the kept faces; after the first synchronisation the new vertices and the kept faces.  10
 * when the first synchronisation finds an error or too small a max_source_out.
 * Memory (ctx-owned, allocated on first use, grown on demand): 8 B per vertex and 353 B per face (an edge table of 6
 * slots of 48 B, the duplicate table of 2 slots of 4 B, 41 B of per-face and per-corner scratch); the surface route
 * also grows the spare surface set to 27 B per vertex and 12 B per face after the repair, and 4 B per added vertex.
 * Errors: SCAN3D_ERR_ARG for a null ctx or out; bad flags; in scan3d_mesh_repair_dev n_vertices, n_faces or
 * max_source_out outside [0, 2^31), a NULL xyz_dev, faces_dev, faces_out_dev or source_out_dev with a non-zero count,
 * a pointer not 4-byte aligned, faces_out_dev equal to faces_dev, and, found on the device, a face index outside
 * [0, n_vertices) or a coordinate that is not finite.  SCAN3D_ERR_CONFIG when 3 n_faces or the output vertex count
 * reaches 2^31.  An argument or state error launches nothing; on any error nothing is written. */
#define SCAN3D_REPAIR_FACES 1
#define SCAN3D_REPAIR_VERTICES 2
typedef struct {
    int64_t vertices, faces;     /* of the mesh after the call */
    int64_t degenerate_faces;    /* dropped: a repeated index */
    int64_t duplicate_faces;     /* dropped: the same three vertices as a face of smaller index */
    int64_t nonmanifold_edges;   /* edges in more than 2 faces after steps 1-2 */
    int64_t nonmanifold_faces;   /* dropped by a non-manifold edge */
    int64_t split_vertices;      /* vertices with more than one fan */
    int64_t vertices_added;
    int64_t boundary_edges;      /* edges in 1 kept face */
    int64_t inconsistent_edges;  /* edges in 2 kept faces whose sides run the same way */
} scan3d_repair_result;

int scan3d_voxel_surface_repair(scan3d_ctx *ctx, int32_t flags, scan3d_repair_result *out);
int scan3d_mesh_repair_dev(scan3d_ctx *ctx, const float *xyz_dev, int64_t n_vertices, const int32_t *faces_dev,
                           int64_t n_faces, int32_t flags, int32_t *faces_out_dev, int32_t *source_out_dev,
                           int64_t max_source_out, scan3d_repair_result *out);

/* ---- coherent orientation and measures of the voxel surface and of device meshes: MeshLab's "Re-Orient all faces
 * coherently" (vcglib tri::Clean::OrientCoherentlyMesh), "Compute Geometric Measures" and "Compute Topological
 * Measures" ------------------------------------------------------------------------------------------------------
 * Every result is a pure function of the mesh: bit-reproducible, independent of scheduling, of the hash and of the SM
 * count.  The arithmetic is in 3dscan_b200/common/scan3d_orient_math.h.
 *
 * Definitions.
 * - A face (a, b, c) has the sides a->b, b->c and c->a.  A face with a repeated index is degenerate: it is in no
 *   patch, has no edges, is never flipped and adds no area or volume (degenerate_faces).  A vertex is referenced when a
 *   face that is not degenerate uses it (unreferenced_vertices counts the others).
 * - The count of an undirected edge is the number of non-degenerate faces with a side on it.  Count 1: a boundary
 *   edge; 3 or more: non-manifold; 2: inconsistent when its two sides run the same way.  On the same faces these are
 *   the repair's boundary_edges, nonmanifold_edges and inconsistent_edges.
 * - A patch is a maximal set of non-degenerate faces joined across edges of count exactly 2.  It is closed when none of
 *   its faces has a boundary or non-manifold edge, and orientable when some choice of flips makes every joining edge
 *   consistent.
 * - Orientation rule.  f0 is the smallest face index of an orientable patch P; sigma(f) = +1 when f keeps its winding
 *   if f0 keeps its own, else -1; n+ counts the faces with sigma = +1 and V0 = sum sigma(f) D(f) (D below, exact).  A
 *   closed patch with V0 != 0 keeps f0's winding exactly when V0 > 0, so its normals point outward.  Any other patch
 *   keeps f0's winding exactly when 2 n+ >= |P|: the fewest faces flip, a tie keeps f0.  A flip turns (a, b, c) into
 *   (a, c, b).  Non-orientable (Moebius-like) patches are left unchanged and counted.  Face order, vertex order, xyz
 *   and rgb never change.  A referenced vertex all of whose non-degenerate faces were flipped has its normal negated
 *   (the sign bit of each component; flipped_normals counts these vertices, with or without normals); every other
 *   normal keeps its bytes.  A second orientation flips nothing.
 * - Volume and area.  c is the midpoint of the exact float bounding box of the referenced vertices, rounded to float.
 *   D(f) = det(p_a - c, p_b - c, p_c - c), six times the signed volume of the tetrahedron (c, f), in double from the
 *   float coordinates in a fixed order; area(f) is the hole filling's triangle area sqrt(l2) * 0.5.  Each term is
 *   rounded to an int64 fixed point whose scale comes from E, the exponent of the largest |p - c| of a referenced
 *   vertex (2^(59 - 3E) for D, 2^(59 - 2E) for the area), and the terms are summed exactly in int128; volume = sum D /
 *   6 and area = sum area, scaled back.  The volume is signed, with the current windings: positive for a closed
 *   surface whose normals point outward.
 * - euler_characteristic = referenced vertices - edges + non-degenerate faces.  For a closed, consistent mesh without
 *   non-manifold vertices (after a repair with SCAN3D_REPAIR_VERTICES), each patch is a closed orientable surface and
 *   genus = patches - euler_characteristic / 2; with non-manifold vertices no genus follows, so none is reported.
 * - watertight = (faces - degenerate_faces > 0) && boundary_edges == nonmanifold_edges == inconsistent_edges == 0.
 *
 * scan3d_voxel_surface_orient orients the held voxel surface in place (faces and normals); the component table stays
 * current and whether the surface is simplified or smoothed does not change.  The decimation's quadric does not depend
 * on the winding, so an oriented raw surface can still be simplified; but an orientation that flipped a face counts as
 * a repair that changed the surface: a fill that adds faces after it makes scan3d_voxel_surface_decimate return
 * SCAN3D_ERR_STATE until the next scan3d_voxel_surface (3dscan_b200/common/scan3d_orient_math.h).
 * scan3d_mesh_orient_dev orients any triangle mesh in device memory of the ctx's GPU in place (xyz_dev float
 * [n_vertices][3], read; normals_dev float [n_vertices][3] or NULL; faces_dev int32 [n_faces][3]), ordered on the ctx
 * stream.  The ctx's camera-grid mesh (scan3d_device_points, scan3d_device_mesh_faces) is a valid input.
 * scan3d_voxel_surface_measure and scan3d_mesh_measure_dev only read; they change no state.
 * Recommended order: extract, components, repair, orient, smooth or decimate, fill, measure.
 * Synchronisation: one per call, after every launch.  Launches: 8 per orientation and 7 per measure, an empty mesh
 * and an error found on the device included: the face-index check with the degenerate faces and the sides into the
 * edge table, the finiteness check with the bounding box, the edge counts with the unions and the exponent, the
 * roots with the patch sums, k_count + k_scan over the patches' smallest faces, the flips; the orientation then
 * writes the flips.
 * Memory (ctx-owned, allocated on first use, grown on demand, shared by both calls): 2 B per vertex and 173 B per face
 * (an edge table of 6 slots of 20 B, 53 B of per-face scratch).
 * Errors: SCAN3D_ERR_ARG for a null ctx or out; in the dev routes n_vertices or n_faces outside [0, 2^31), a NULL
 * xyz_dev or faces_dev with a non-zero count, a pointer not 4-byte aligned, and, found on the device, a face index
 * outside [0, n_vertices) or a coordinate that is not finite (of any vertex).  SCAN3D_ERR_CONFIG when 6 n_faces
 * reaches 2^32.  SCAN3D_ERR_STATE for the surface routes without a held surface.  An argument or state error
 * launches nothing; on any error nothing is written. */
typedef struct {
    int64_t vertices, faces;
    int64_t degenerate_faces;
    int64_t patches, closed_patches, nonorientable_patches;
    int64_t flipped_faces;
    int64_t flipped_normals;            /* referenced vertices all of whose faces were flipped */
    int64_t inconsistent_edges_before;
    int64_t inconsistent_edges;         /* after the call: those inside non-orientable patches */
} scan3d_orient_result;

typedef struct {
    int64_t vertices, faces;
    int64_t degenerate_faces;
    int64_t patches, closed_patches, nonorientable_patches;
    int64_t unreferenced_vertices;
    int64_t edges, boundary_edges, nonmanifold_edges, inconsistent_edges;
    int64_t euler_characteristic;
    int64_t watertight;                 /* 1 or 0 */
    double area, volume;                /* volume signed, with the current windings */
    float bbox_min[3], bbox_max[3];     /* of the referenced vertices; zeros when there are none */
} scan3d_measure_result;

int scan3d_voxel_surface_orient(scan3d_ctx *ctx, scan3d_orient_result *out);
int scan3d_mesh_orient_dev(scan3d_ctx *ctx, const float *xyz_dev, float *normals_dev, int64_t n_vertices,
                           int32_t *faces_dev, int64_t n_faces, scan3d_orient_result *out);
int scan3d_voxel_surface_measure(scan3d_ctx *ctx, scan3d_measure_result *out);
int scan3d_mesh_measure_dev(scan3d_ctx *ctx, const float *xyz_dev, int64_t n_vertices, const int32_t *faces_dev,
                            int64_t n_faces, scan3d_measure_result *out);

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
