// scan3d_api.cu -- the C ABI declared in include/scan3d.h: context, calibration, stage entries,
// the fused entry, result getters and the PLY writer.  No CPU compute path exists here: every
// compute entry launches CUDA kernels and fails with SCAN3D_ERR_CUDA when that is impossible.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "scan3d_internal.h"
#include "../common/scan3d_pattern_profile.h"
#include "../common/scan3d_aux_math.h"

using namespace s3d;

static thread_local std::string g_create_error;

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                \
            return SCAN3D_ERR_CUDA;                                                       \
        }                                                                                 \
    } while (0)

static int fail(scan3d_ctx* ctx, int code, const char* msg)
{
    if (ctx) ctx->err = msg;
    return code;
}

static size_t npix(const scan3d_ctx* c) { return (size_t)c->cfg.W * c->cfg.H; }

template <class T>
static cudaError_t dalloc(T** p, size_t n)
{
    return cudaMalloc((void**)p, n * sizeof(T));
}

// ---- host-side calibration algebra (once per calibration; 7/triangulation.cpp:1061-1126) ----
static void rodrigues_host(const double r[3], double R[9])
{
    // cvRodrigues2, vector -> matrix
    double rx = r[0], ry = r[1], rz = r[2];
    const double theta = sqrt(rx * rx + ry * ry + rz * rz);
    if (theta < 2.2204460492503131e-16) {
        for (int k = 0; k < 9; k++) R[k] = (k % 4 == 0) ? 1.0 : 0.0;
        return;
    }
    const double c = cos(theta), s = sin(theta), c1 = 1. - c, it = 1. / theta;
    rx *= it; ry *= it; rz *= it;
    const double eye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    const double rrt[9] = {rx * rx, rx * ry, rx * rz, rx * ry, ry * ry, ry * rz, rx * rz, ry * rz, rz * rz};
    const double rx_[9] = {0, -rz, ry, rz, 0, -rx, -ry, rx, 0};
    for (int k = 0; k < 9; k++) {
        R[k] = c * eye[k] + c1 * rrt[k] + s * rx_[k];   // host TU is built with -ffp-contract=off
    }
}

static void projection_matrix_host(const double K[9], const double rvec[3], const double t[3], double A[12])
{
    double R[9], Rt[12];
    rodrigues_host(rvec, R);
    for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) Rt[i * 4 + j] = R[i * 3 + j];
        Rt[i * 4 + 3] = t[i];
    }
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 4; j++) {
            double s = 0.0;
            for (int k = 0; k < 3; k++) s += K[i * 3 + k] * Rt[k * 4 + j];
            A[i * 4 + j] = s;
        }
}

extern "C" {

int scan3d_version(void) { return SCAN3D_VERSION; }

const char* scan3d_last_error(const scan3d_ctx* ctx)
{
    return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

int64_t scan3d_stack_bytes(const scan3d_config* c)
{
    if (!c) return 0;
    int64_t planes = c->N + 2 * c->M_v;
    if (c->dirs == 2) planes += c->N + 2 * c->M_h;
    return planes * (int64_t)c->W * c->H;
}

static int validate(const scan3d_config* c, std::string* why)
{
    if (!c) { *why = "null config"; return 0; }
    if (c->W < 1 || c->H < 1 || (int64_t)c->W * c->H > 0x7fffffffLL) { *why = "bad W/H"; return 0; }
    if (c->dirs != 1 && c->dirs != 2) { *why = "dirs must be 1 or 2"; return 0; }
    if (c->N < 3 || c->N > 16) { *why = "N must be in 3..16"; return 0; }
    if (c->M_v < 1 || c->M_v > 15 || (c->dirs == 2 && (c->M_h < 1 || c->M_h > 15))) { *why = "M must be in 1..15"; return 0; }
    if (c->fw_v < 1 || (c->dirs == 2 && c->fw_h < 1)) { *why = "fringe width must be >= 1"; return 0; }
    if (c->dirs == 2 && (c->PW < 1 || c->PH < 1)) { *why = "bad projector size"; return 0; }
    const int Ht = c->H_total > 0 ? c->H_total : c->H;
    if (c->row0 < 0 || c->row0 + c->H > Ht) { *why = "row shard outside the frame"; return 0; }
    if ((c->flags & SCAN3D_FLAG_MODULATION_MASK) && (c->N != 3 || c->row0 != 0 || Ht != c->H)) {
        *why = "the modulation criterion is defined for 3-step patterns (3/wrapped_phase.cpp:84) and needs the whole frame";
        return 0;
    }
    return 1;
}

int scan3d_create(const scan3d_config* cfg, int device, scan3d_ctx** out)
{
    if (!out) { g_create_error = "null out pointer"; return SCAN3D_ERR_ARG; }
    *out = nullptr;
    std::string why;
    if (!validate(cfg, &why)) { g_create_error = why; return SCAN3D_ERR_CONFIG; }
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
        return SCAN3D_ERR_CUDA;
    }
    scan3d_ctx* ctx = new (std::nothrow) scan3d_ctx();
    if (!ctx) { g_create_error = "out of host memory"; return SCAN3D_ERR_CUDA; }
    ctx->cfg = *cfg;
    if (ctx->cfg.H_total <= 0) ctx->cfg.H_total = cfg->H;
    ctx->device = device;
    int rc = [&]() -> int {
        int sms = 0;
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        ctx->sm_count = sms;
        CK(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
        ctx->stream = ctx->own_stream;
        const size_t n = npix(ctx);
        const int D = cfg->dirs;
        for (int d = 0; d < D; d++) {
            CK(dalloc(&ctx->unwrapped[d], n));
            CK(dalloc(&ctx->code[d], n));
        }
        CK(dalloc(&ctx->mask[0], n));
        CK(dalloc(&ctx->valid, n));
        if (D == 2) {
            CK(dalloc(&ctx->cpmap, n));
            CK(dalloc(&ctx->pts, 3 * n));
            if (cfg->flags & SCAN3D_FLAG_POINT_PIXELS) CK(dalloc(&ctx->pix, n));
        }
        CK(dalloc(&ctx->d_count, 4));
        CK(cudaMemsetAsync(ctx->d_count, 0, 16, ctx->stream));
        const int ntiles = fused_num_tiles(ctx->cfg);
        CK(dalloc(&ctx->tile_state, (size_t)ntiles + 1));
        CK(cudaMemsetAsync(ctx->tile_state, 0, ((size_t)ntiles + 1) * 8, ctx->stream));
        if (getenv("SCAN3D_TRACE")) {
            CK(dalloc(&ctx->trace, (size_t)1024 * 64 * 8));
            CK(cudaMemsetAsync(ctx->trace, 0, (size_t)1024 * 64 * 8 * 8, ctx->stream));
        }
        CK(dalloc(&ctx->sched_ctr, 4));
        CK(cudaMemsetAsync(ctx->sched_ctr, 0, 16, ctx->stream));
        CK(dalloc(&ctx->tile_flags, (size_t)ntiles + 16));
        CK(dalloc(&ctx->tile_list, (size_t)ntiles + 16));
        CK(dalloc(&ctx->atan_tab, (size_t)ATAN_TAB_DOUBLES));
        double tab[ATAN_TAB_DOUBLES];
        fill_atan_table(tab);
        CK(cudaMemcpyAsync(ctx->atan_tab, tab, sizeof(tab), cudaMemcpyHostToDevice, ctx->stream));
        CK(dalloc(&ctx->nstep_w, 128));
        double w[128];
        memset(w, 0, sizeof(w));
        for (int k = 0; k < cfg->N && k < 64; k++) {
            const double a = 2.0 * 3.14159265358979323846 * (double)k / (double)cfg->N;
            w[k] = sin(a);
            w[64 + k] = cos(a);
        }
        CK(cudaMemcpyAsync(ctx->nstep_w, w, sizeof(w), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        // exact-quotient shortcut (scan3d_math.cuh div_const): check it against IEEE division on
        // every fringe order this config can produce; any mismatch disables the shortcut
        {
            const int Mmax = cfg->dirs == 2 && cfg->M_h > cfg->M_v ? cfg->M_h : cfg->M_v;
            bool ok = true;
            const double y7 = 1.0 / 7.0;
            for (int code = 0; code < (1 << Mmax) && ok; code++) {
                const double a = ((double)code * 2.0) * 22.0;
                const double q0 = a * y7;
                const double q = fma(fma(-q0, 7.0, a), y7, q0);
                ok = q == a / 7.0;
            }
            ctx->fast_div_ok = ok;
        }
        return SCAN3D_OK;
    }();
    if (rc != SCAN3D_OK) {
        g_create_error = ctx->err;
        scan3d_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return SCAN3D_OK;
}

void scan3d_destroy(scan3d_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    void* ptrs[] = {ctx->cam_lut, ctx->proj_lut, ctx->atan_tab, ctx->nstep_w, ctx->wrapped[0], ctx->wrapped[1],
                    ctx->unwrapped[0], ctx->unwrapped[1], ctx->code[0], ctx->code[1], ctx->mask[0],
                    ctx->mask[1], ctx->valid, ctx->cpmap, ctx->xyz, ctx->pts, ctx->pix, ctx->rgb,
                    ctx->texture, ctx->d_count, ctx->block_counts, ctx->tile_state, ctx->sched_ctr, ctx->stage_pts, ctx->stage_vb, ctx->tile_flags, ctx->tile_list, ctx->trace, ctx->d_stack, ctx->d_roi, ctx->d_undist, ctx->roi_eff, ctx->roi_eff_h, ctx->roi_strict, ctx->pattern_profiles,
                    ctx->undist_xy[0], ctx->undist_xy[1], ctx->undist_frac[0], ctx->undist_frac[1],
                    ctx->mesh_idx, ctx->mesh_counts, ctx->mesh_totals, ctx->mesh_faces, ctx->mesh_normals,
                    ctx->vox.keys, ctx->vox.acc, ctx->vox.ordinal, ctx->vox.ord2slot, ctx->vox.state,
                    ctx->vox_point_slot, ctx->vox_flags, ctx->vox_xyz, ctx->vox_nrm, ctx->vox_rgb, ctx->vox_cnt};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int scan3d_set_stream(scan3d_ctx* ctx, void* cuda_stream)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return SCAN3D_OK;
}

int scan3d_sync(scan3d_ctx* ctx)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

int64_t scan3d_launch_count(const scan3d_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------
int scan3d_set_calibration(scan3d_ctx* ctx, const scan3d_calib* cal)
{
    if (!ctx || !cal) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    ctx->hcal = *cal;
    DeviceCalib& d = ctx->dcal;
    projection_matrix_host(cal->Kc, cal->rc, cal->tc, d.Ac);
    projection_matrix_host(cal->Kp, cal->rp, cal->tp, d.Ap);
    memcpy(d.Kc, cal->Kc, sizeof(d.Kc));
    memcpy(d.dc, cal->dc, sizeof(d.dc));
    memcpy(d.Kp, cal->Kp, sizeof(d.Kp));
    memcpy(d.dp, cal->dp, sizeof(d.dp));
    d.ifx_c = 1. / cal->Kc[0]; d.ify_c = 1. / cal->Kc[4];
    d.ifx_p = 1. / cal->Kp[0]; d.ify_p = 1. / cal->Kp[4];
    auto std_form = [](const double* K) {
        return K[1] == 0.0 && K[3] == 0.0 && K[6] == 0.0 && K[7] == 0.0 && K[8] == 1.0;
    };
    d.cam_std = std_form(cal->Kc);
    d.proj_std = std_form(cal->Kp);
    d.fast_div_ok = ctx->fast_div_ok ? 1 : 0;
    d.cam_distorted = d.proj_distorted = 0;
    for (int i = 0; i < 5; i++) {
        if (cal->dc[i] != 0.0) d.cam_distorted = 1;
        if (cal->dp[i] != 0.0) d.proj_distorted = 1;
    }
    if (ctx->cam_lut) { cudaFree(ctx->cam_lut); ctx->cam_lut = nullptr; }
    if (ctx->proj_lut) { cudaFree(ctx->proj_lut); ctx->proj_lut = nullptr; }
    for (int k = 0; k < 2; k++) {   // cv::undistort maps belong to the previous calibration
        if (ctx->undist_xy[k]) { cudaFree(ctx->undist_xy[k]); ctx->undist_xy[k] = nullptr; }
        if (ctx->undist_frac[k]) { cudaFree(ctx->undist_frac[k]); ctx->undist_frac[k] = nullptr; }
    }
    if (ctx->cfg.dirs == 2) {
        // a table also for an intrinsic matrix that is not [fx 0 cx; 0 fy cy; 0 0 1] (skew, ...): the kernels' table-free
        // route then only ever sees the standard form (4 operations per coordinate, no division)
        if (d.cam_distorted || !d.cam_std) {
            CK(dalloc(&ctx->cam_lut, npix(ctx)));
            CK(launch_undistort_lut(nullptr, d, false, ctx->cfg.W, ctx->cfg.H, ctx->cfg.row0, ctx->cam_lut, ctx->stream));
            ctx->launches++;
        }
        if (d.proj_distorted || !d.proj_std) {
            CK(dalloc(&ctx->proj_lut, (size_t)ctx->cfg.PW * ctx->cfg.PH));
            CK(launch_undistort_lut(nullptr, d, true, ctx->cfg.PW, ctx->cfg.PH, 0, ctx->proj_lut, ctx->stream));
            ctx->launches++;
        }
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->has_calib = true;
    return SCAN3D_OK;
}

int scan3d_get_projection_matrices(scan3d_ctx* ctx, double A_cam[12], double A_proj[12])
{
    if (!ctx || !ctx->has_calib) return fail(ctx, SCAN3D_ERR_STATE, "calibration not set");
    if (A_cam) memcpy(A_cam, ctx->dcal.Ac, 12 * sizeof(double));
    if (A_proj) memcpy(A_proj, ctx->dcal.Ap, 12 * sizeof(double));
    return SCAN3D_OK;
}

int scan3d_set_texture(scan3d_ctx* ctx, const uint8_t* bgr_host)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (!bgr_host) {
        if (ctx->texture) { cudaFree(ctx->texture); ctx->texture = nullptr; }
        return SCAN3D_OK;
    }
    if (!ctx->texture) CK(dalloc(&ctx->texture, 3 * npix(ctx)));
    if (!ctx->rgb) CK(dalloc(&ctx->rgb, 3 * npix(ctx)));
    CK(cudaMemcpyAsync(ctx->texture, bgr_host, 3 * npix(ctx), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

// ------------------------------------------------------------------------------------------
// stage entries
// ------------------------------------------------------------------------------------------
static int ensure_stage_planes(scan3d_ctx* ctx, int dir)
{
    const size_t n = npix(ctx);
    if (!ctx->wrapped[dir]) CK(dalloc(&ctx->wrapped[dir], n));
    if (!ctx->mask[dir]) CK(dalloc(&ctx->mask[dir], n));
    return SCAN3D_OK;
}

static inline float* points_of(const scan3d_ctx* ctx) { return ctx->pts_ext ? ctx->pts_ext : ctx->pts; }

// SCAN3D_FLAG_STRICT_REFERENCE: replace the caller's ROI by the plane check_I_mod_criteria derives from it as committed
static int strict_roi(scan3d_ctx* ctx, const uint8_t** roi_dev)
{
    if (!(ctx->cfg.flags & SCAN3D_FLAG_STRICT_REFERENCE)) return SCAN3D_OK;
    const size_t n = (size_t)ctx->cfg.W * ctx->cfg.H_total;
    if (!ctx->roi_strict) CK(dalloc(&ctx->roi_strict, n));
    CK(launch_strict_roi(*roi_dev, ctx->roi_strict, n, ctx->cfg.N, ctx->stream));
    ctx->launches++;
    *roi_dev = ctx->roi_strict;
    return SCAN3D_OK;
}

static int roi_bytes(const scan3d_ctx* ctx, size_t* out)
{
    *out = (size_t)ctx->cfg.W * ctx->cfg.H_total;
    return 0;
}

int scan3d_compute_wrapped_phase_dev(scan3d_ctx* ctx, int dir, const uint8_t* fringe_dev, const uint8_t* roi_dev)
{
    if (!ctx || !fringe_dev || !roi_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (dir < 0 || dir >= ctx->cfg.dirs) return fail(ctx, SCAN3D_ERR_ARG, "bad pattern_type");
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_stage_planes(ctx, dir);
    if (rc) return rc;
    const Shape s = shape_of(ctx->cfg);
    if (!ctx->in_reconstruct) {       // (scan3d_reconstruct_dev has already done it)
        rc = strict_roi(ctx, &roi_dev);
        if (rc) return rc;
    }
    if (ctx->cfg.flags & SCAN3D_FLAG_MODULATION_MASK) {
        if (!ctx->roi_eff) CK(dalloc(&ctx->roi_eff, npix(ctx)));
        CK(launch_modulation_roi(s, fringe_dev, roi_dev, ctx->roi_eff, ctx->stream));
        ctx->launches++;
        roi_dev = ctx->roi_eff;
    }
    CK(launch_wrapped(s, ctx->cfg.N, fringe_dev, roi_dev, ctx->wrapped[dir], ctx->atan_tab, ctx->nstep_w, false, ctx->stream));
    CK(launch_mask(s, roi_dev, ctx->mask[dir], ctx->stream));
    ctx->launches += 2;
    ctx->have_wrapped[dir] = true;
    ctx->have_unwrapped[dir] = false;
    ctx->have_cpmap = ctx->have_valid = ctx->have_xyz = ctx->have_points = ctx->have_mesh = false;
    return SCAN3D_OK;
}

// The host-pointer entries stage their inputs in the context's own buffers (allocated on first use, sized for a whole
// capture stack, kept until scan3d_destroy): no allocation or free per call.
static int ensure_staging(scan3d_ctx* ctx)
{
    const size_t sb = (size_t)scan3d_stack_bytes(&ctx->cfg);
    size_t rb;
    roi_bytes(ctx, &rb);
    if (!ctx->d_stack) CK(cudaMalloc((void**)&ctx->d_stack, sb));
    if (!ctx->d_roi) CK(cudaMalloc((void**)&ctx->d_roi, rb));
    return SCAN3D_OK;
}

int scan3d_compute_wrapped_phase(scan3d_ctx* ctx, int dir, const uint8_t* fringe_host, const uint8_t* roi_host)
{
    if (!ctx || !fringe_host || !roi_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    const size_t fb = (size_t)ctx->cfg.N * npix(ctx);
    size_t rb;
    roi_bytes(ctx, &rb);
    int rc = ensure_staging(ctx);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_stack, fringe_host, fb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_roi, roi_host, rb, cudaMemcpyHostToDevice, ctx->stream));
    rc = scan3d_compute_wrapped_phase_dev(ctx, dir, ctx->d_stack, ctx->d_roi);
    CK(cudaStreamSynchronize(ctx->stream));      // the caller may reuse its buffers, the next entry may restage
    return rc;
}

int scan3d_unwrap_phase_dev(scan3d_ctx* ctx, int dir, const uint8_t* gray_dev, const uint8_t* inv_dev)
{
    if (!ctx || !gray_dev || !inv_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (dir < 0 || dir >= ctx->cfg.dirs) return fail(ctx, SCAN3D_ERR_ARG, "bad pattern_type");
    if (!ctx->have_wrapped[dir]) return fail(ctx, SCAN3D_ERR_STATE, "unwrap_phase before compute_wrapped_phase");
    CK(cudaSetDevice(ctx->device));
    const Shape s = shape_of(ctx->cfg);
    const int M = dir == 0 ? ctx->cfg.M_v : ctx->cfg.M_h;
    CK(launch_unwrap(s, dir, M, gray_dev, inv_dev, ctx->wrapped[dir], ctx->mask[dir], ctx->code[dir],
                     ctx->unwrapped[dir], ctx->stream));
    ctx->launches++;
    ctx->have_unwrapped[dir] = true;
    ctx->have_cpmap = ctx->have_valid = ctx->have_xyz = ctx->have_points = ctx->have_mesh = false;
    return SCAN3D_OK;
}

int scan3d_unwrap_phase(scan3d_ctx* ctx, int dir, const uint8_t* gray_host, const uint8_t* inv_host)
{
    if (!ctx || !gray_host || !inv_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (dir < 0 || dir >= ctx->cfg.dirs) return fail(ctx, SCAN3D_ERR_ARG, "bad pattern_type");
    CK(cudaSetDevice(ctx->device));
    const int M = dir == 0 ? ctx->cfg.M_v : ctx->cfg.M_h;
    const size_t b = (size_t)M * npix(ctx);
    int rc = ensure_staging(ctx);                // 2 M frames <= the stack's dirs * (N + 2 M)
    if (rc) return rc;
    uint8_t* d = ctx->d_stack;
    CK(cudaMemcpyAsync(d, gray_host, b, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d + b, inv_host, b, cudaMemcpyHostToDevice, ctx->stream));
    rc = scan3d_unwrap_phase_dev(ctx, dir, d, d + b);
    CK(cudaStreamSynchronize(ctx->stream));
    return rc;
}

int scan3d_compute_c_p_map(scan3d_ctx* ctx)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (ctx->cfg.dirs != 2) return fail(ctx, SCAN3D_ERR_STATE, "compute_c_p_map needs both directions");
    if (!ctx->have_unwrapped[0] || !ctx->have_unwrapped[1]) return fail(ctx, SCAN3D_ERR_STATE, "compute_c_p_map before unwrap_phase(0) and (1)");
    CK(cudaSetDevice(ctx->device));
    const Shape s = shape_of(ctx->cfg);
    CK(launch_cpmap(s, ctx->cfg.fw_v, ctx->cfg.fw_h, ctx->unwrapped[0], ctx->unwrapped[1], ctx->mask[0],
                    ctx->mask[1], ctx->cpmap, ctx->valid, ctx->stream));
    ctx->launches++;
    ctx->have_cpmap = ctx->have_valid = true;
    ctx->have_xyz = ctx->have_points = ctx->have_mesh = false;
    return SCAN3D_OK;
}

int scan3d_triangulate(scan3d_ctx* ctx)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->has_calib) return fail(ctx, SCAN3D_ERR_STATE, "triangulate before set_calibration");
    if (!ctx->have_cpmap) return fail(ctx, SCAN3D_ERR_STATE, "triangulate before compute_c_p_map");
    CK(cudaSetDevice(ctx->device));
    if (!ctx->xyz) CK(dalloc(&ctx->xyz, 3 * npix(ctx)));
    const Shape s = shape_of(ctx->cfg);
    CK(launch_triangulate(s, ctx->dcal, ctx->cam_lut, ctx->proj_lut, ctx->cpmap, ctx->valid, ctx->xyz, ctx->stream));
    ctx->launches++;
    ctx->have_xyz = true;
    ctx->have_points = ctx->have_mesh = false;
    return SCAN3D_OK;
}

int scan3d_compact_points(scan3d_ctx* ctx, int64_t* count_out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->have_xyz) return fail(ctx, SCAN3D_ERR_STATE, "compact_points before triangulate");
    CK(cudaSetDevice(ctx->device));
    const size_t n = npix(ctx);
    if (!ctx->block_counts) CK(dalloc(&ctx->block_counts, (n + 1023) / 1024 + 1));
    if (!ctx->pix) CK(dalloc(&ctx->pix, n));
    if (ctx->texture && !ctx->rgb) CK(dalloc(&ctx->rgb, 3 * n));
    const Shape s = shape_of(ctx->cfg);
    int nl = 0;
    CK(launch_compact(s, ctx->xyz, ctx->valid, ctx->texture, ctx->block_counts, points_of(ctx), ctx->pix,
                      ctx->texture ? ctx->rgb : nullptr, ctx->d_count, ctx->stream, &nl));
    ctx->launches += nl;
    ctx->have_points = true;
    ctx->have_mesh = false;
    if (count_out) return scan3d_point_count(ctx, count_out);
    return SCAN3D_OK;
}

// ------------------------------------------------------------------------------------------
// fused entry
// ------------------------------------------------------------------------------------------
static int reconstruct_stagewise(scan3d_ctx* ctx, const uint8_t* stack, const uint8_t* roi)
{
    // shape-generic route: the same stage kernels, chained (used when the single-pass kernel
    // does not support the shape: W % 16 != 0, generic N, or a stack too large for shared memory)
    const size_t n = npix(ctx);
    const scan3d_config& c = ctx->cfg;
    const uint8_t* p = stack;
    for (int d = 0; d < c.dirs; d++) {
        const int M = d == 0 ? c.M_v : c.M_h;
        int rc = scan3d_compute_wrapped_phase_dev(ctx, d, p, roi);
        if (rc) return rc;
        p += (size_t)c.N * n;
        rc = scan3d_unwrap_phase_dev(ctx, d, p, p + (size_t)M * n);
        if (rc) return rc;
        p += 2 * (size_t)M * n;
    }
    if (c.dirs == 1) {
        CK(cudaMemcpyAsync(ctx->valid, ctx->mask[0], n, cudaMemcpyDeviceToDevice, ctx->stream));
        ctx->have_valid = true;
        return SCAN3D_OK;
    }
    int rc = scan3d_compute_c_p_map(ctx);
    if (rc) return rc;
    rc = scan3d_triangulate(ctx);
    if (rc) return rc;
    rc = scan3d_compact_points(ctx, nullptr);
    if (rc || !ctx->reg_on) return rc;
    // scan3d_set_registration on the shape-generic route: the same transform over the compacted points, in place
    // (all n = W*H slots: the count stays on the device; slots past it hold stale floats nobody reads)
    CK(launch_register_points(points_of(ctx), points_of(ctx), (long long)n, ctx->reg_R, ctx->reg_t[0], ctx->reg_t[1], ctx->reg_t[2],
                              ctx->sm_count, ctx->stream));
    ctx->launches++;
    return SCAN3D_OK;
}

int scan3d_reconstruct_dev(scan3d_ctx* ctx, const uint8_t* stack_dev, const uint8_t* roi_dev)
{
    if (!ctx || !stack_dev || !roi_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (ctx->cfg.dirs == 2 && !ctx->has_calib) return fail(ctx, SCAN3D_ERR_STATE, "reconstruct before set_calibration");
    CK(cudaSetDevice(ctx->device));
    ctx->have_mesh = false;
    {
        const int rc = strict_roi(ctx, &roi_dev);
        if (rc) return rc;
    }
    if (!ctx->fast_div_ok || !fused7_supported(ctx->cfg)) {
        ctx->in_reconstruct = true;
        const int rc = reconstruct_stagewise(ctx, stack_dev, roi_dev);
        ctx->in_reconstruct = false;
        return rc;
    }
    const scan3d_config& c = ctx->cfg;
    FusedArgs a{};
    a.stack = stack_dev; a.roi = roi_dev;
    if (c.flags & SCAN3D_FLAG_MODULATION_MASK) {
        // check_I_mod_criteria's modulation criterion (3/wrapped_phase.cpp:84-104): one effective ROI plane per
        // direction from that direction's three fringe images (a pre-pass: the mask recurrence needs it two rows up)
        const Shape s = shape_of(c);
        const size_t n = npix(ctx);
        if (!ctx->roi_eff) CK(dalloc(&ctx->roi_eff, n));
        CK(launch_modulation_roi(s, stack_dev, roi_dev, ctx->roi_eff, ctx->stream));
        ctx->launches++;
        a.roi = ctx->roi_eff;
        a.roi2 = ctx->roi_eff;
        a.roi_list = roi_dev;
        if (c.dirs == 2) {
            if (!ctx->roi_eff_h) CK(dalloc(&ctx->roi_eff_h, n));
            CK(launch_modulation_roi(s, stack_dev + (size_t)(c.N + 2 * c.M_v) * n, roi_dev, ctx->roi_eff_h, ctx->stream));
            ctx->launches++;
            a.roi2 = ctx->roi_eff_h;
        }
    }
    a.unw_v = ctx->unwrapped[0]; a.unw_h = ctx->unwrapped[1];
    a.code_v = ctx->code[0]; a.code_h = ctx->code[1];
    a.valid = ctx->valid; a.cpmap = ctx->cpmap;
    a.pts = points_of(ctx); a.pix = ctx->pix;
    a.rgb = ctx->texture ? ctx->rgb : nullptr; a.texture = ctx->texture;
    a.d_count = ctx->d_count; a.tile_state = ctx->tile_state; a.trace = ctx->trace; a.tile_flags = ctx->tile_flags; a.tile_list = ctx->tile_list + 1; a.n_list = ctx->tile_list;
    a.cam_lut = ctx->cam_lut; a.proj_lut = ctx->proj_lut; a.atan_tab = ctx->atan_tab;
    if (ctx->trace) CK(cudaMemsetAsync(ctx->trace, 0, (size_t)1024 * 64 * 8 * 8, ctx->stream));   // diagnostics only
    a.epoch = ++ctx->epoch;
    if ((ctx->epoch & 0x3fffffffu) == 0) {   // epoch wrapped: clear the look-back words once
        CK(cudaMemsetAsync(ctx->tile_state, 0, ((size_t)fused_num_tiles(c) + 1) * 8, ctx->stream));
        a.epoch = ++ctx->epoch;
    }
    a.tmap_cache = &ctx->tmaps;
    a.ctas_per_sm = ctx->cta_limit;
    const bool fold_reg = ctx->reg_on && fused7_folds_registration(c);
    a.reg_on = fold_reg ? 1 : 0;
    memcpy(a.reg_R, ctx->reg_R, sizeof(a.reg_R));
    memcpy(a.reg_t, ctx->reg_t, sizeof(a.reg_t));
    a.W = c.W; a.H = c.H; a.row0 = c.row0; a.H_total = c.H_total; a.PW = c.PW; a.PH = c.PH;
    a.N = c.N; a.M_v = c.M_v; a.M_h = c.M_h; a.fw_v = c.fw_v; a.fw_h = c.fw_h;
    a.fw_v_d = (double)c.fw_v; a.fw_h_d = (double)c.fw_h;
#if S3D_BUILD_V8
    static const int impl = getenv("SCAN3D_FUSED_IMPL") ? atoi(getenv("SCAN3D_FUSED_IMPL")) : 7;
    if (impl >= 8 && fused8_supported(c)) {
        a.sched_ctr = ctx->sched_ctr;
        a.pos_base = ctx->sched_base;
        if (c.dirs == 2 && !ctx->stage_pts) {
            CK(dalloc(&ctx->stage_pts, fused8_stage_floats(ctx->sm_count)));
            CK(dalloc(&ctx->stage_vb, fused8_stage_vb_words(ctx->sm_count)));
        }
        a.stage_pts = ctx->stage_pts;
        a.stage_vb = ctx->stage_vb;
        uint32_t advance = 0;
        CK(launch_fused8(c, a, ctx->dcal, ctx->sm_count, &ctx->tmaps, &advance, ctx->stream));
        ctx->sched_base += advance;
        ctx->launches += 1;   // the one persistent kernel
    } else
#endif
    {
        CK(launch_fused7(c, a, ctx->dcal, ctx->sm_count, ctx->stream));
        ctx->launches += 3;   // work-list flags, work-list scan, persistent fused kernel
    }
    if (ctx->reg_on && !fold_reg && c.dirs == 2) {
        // shapes without the folding variant: the same transform as one more pass over the compacted points
        CK(launch_register_points(points_of(ctx), points_of(ctx), (long long)npix(ctx), ctx->reg_R, ctx->reg_t[0], ctx->reg_t[1],
                                  ctx->reg_t[2], ctx->sm_count, ctx->stream));
        ctx->launches++;
    }
    ctx->have_wrapped[0] = ctx->have_wrapped[1] = false;
    ctx->have_unwrapped[0] = true;
    ctx->have_unwrapped[1] = c.dirs == 2;
    ctx->have_cpmap = c.dirs == 2;
    ctx->have_valid = true;
    ctx->have_xyz = false;
    ctx->have_points = c.dirs == 2;
    ctx->have_mesh = false;
    return SCAN3D_OK;
}

int scan3d_reconstruct(scan3d_ctx* ctx, const uint8_t* stack_host, const uint8_t* roi_host, int64_t* count_out)
{
    if (!ctx || !stack_host || !roi_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    const size_t sb = (size_t)scan3d_stack_bytes(&ctx->cfg);
    size_t rb;
    roi_bytes(ctx, &rb);
    if (int rs = ensure_staging(ctx)) return rs;
    CK(cudaMemcpyAsync(ctx->d_stack, stack_host, sb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_roi, roi_host, rb, cudaMemcpyHostToDevice, ctx->stream));
    int rc = scan3d_reconstruct_dev(ctx, ctx->d_stack, ctx->d_roi);
    if (rc) return rc;
    if (count_out) {
        if (ctx->cfg.dirs == 2) return scan3d_point_count(ctx, count_out);
        *count_out = 0;
    }
    return scan3d_sync(ctx);
}

int scan3d_set_cta_limit(scan3d_ctx* ctx, int ctas_per_sm)
{
    if (!ctx || ctas_per_sm < 0) return SCAN3D_ERR_ARG;
    ctx->cta_limit = ctas_per_sm;
    return SCAN3D_OK;
}

int scan3d_set_registration(scan3d_ctx* ctx, int enable, float theta_deg, float tx, float ty, float tz)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (ctx->cfg.dirs != 2) return fail(ctx, SCAN3D_ERR_STATE, "no point cloud in a one-direction configuration");
    ctx->reg_on = enable != 0;
    if (ctx->reg_on) {
        s3a::register_rotation(theta_deg, ctx->reg_R);
        ctx->reg_t[0] = tx; ctx->reg_t[1] = ty; ctx->reg_t[2] = tz;
    }
    return SCAN3D_OK;
}

int scan3d_reconstruct_raw_dev(scan3d_ctx* ctx, const uint8_t* raw_stack_dev, const uint8_t* roi_dev)
{
    if (!ctx || !raw_stack_dev || !roi_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    const size_t sb = (size_t)scan3d_stack_bytes(&ctx->cfg);
    if (!ctx->d_undist) CK(cudaMalloc((void**)&ctx->d_undist, sb));
    const int frames = (int)(sb / npix(ctx));
    int rc = scan3d_undistort_frames_dev(ctx, 0, raw_stack_dev, frames, ctx->d_undist);      // 2/project_pattern.cpp:220,234
    if (rc) return rc;
    return scan3d_reconstruct_dev(ctx, ctx->d_undist, roi_dev);
}

int scan3d_reconstruct_raw(scan3d_ctx* ctx, const uint8_t* raw_stack_host, const uint8_t* roi_host, int64_t* count_out)
{
    if (!ctx || !raw_stack_host || !roi_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    const size_t sb = (size_t)scan3d_stack_bytes(&ctx->cfg);
    size_t rb;
    roi_bytes(ctx, &rb);
    if (int rs = ensure_staging(ctx)) return rs;
    CK(cudaMemcpyAsync(ctx->d_stack, raw_stack_host, sb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_roi, roi_host, rb, cudaMemcpyHostToDevice, ctx->stream));
    int rc = scan3d_reconstruct_raw_dev(ctx, ctx->d_stack, ctx->d_roi);
    if (rc) return rc;
    if (count_out) {
        if (ctx->cfg.dirs == 2) return scan3d_point_count(ctx, count_out);
        *count_out = 0;
    }
    return scan3d_sync(ctx);
}

// ------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------
static void* plane_ptr(scan3d_ctx* ctx, int plane, size_t* elt)
{
    switch (plane) {
        case SCAN3D_PLANE_WRAPPED_V: *elt = 4; return ctx->wrapped[0];
        case SCAN3D_PLANE_WRAPPED_H: *elt = 4; return ctx->wrapped[1];
        case SCAN3D_PLANE_UNWRAPPED_V: *elt = 4; return ctx->unwrapped[0];
        case SCAN3D_PLANE_UNWRAPPED_H: *elt = 4; return ctx->unwrapped[1];
        case SCAN3D_PLANE_CODE_V: *elt = 2; return ctx->code[0];
        case SCAN3D_PLANE_CODE_H: *elt = 2; return ctx->code[1];
        case SCAN3D_PLANE_MASK: *elt = 1; return ctx->mask[0];
        case S3D_PLANE_MASK_H: *elt = 1; return ctx->mask[1];
        case SCAN3D_PLANE_VALID: *elt = 1; return ctx->valid;
        case SCAN3D_PLANE_CPMAP: *elt = 8; return ctx->cpmap;
        case SCAN3D_PLANE_XYZ: *elt = 24; return ctx->xyz;
        default: *elt = 0; return nullptr;
    }
}

// has the plane been produced by a compute entry since the context was created / the inputs last changed?
static bool plane_ready(const scan3d_ctx* ctx, int plane)
{
    switch (plane) {
        case SCAN3D_PLANE_WRAPPED_V: case SCAN3D_PLANE_MASK: return ctx->have_wrapped[0];
        case SCAN3D_PLANE_WRAPPED_H: case S3D_PLANE_MASK_H: return ctx->have_wrapped[1];
        case SCAN3D_PLANE_UNWRAPPED_V: case SCAN3D_PLANE_CODE_V: return ctx->have_unwrapped[0];
        case SCAN3D_PLANE_UNWRAPPED_H: case SCAN3D_PLANE_CODE_H: return ctx->have_unwrapped[1];
        case SCAN3D_PLANE_VALID: return ctx->have_valid;
        case SCAN3D_PLANE_CPMAP: return ctx->have_cpmap;
        case SCAN3D_PLANE_XYZ: return ctx->have_xyz;
        default: return false;
    }
}

int64_t scan3d_plane_bytes(const scan3d_ctx* ctx, int plane)
{
    if (!ctx) return 0;
    size_t elt = 0;
    plane_ptr(const_cast<scan3d_ctx*>(ctx), plane, &elt);
    return (int64_t)(elt * npix(ctx));
}

void* scan3d_device_plane(scan3d_ctx* ctx, int plane)
{
    if (!ctx || !plane_ready(ctx, plane)) return nullptr;     // (a plane nothing has written is not handed out)
    size_t elt;
    return plane_ptr(ctx, plane, &elt);
}

int scan3d_get_plane(scan3d_ctx* ctx, int plane, void* dst_host)
{
    if (!ctx || !dst_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    size_t elt;
    void* src = plane_ptr(ctx, plane, &elt);
    if (!src || !plane_ready(ctx, plane))
        return fail(ctx, SCAN3D_ERR_STATE, "plane not available: no compute entry has produced it (the single-pass entry "
                                           "keeps wrapped phases and per-direction masks in registers)");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dst_host, src, elt * npix(ctx), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

int scan3d_get_code_i32(scan3d_ctx* ctx, int dir, int32_t* dst_host)
{
    if (!ctx || !dst_host || dir < 0 || dir >= ctx->cfg.dirs) return fail(ctx, SCAN3D_ERR_ARG, "bad argument");
    std::vector<int16_t> tmp(npix(ctx));
    int rc = scan3d_get_plane(ctx, dir == 0 ? SCAN3D_PLANE_CODE_V : SCAN3D_PLANE_CODE_H, tmp.data());
    if (rc) return rc;
    for (size_t i = 0; i < tmp.size(); i++) dst_host[i] = tmp[i];
    return SCAN3D_OK;
}

int scan3d_get_cpmap_i64(scan3d_ctx* ctx, int64_t* dst_host)
{
    if (!ctx || !dst_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    std::vector<int32_t> tmp(2 * npix(ctx));
    int rc = scan3d_get_plane(ctx, SCAN3D_PLANE_CPMAP, tmp.data());
    if (rc) return rc;
    for (size_t i = 0; i < tmp.size(); i++) dst_host[i] = tmp[i];
    return SCAN3D_OK;
}

int scan3d_point_count(scan3d_ctx* ctx, int64_t* count_out)
{
    if (!ctx || !count_out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!ctx->have_points) return fail(ctx, SCAN3D_ERR_STATE, "no compacted points yet");
    CK(cudaSetDevice(ctx->device));
    uint32_t c = 0;
    CK(cudaMemcpyAsync(&c, ctx->d_count, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *count_out = c;
    return SCAN3D_OK;
}

int scan3d_get_points(scan3d_ctx* ctx, float* xyz_host, uint32_t* pix_host, uint8_t* rgb_host, int64_t max_points)
{
    int64_t n = 0;
    int rc = scan3d_point_count(ctx, &n);
    if (rc) return rc;
    if (n > max_points) n = max_points;
    if (n <= 0) return SCAN3D_OK;
    if (xyz_host) CK(cudaMemcpyAsync(xyz_host, points_of(ctx), (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    if (pix_host) {
        if (!ctx->pix) return fail(ctx, SCAN3D_ERR_STATE, "pixel indices were not produced (stage API or SCAN3D point-pixel flag)");
        CK(cudaMemcpyAsync(pix_host, ctx->pix, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (rgb_host) {
        if (ctx->rgb && ctx->texture) CK(cudaMemcpyAsync(rgb_host, ctx->rgb, (size_t)n * 3, cudaMemcpyDeviceToHost, ctx->stream));
        else memset(rgb_host, 0, (size_t)n * 3);
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

void* scan3d_device_points(scan3d_ctx* ctx) { return ctx ? points_of(ctx) : nullptr; }

static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");

int scan3d_peer_alloc(int device, int64_t bytes, void** dev_ptr, uint8_t handle_out[64])
{
    if (!dev_ptr || !handle_out || bytes <= 0) return SCAN3D_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return SCAN3D_ERR_CUDA;
    void* p = nullptr;
    if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); return SCAN3D_ERR_CUDA; }
    cudaIpcMemHandle_t h;
    if (cudaIpcGetMemHandle(&h, p) != cudaSuccess) { cudaGetLastError(); cudaFree(p); return SCAN3D_ERR_CUDA; }
    memcpy(handle_out, &h, 64);
    *dev_ptr = p;
    return SCAN3D_OK;
}

int scan3d_peer_free(int device, void* dev_ptr)
{
    if (cudaSetDevice(device) != cudaSuccess) return SCAN3D_ERR_CUDA;
    return cudaFree(dev_ptr) == cudaSuccess ? SCAN3D_OK : SCAN3D_ERR_CUDA;
}

int scan3d_peer_open(int device, const uint8_t handle[64], void** dev_ptr)
{
    if (!dev_ptr || !handle) return SCAN3D_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return SCAN3D_ERR_CUDA;     // the ACCESSING device: lazy peer access is set up for it
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void* p = nullptr;
    if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return SCAN3D_ERR_CUDA; }
    *dev_ptr = p;
    return SCAN3D_OK;
}

int scan3d_peer_close(int device, void* dev_ptr)
{
    if (cudaSetDevice(device) != cudaSuccess) return SCAN3D_ERR_CUDA;
    return cudaIpcCloseMemHandle(dev_ptr) == cudaSuccess ? SCAN3D_OK : SCAN3D_ERR_CUDA;
}

int scan3d_set_points_buffer(scan3d_ctx* ctx, void* points_dev, int64_t capacity_points)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (ctx->cfg.dirs != 2) return fail(ctx, SCAN3D_ERR_STATE, "no point cloud in a one-direction configuration");
    if (points_dev && capacity_points < (int64_t)npix(ctx)) return fail(ctx, SCAN3D_ERR_ARG, "points buffer smaller than W*H points");
    if (points_dev && ((uintptr_t)points_dev & 15)) return fail(ctx, SCAN3D_ERR_ARG, "points buffer must be 16-byte aligned");
    if (points_dev) {
        // memory of another GPU (mapped through CUDA IPC, or allocated there by this process):
        // kernels of this context's device need peer access to it
        CK(cudaSetDevice(ctx->device));
        cudaPointerAttributes attr;
        CK(cudaPointerGetAttributes(&attr, points_dev));
        if (attr.type != cudaMemoryTypeDevice) return fail(ctx, SCAN3D_ERR_ARG, "points buffer is not device memory");
        if (attr.device != ctx->device) {
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, ctx->device, attr.device));
            if (!can) return fail(ctx, SCAN3D_ERR_ARG, "no peer access from this context's GPU to the points buffer's GPU");
            const cudaError_t e = cudaDeviceEnablePeerAccess(attr.device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (e != cudaSuccess) return fail(ctx, SCAN3D_ERR_CUDA, cudaGetErrorString(e));
        }
    }
    ctx->pts_ext = (float*)points_dev;
    ctx->have_points = ctx->have_mesh = false;
    return SCAN3D_OK;
}
void* scan3d_device_point_pixels(scan3d_ctx* ctx) { return ctx ? ctx->pix : nullptr; }
void* scan3d_device_point_count(scan3d_ctx* ctx) { return ctx ? ctx->d_count : nullptr; }

// pcl::io::savePLYFile-style vertex list (8/save_point_cloud.cpp:216-217)
int scan3d_write_ply(scan3d_ctx* ctx, const char* path, int binary)
{
    if (!ctx || !path) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    int64_t n = 0;
    int rc = scan3d_point_count(ctx, &n);
    if (rc) return rc;
    std::vector<float> xyz((size_t)n * 3);
    std::vector<uint8_t> rgb((size_t)n * 3);
    rc = scan3d_get_points(ctx, xyz.data(), nullptr, rgb.data(), n);
    if (rc) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ctx, SCAN3D_ERR_IO, "cannot open PLY for writing");
    fprintf(f, "ply\nformat %s 1.0\ncomment scan3d-b200\nelement vertex %lld\n"
               "property float x\nproperty float y\nproperty float z\n"
               "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n",
            binary ? "binary_little_endian" : "ascii", (long long)n);
    if (binary) {
        std::vector<uint8_t> rec((size_t)n * 15);
        for (int64_t i = 0; i < n; i++) {
            memcpy(&rec[(size_t)i * 15], &xyz[(size_t)i * 3], 12);
            memcpy(&rec[(size_t)i * 15 + 12], &rgb[(size_t)i * 3], 3);
        }
        fwrite(rec.data(), 1, rec.size(), f);
    } else {
        for (int64_t i = 0; i < n; i++)
            fprintf(f, "%.9g %.9g %.9g %u %u %u\n", xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2],
                    rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2]);
    }
    const bool ok = fclose(f) == 0;
    return ok ? SCAN3D_OK : fail(ctx, SCAN3D_ERR_IO, "PLY write failed");
}

// The vertex element "x y z nx ny nz red green blue" of scan3d_write_mesh_ply and scan3d_write_voxel_ply: the header
// (extra_header, e.g. a face element, goes before end_header) and the n vertex records, ascii (%.9g) or binary.
static void write_ply_with_normals(FILE* f, int binary, int64_t n, const float* xyz, const float* nrm, const uint8_t* rgb,
                                   const char* extra_header)
{
    fprintf(f, "ply\nformat %s 1.0\ncomment scan3d-b200\nelement vertex %lld\n"
               "property float x\nproperty float y\nproperty float z\n"
               "property float nx\nproperty float ny\nproperty float nz\n"
               "property uchar red\nproperty uchar green\nproperty uchar blue\n%send_header\n",
            binary ? "binary_little_endian" : "ascii", (long long)n, extra_header);
    if (binary) {
        std::vector<uint8_t> rec((size_t)n * 27);
        for (int64_t i = 0; i < n; i++) {
            memcpy(&rec[(size_t)i * 27], &xyz[(size_t)i * 3], 12);
            memcpy(&rec[(size_t)i * 27 + 12], &nrm[(size_t)i * 3], 12);
            memcpy(&rec[(size_t)i * 27 + 24], &rgb[(size_t)i * 3], 3);
        }
        fwrite(rec.data(), 1, rec.size(), f);
    } else {
        for (int64_t i = 0; i < n; i++)
            fprintf(f, "%.9g %.9g %.9g %.9g %.9g %.9g %u %u %u\n", xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], nrm[3 * i],
                    nrm[3 * i + 1], nrm[3 * i + 2], rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2]);
    }
}

// ------------------------------------------------------------------------------------------
// camera-grid mesh of the compacted points (common/scan3d_mesh_math.h has the exact rules)
// ------------------------------------------------------------------------------------------
int scan3d_build_mesh(scan3d_ctx* ctx, float max_edge)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    const scan3d_config& c = ctx->cfg;
    if (c.dirs != 2) return fail(ctx, SCAN3D_ERR_STATE, "no point cloud in a one-direction configuration");
    if (c.row0 != 0 || c.H_total != c.H)
        return fail(ctx, SCAN3D_ERR_CONFIG, "the mesh needs the whole frame (a shard's last cell row needs the next shard's first row)");
    if ((int64_t)c.W * c.H >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_CONFIG, "W*H must be below 2^31 (int32 point indices)");
    if (!(max_edge > 0.0f)) return fail(ctx, SCAN3D_ERR_ARG, "max_edge must be > 0 (+inf: no length limit)");
    if (!ctx->have_points) return fail(ctx, SCAN3D_ERR_STATE, "build_mesh before the points are computed");
    CK(cudaSetDevice(ctx->device));
    const size_t n = npix(ctx);
    const size_t nb = (n + POINT_BLOCK - 1) / POINT_BLOCK;
    const size_t max_faces = 2 * (size_t)(c.W - 1) * (size_t)(c.H - 1);
    if (!ctx->block_counts) CK(dalloc(&ctx->block_counts, nb + 1));
    if (!ctx->mesh_idx) CK(dalloc(&ctx->mesh_idx, n));
    if (!ctx->mesh_counts) CK(dalloc(&ctx->mesh_counts, nb));
    if (!ctx->mesh_totals) CK(dalloc(&ctx->mesh_totals, 2));
    if (!ctx->mesh_faces) CK(dalloc(&ctx->mesh_faces, 3 * std::max(max_faces, (size_t)1)));
    if (!ctx->mesh_normals) CK(dalloc(&ctx->mesh_normals, 3 * n));
    CK(launch_mesh(ctx->valid, points_of(ctx), c.W, c.H, max_edge, ctx->mesh_idx, ctx->block_counts, ctx->mesh_counts,
                   ctx->mesh_totals, ctx->mesh_faces, ctx->mesh_normals, ctx->stream));
    ctx->launches += MESH_LAUNCHES;
    ctx->have_mesh = true;
    return SCAN3D_OK;
}

int scan3d_mesh_face_count(scan3d_ctx* ctx, int64_t* count_out)
{
    if (!ctx || !count_out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!ctx->have_mesh) return fail(ctx, SCAN3D_ERR_STATE, "no mesh of the current points: call scan3d_build_mesh");
    CK(cudaSetDevice(ctx->device));
    uint32_t nf = 0;
    CK(cudaMemcpyAsync(&nf, ctx->mesh_totals + 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *count_out = nf;
    return SCAN3D_OK;
}

int scan3d_get_mesh(scan3d_ctx* ctx, int32_t* faces_host, float* normals_host, int64_t max_faces)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    int64_t nf = 0, np = 0;
    int rc = scan3d_mesh_face_count(ctx, &nf);
    if (rc) return rc;
    rc = scan3d_point_count(ctx, &np);
    if (rc) return rc;
    if (nf > max_faces) nf = max_faces;
    if (faces_host && nf > 0)
        CK(cudaMemcpyAsync(faces_host, ctx->mesh_faces, (size_t)nf * 12, cudaMemcpyDeviceToHost, ctx->stream));
    if (normals_host && np > 0)
        CK(cudaMemcpyAsync(normals_host, ctx->mesh_normals, (size_t)np * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

void* scan3d_device_mesh_faces(scan3d_ctx* ctx) { return ctx && ctx->have_mesh ? ctx->mesh_faces : nullptr; }
void* scan3d_device_point_normals(scan3d_ctx* ctx) { return ctx && ctx->have_mesh ? ctx->mesh_normals : nullptr; }

int scan3d_write_mesh_ply(scan3d_ctx* ctx, const char* path, int binary)
{
    if (!ctx || !path) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    int64_t np = 0, nf = 0;
    int rc = scan3d_mesh_face_count(ctx, &nf);
    if (rc) return rc;
    rc = scan3d_point_count(ctx, &np);
    if (rc) return rc;
    std::vector<float> xyz((size_t)np * 3), nrm((size_t)np * 3);
    std::vector<uint8_t> rgb((size_t)np * 3);
    std::vector<int32_t> faces((size_t)nf * 3);
    rc = scan3d_get_points(ctx, xyz.data(), nullptr, rgb.data(), np);
    if (rc) return rc;
    rc = scan3d_get_mesh(ctx, faces.data(), nrm.data(), nf);
    if (rc) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ctx, SCAN3D_ERR_IO, "cannot open PLY for writing");
    char face_header[96];
    snprintf(face_header, sizeof(face_header), "element face %lld\nproperty list uchar int vertex_indices\n", (long long)nf);
    write_ply_with_normals(f, binary, np, xyz.data(), nrm.data(), rgb.data(), face_header);
    if (binary) {
        std::vector<uint8_t> frec((size_t)nf * 13);
        for (int64_t i = 0; i < nf; i++) {
            frec[(size_t)i * 13] = 3;
            memcpy(&frec[(size_t)i * 13 + 1], &faces[(size_t)i * 3], 12);
        }
        fwrite(frec.data(), 1, frec.size(), f);
    } else {
        for (int64_t i = 0; i < nf; i++) fprintf(f, "3 %d %d %d\n", faces[3 * i], faces[3 * i + 1], faces[3 * i + 2]);
    }
    const bool ok = fclose(f) == 0;
    return ok ? SCAN3D_OK : fail(ctx, SCAN3D_ERR_IO, "PLY write failed");
}

// ------------------------------------------------------------------------------------------
// voxel-grid merge of registered views (include/scan3d.h and common/scan3d_voxel_math.h have the exact rules)
// ------------------------------------------------------------------------------------------
static void free_ptr(void* p)
{
    if (p) cudaFree(p);
}

int scan3d_voxel_begin(scan3d_ctx* ctx, float voxel_size, int64_t max_voxels)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!(voxel_size > 0.0f && voxel_size - voxel_size == 0.0f))
        return fail(ctx, SCAN3D_ERR_ARG, "voxel_size must be finite and > 0");
    if (max_voxels < 1 || max_voxels >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_ARG, "max_voxels must be in [1, 2^31)");
    CK(cudaSetDevice(ctx->device));
    ctx->vox_begun = ctx->vox_fresh = false;
    VoxelTable& t = ctx->vox;
    const uint32_t cap = voxel_table_capacity((uint32_t)max_voxels, ctx->sm_count);
    if (cap > ctx->vox_alloc_cap) {
        free_ptr(t.keys); free_ptr(t.acc); free_ptr(t.ordinal);
        t.keys = nullptr; t.acc = nullptr; t.ordinal = nullptr;
        ctx->vox_alloc_cap = 0;
        CK(dalloc(&t.keys, cap));
        CK(dalloc(&t.acc, cap));
        CK(dalloc(&t.ordinal, cap));
        ctx->vox_alloc_cap = cap;
    }
    if ((uint32_t)max_voxels > ctx->vox_alloc_max) {
        free_ptr(t.ord2slot); free_ptr(ctx->vox_xyz); free_ptr(ctx->vox_nrm); free_ptr(ctx->vox_rgb); free_ptr(ctx->vox_cnt);
        t.ord2slot = nullptr; ctx->vox_xyz = ctx->vox_nrm = nullptr; ctx->vox_rgb = nullptr; ctx->vox_cnt = nullptr;
        ctx->vox_alloc_max = 0;
        const size_t m = (size_t)max_voxels;
        CK(dalloc(&t.ord2slot, m));
        CK(dalloc(&ctx->vox_xyz, 3 * m));
        CK(dalloc(&ctx->vox_nrm, 3 * m));
        CK(dalloc(&ctx->vox_rgb, 3 * m));
        CK(dalloc(&ctx->vox_cnt, m));
        ctx->vox_alloc_max = (uint32_t)max_voxels;
    }
    const size_t n = npix(ctx);
    if (!t.state) CK(dalloc(&t.state, 1));
    if (!ctx->vox_point_slot) CK(dalloc(&ctx->vox_point_slot, n));
    if (!ctx->vox_flags) CK(dalloc(&ctx->vox_flags, n));
    if (!ctx->block_counts) CK(dalloc(&ctx->block_counts, (n + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    CK(cudaMemsetAsync(t.keys, 0xff, (size_t)cap * sizeof(*t.keys), ctx->stream));
    CK(cudaMemsetAsync(t.acc, 0, (size_t)cap * sizeof(*t.acc), ctx->stream));
    CK(cudaMemsetAsync(t.ordinal, 0xff, (size_t)cap * sizeof(*t.ordinal), ctx->stream));
    CK(cudaMemsetAsync(t.state, 0, sizeof(*t.state), ctx->stream));
    t.cap = cap;
    t.max_voxels = (uint32_t)max_voxels;
    t.S = (double)voxel_size;
    ctx->vox_bound = 0;
    ctx->vox_chunks = 0;
    ctx->vox_begun = true;
    return SCAN3D_OK;
}

// one add of <= W*H points (n_dev: the count is on the device)
static int voxel_add(scan3d_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgb, const uint32_t* n_dev,
                     uint32_t plane)
{
    CK(launch_voxel_add(ctx->vox, xyz, nrm, rgb, n_dev, plane, ctx->vox_point_slot, ctx->vox_flags, ctx->block_counts,
                        (int)(ctx->vox_chunks & 1), ctx->stream));
    ctx->vox_chunks++;
    ctx->launches += VOXEL_ADD_LAUNCHES;
    return SCAN3D_OK;
}

static const uint64_t VOXEL_MAX_POINTS = 0xffffffffull;   // point indices since begin are uint32

int scan3d_voxel_add_points(scan3d_ctx* ctx)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->vox_begun) return fail(ctx, SCAN3D_ERR_STATE, "voxel add before scan3d_voxel_begin");
    if (ctx->cfg.dirs != 2) return fail(ctx, SCAN3D_ERR_STATE, "no point cloud in a one-direction configuration");
    if (!ctx->have_points) return fail(ctx, SCAN3D_ERR_STATE, "voxel add before the points are computed");
    const uint64_t ub = npix(ctx);
    if (ctx->vox_bound + ub > VOXEL_MAX_POINTS)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more than 2^32 - 1 points since scan3d_voxel_begin (W*H counted per ctx add)");
    CK(cudaSetDevice(ctx->device));
    ctx->vox_bound += ub;
    ctx->vox_fresh = false;
    return voxel_add(ctx, points_of(ctx), ctx->have_mesh ? ctx->mesh_normals : nullptr,
                     ctx->texture && ctx->rgb ? ctx->rgb : nullptr, ctx->d_count, (uint32_t)ub);
}

int scan3d_voxel_add_points_dev(scan3d_ctx* ctx, const float* xyz_dev, const float* normals_dev, const uint8_t* rgb_dev,
                                int64_t n)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (n < 0) return fail(ctx, SCAN3D_ERR_ARG, "n < 0");
    if (!xyz_dev && n > 0) return fail(ctx, SCAN3D_ERR_ARG, "null xyz_dev");
    if (((uintptr_t)xyz_dev & 3) || ((uintptr_t)normals_dev & 3))
        return fail(ctx, SCAN3D_ERR_ARG, "xyz_dev and normals_dev must be 4-byte aligned");
    if (!ctx->vox_begun) return fail(ctx, SCAN3D_ERR_STATE, "voxel add before scan3d_voxel_begin");
    if (ctx->vox_bound + (uint64_t)n > VOXEL_MAX_POINTS)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more than 2^32 - 1 points since scan3d_voxel_begin");
    CK(cudaSetDevice(ctx->device));
    ctx->vox_bound += (uint64_t)n;
    ctx->vox_fresh = false;
    const int64_t chunk = (int64_t)npix(ctx);   // the per-point scratch holds W*H points
    for (int64_t off = 0; off < n; off += chunk) {
        const int64_t k = std::min(chunk, n - off);
        const int rc = voxel_add(ctx, xyz_dev + 3 * off, normals_dev ? normals_dev + 3 * off : nullptr,
                                 rgb_dev ? rgb_dev + 3 * off : nullptr, nullptr, (uint32_t)k);
        if (rc) return rc;
    }
    return SCAN3D_OK;
}

int scan3d_voxel_finish(scan3d_ctx* ctx)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->vox_begun) return fail(ctx, SCAN3D_ERR_STATE, "voxel finish before scan3d_voxel_begin");
    CK(cudaSetDevice(ctx->device));
    CK(launch_voxel_finish(ctx->vox, (int)(ctx->vox_chunks & 1), ctx->vox_xyz, ctx->vox_nrm, ctx->vox_rgb, ctx->vox_cnt,
                           ctx->sm_count, ctx->stream));
    ctx->launches += 1;
    ctx->vox_fresh = true;
    return SCAN3D_OK;
}

int scan3d_voxel_count(scan3d_ctx* ctx, int64_t* voxels_out, int64_t* dropped_out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->vox_begun || !ctx->vox_fresh)
        return fail(ctx, SCAN3D_ERR_STATE, "no voxel outputs of the current adds: call scan3d_voxel_finish");
    CK(cudaSetDevice(ctx->device));
    VoxelState st;
    CK(cudaMemcpyAsync(&st, ctx->vox.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st.overflow || st.occupied > ctx->vox.max_voxels)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more distinct voxels than max_voxels: begin again with a larger max_voxels");
    if (voxels_out) *voxels_out = st.total[ctx->vox_chunks & 1];
    if (dropped_out) *dropped_out = (int64_t)st.dropped;
    return SCAN3D_OK;
}

int scan3d_get_voxels(scan3d_ctx* ctx, float* xyz_host, float* normals_host, uint8_t* rgb_host, uint32_t* counts_host,
                      int64_t max_voxels)
{
    int64_t n = 0;
    int rc = scan3d_voxel_count(ctx, &n, nullptr);
    if (rc) return rc;
    if (n > max_voxels) n = max_voxels;
    if (n <= 0) return SCAN3D_OK;
    if (xyz_host) CK(cudaMemcpyAsync(xyz_host, ctx->vox_xyz, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    if (normals_host) CK(cudaMemcpyAsync(normals_host, ctx->vox_nrm, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    if (rgb_host) CK(cudaMemcpyAsync(rgb_host, ctx->vox_rgb, (size_t)n * 3, cudaMemcpyDeviceToHost, ctx->stream));
    if (counts_host) CK(cudaMemcpyAsync(counts_host, ctx->vox_cnt, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

int scan3d_write_voxel_ply(scan3d_ctx* ctx, const char* path, int binary)
{
    if (!ctx || !path) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    int64_t n = 0;
    int rc = scan3d_voxel_count(ctx, &n, nullptr);
    if (rc) return rc;
    std::vector<float> xyz((size_t)n * 3), nrm((size_t)n * 3);
    std::vector<uint8_t> rgb((size_t)n * 3);
    rc = scan3d_get_voxels(ctx, xyz.data(), nrm.data(), rgb.data(), nullptr, n);
    if (rc) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ctx, SCAN3D_ERR_IO, "cannot open PLY for writing");
    write_ply_with_normals(f, binary, n, xyz.data(), nrm.data(), rgb.data(), "");
    const bool ok = fclose(f) == 0;
    return ok ? SCAN3D_OK : fail(ctx, SCAN3D_ERR_IO, "PLY write failed");
}

// ------------------------------------------------------------------------------------------
// stage 1: projector patterns on the device
// ------------------------------------------------------------------------------------------
int64_t scan3d_pattern_bytes(const scan3d_config* c, int dir)
{
    if (!c || dir < 0 || dir > 1 || c->PW < 1 || c->PH < 1) return 0;
    return (int64_t)(c->N + 2 * (dir == 0 ? c->M_v : c->M_h)) * c->PW * c->PH;
}

int scan3d_generate_patterns_dev(scan3d_ctx* ctx, int dir, uint8_t* patterns_dev)
{
    if (!ctx || !patterns_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    const scan3d_config& c = ctx->cfg;
    if (dir < 0 || dir > 1 || c.PW < 1 || c.PH < 1) return fail(ctx, SCAN3D_ERR_ARG, "bad direction or projector size");
    if (c.PW % 16 != 0 || ((uintptr_t)patterns_dev & 15)) return fail(ctx, SCAN3D_ERR_ARG, "PW and the destination must be multiples of 16");
    CK(cudaSetDevice(ctx->device));
    const int M = dir == 0 ? c.M_v : c.M_h, fw = dir == 0 ? c.fw_v : c.fw_h;
    const int len = dir == 0 ? c.PW : c.PH, lenp = (len + 15) & ~15, np = c.N + 2 * M;
    const size_t max_prof = (size_t)(16 + 2 * 15) * (((size_t)std::max(c.PW, c.PH) + 15) & ~(size_t)15);
    if (!ctx->pattern_profiles) CK(dalloc(&ctx->pattern_profiles, 2 * max_prof));
    uint8_t* d_prof = ctx->pattern_profiles + (size_t)dir * max_prof;
    if (!ctx->have_profiles[dir]) {      // the profiles depend on the configuration only: once per context
        std::vector<uint8_t> prof((size_t)np * lenp, 0);
        for (int k = 0; k < c.N; k++) s3d_profile::pattern_profile(0, c.N, fw, k, len, &prof[(size_t)k * lenp]);
        for (int k = 0; k < M; k++) {
            s3d_profile::pattern_profile(1, M, fw, k, len, &prof[(size_t)(c.N + k) * lenp]);
            s3d_profile::pattern_profile(2, M, fw, k, len, &prof[(size_t)(c.N + M + k) * lenp]);
        }
        CK(cudaMemcpyAsync(d_prof, prof.data(), prof.size(), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));      // prof is a local
        ctx->have_profiles[dir] = true;
    }
    CK(launch_expand_patterns(d_prof, lenp, np, patterns_dev, c.PW, c.PH, dir, ctx->stream));
    ctx->launches++;
    return SCAN3D_OK;
}

int scan3d_generate_patterns(scan3d_ctx* ctx, int dir, uint8_t* patterns_host)
{
    if (!ctx || !patterns_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    const int64_t bytes = scan3d_pattern_bytes(&ctx->cfg, dir);
    if (bytes <= 0) return fail(ctx, SCAN3D_ERR_ARG, "bad direction or projector size");
    CK(cudaSetDevice(ctx->device));
    uint8_t* d = nullptr;
    CK(cudaMalloc((void**)&d, (size_t)bytes));
    int rc = scan3d_generate_patterns_dev(ctx, dir, d);
    cudaError_t e = cudaSuccess;
    if (rc == SCAN3D_OK) e = cudaMemcpyAsync(patterns_host, d, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream);
    const cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (rc) return rc;
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(ctx, SCAN3D_ERR_CUDA, cudaGetErrorString(e != cudaSuccess ? e : e2));
    return SCAN3D_OK;
}

int scan3d_write_pcd(scan3d_ctx* ctx, const char* path)
{
    if (!ctx || !path) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    int64_t n = 0;
    int rc = scan3d_point_count(ctx, &n);
    if (rc) return rc;
    std::vector<float> xyz((size_t)n * 3);
    std::vector<uint8_t> rgb((size_t)n * 3);
    rc = scan3d_get_points(ctx, xyz.data(), nullptr, rgb.data(), n);
    if (rc) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ctx, SCAN3D_ERR_IO, "cannot open PCD for writing");
    fprintf(f, "# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z rgb\nSIZE 4 4 4 4\n"
               "TYPE F F F F\nCOUNT 1 1 1 1\nWIDTH %lld\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS %lld\nDATA ascii\n",
            (long long)n, (long long)n);
    for (int64_t i = 0; i < n; i++) {
        const uint32_t packed = ((uint32_t)rgb[3 * i] << 16) | ((uint32_t)rgb[3 * i + 1] << 8) | rgb[3 * i + 2];
        float c;
        memcpy(&c, &packed, 4);
        fprintf(f, "%.8g %.8g %.8g %.8g\n", xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], c);
    }
    const bool ok = fclose(f) == 0;
    return ok ? SCAN3D_OK : fail(ctx, SCAN3D_ERR_IO, "PCD write failed");
}

// ---- self-test entry (not part of the reference boundary): (float)atan2(y,x) on the GPU ----
int scan3d_debug_atan2(scan3d_ctx* ctx, const double* y_host, const double* x_host, float* out_host, int n, int mode)
{
    if (!ctx || !y_host || !x_host || !out_host || n <= 0) return fail(ctx, SCAN3D_ERR_ARG, "bad argument");
    CK(cudaSetDevice(ctx->device));
    double *dy = nullptr, *dx = nullptr;
    float* dout = nullptr;
    cudaError_t e = cudaMalloc((void**)&dy, (size_t)n * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&dx, (size_t)n * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&dout, (size_t)n * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dy, y_host, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dx, x_host, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = launch_debug_atan2(dy, dx, dout, n, mode, ctx->atan_tab, ctx->stream);
    if (e == cudaSuccess) {
        ctx->launches++;
        e = cudaMemcpyAsync(out_host, dout, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream);
    }
    const cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    cudaFree(dy); cudaFree(dx); cudaFree(dout);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(ctx, SCAN3D_ERR_CUDA, cudaGetErrorString(e != cudaSuccess ? e : e2));
    return SCAN3D_OK;
}

// ---- diagnostics: pipeline timeline of the last fused launch (library built with
//      SCAN3D_BUILD_TRACE=1, context created with SCAN3D_TRACE=1 in the environment) ----
int scan3d_debug_get_trace(scan3d_ctx* ctx, uint64_t* out_host, int64_t n_words)
{
#if !defined(S3D_TRACE) || !S3D_TRACE
    return fail(ctx, SCAN3D_ERR_STATE, "this build has no trace hooks: rebuild with SCAN3D_BUILD_TRACE=1");
#endif
    if (!ctx || !out_host || !ctx->trace) return fail(ctx, SCAN3D_ERR_STATE, "tracing is not enabled");
    CK(cudaSetDevice(ctx->device));
    if (n_words > 1024 * 64 * 8) n_words = 1024 * 64 * 8;
    CK(cudaMemcpyAsync(out_host, ctx->trace, (size_t)n_words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

// ---- self-test entry: exact-quotient shortcut vs IEEE division over every float phase ----
int scan3d_debug_divcheck(scan3d_ctx* ctx, uint64_t* mismatches)
{
    if (!ctx || !mismatches) return fail(ctx, SCAN3D_ERR_ARG, "bad argument");
    CK(cudaSetDevice(ctx->device));
    unsigned long long* d = nullptr;
    CK(cudaMalloc((void**)&d, 8));
    unsigned long long h = 0;
    cudaError_t e = cudaMemsetAsync(d, 0, 8, ctx->stream);
    if (e == cudaSuccess) e = launch_debug_divcheck(d, ctx->stream);
    if (e == cudaSuccess) { ctx->launches++; e = cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, ctx->stream); }
    const cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(ctx, SCAN3D_ERR_CUDA, cudaGetErrorString(e != cudaSuccess ? e : e2));
    *mismatches = h;
    return SCAN3D_OK;
}

}  // extern "C"
