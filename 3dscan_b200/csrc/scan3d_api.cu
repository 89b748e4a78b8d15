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
#include "../common/scan3d_align_math.h"
#include "../common/scan3d_surface_math.h"
#include "../common/scan3d_decimate_math.h"
#include "../common/scan3d_orient_math.h"

using namespace s3d;

static thread_local std::string g_create_error;

static size_t npix(const scan3d_ctx* c) { return (size_t)c->cfg.W * c->cfg.H; }

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
            CK(ctx->unwrapped[d].ensure(n));
            CK(ctx->code[d].ensure(n));
        }
        CK(ctx->mask[0].ensure(n));
        CK(ctx->valid.ensure(n));
        if (D == 2) {
            CK(ctx->cpmap.ensure(n));
            CK(ctx->pts.ensure(3 * n));
            if (cfg->flags & SCAN3D_FLAG_POINT_PIXELS) CK(ctx->pix.ensure(n));
        }
        CK(ctx->d_count.ensure(4));
        CK(cudaMemsetAsync(ctx->d_count, 0, 16, ctx->stream));
        const int ntiles = fused_num_tiles(ctx->cfg);
        CK(ctx->tile_state.ensure((size_t)ntiles + 1));
        CK(cudaMemsetAsync(ctx->tile_state, 0, ((size_t)ntiles + 1) * 8, ctx->stream));
        if (getenv("SCAN3D_TRACE")) {
            CK(ctx->trace.ensure((size_t)1024 * 64 * 8));
            CK(cudaMemsetAsync(ctx->trace, 0, (size_t)1024 * 64 * 8 * 8, ctx->stream));
        }
        CK(ctx->tile_flags.ensure((size_t)ntiles + 16));
        CK(ctx->tile_list.ensure((size_t)ntiles + 16));
        CK(ctx->atan_tab.ensure((size_t)ATAN_TAB_DOUBLES));
        double tab[ATAN_TAB_DOUBLES];
        fill_atan_table(tab);
        CK(cudaMemcpyAsync(ctx->atan_tab, tab, sizeof(tab), cudaMemcpyHostToDevice, ctx->stream));
        const int n_codes = 1 << (cfg->dirs == 2 && cfg->M_h > cfg->M_v ? cfg->M_h : cfg->M_v);
        std::vector<double> code_term(n_codes);
        fill_code_term_table(code_term.data(), n_codes);
        CK(ctx->code_term.ensure((size_t)n_codes));
        CK(cudaMemcpyAsync(ctx->code_term, code_term.data(), n_codes * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(ctx->nstep_w.ensure(128));
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
    const cudaStream_t own = ctx->own_stream;
    if (own) cudaStreamSynchronize(own);
    delete ctx;                                   // frees every buffer, before their stream goes
    if (own) cudaStreamDestroy(own);
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
    {
        double Rc[9];
        rodrigues_host(cal->rc, Rc);
        camera_frame_calib(cal->Kc, Rc, cal->tc, d.Ap, &d);
    }
    d.proj_std = std_form(cal->Kp);
    d.fast_div_ok = ctx->fast_div_ok ? 1 : 0;
    d.cam_distorted = d.proj_distorted = 0;
    for (int i = 0; i < 5; i++) {
        if (cal->dc[i] != 0.0) d.cam_distorted = 1;
        if (cal->dp[i] != 0.0) d.proj_distorted = 1;
    }
    ctx->cam_lut.release();
    ctx->proj_lut.release();
    for (int k = 0; k < 2; k++) {   // cv::undistort maps belong to the previous calibration
        ctx->undist_xy[k].release();
        ctx->undist_frac[k].release();
    }
    if (ctx->cfg.dirs == 2) {
        // a table also for an intrinsic matrix that is not [fx 0 cx; 0 fy cy; 0 0 1] (skew, ...): the kernels' table-free
        // route then only ever sees the standard form (4 operations per coordinate, no division)
        if (d.cam_distorted || !d.cam_std) {
            CK(ctx->cam_lut.ensure(npix(ctx)));
            CK(launch_undistort_lut(nullptr, d, false, ctx->cfg.W, ctx->cfg.H, ctx->cfg.row0, ctx->cam_lut, ctx->stream));
            ctx->launches++;
        }
        if (d.proj_distorted || !d.proj_std) {
            CK(ctx->proj_lut.ensure((size_t)ctx->cfg.PW * ctx->cfg.PH));
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
        ctx->texture.release();
        ctx->results.drop(POINT_COLOURS);
        return SCAN3D_OK;
    }
    CK(ctx->texture.ensure(3 * npix(ctx)));
    CK(ctx->rgb.ensure(3 * npix(ctx)));
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
    CK(ctx->wrapped[dir].ensure(n));
    CK(ctx->mask[dir].ensure(n));
    return SCAN3D_OK;
}

static inline float* points_of(const scan3d_ctx* ctx) { return ctx->pts_ext ? ctx->pts_ext : ctx->pts; }

// SCAN3D_FLAG_STRICT_REFERENCE: replace the caller's ROI by the plane check_I_mod_criteria derives from it as committed
static int strict_roi(scan3d_ctx* ctx, const uint8_t** roi_dev)
{
    if (!(ctx->cfg.flags & SCAN3D_FLAG_STRICT_REFERENCE)) return SCAN3D_OK;
    const size_t n = (size_t)ctx->cfg.W * ctx->cfg.H_total;
    CK(ctx->roi_strict.ensure(n));
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

// compute_wrapped_phase on the effective ROI (strict_roi applied), after the caller dropped the direction's results
static int wrapped_phase(scan3d_ctx* ctx, int dir, const uint8_t* fringe_dev, const uint8_t* roi_dev)
{
    const int rc = ensure_stage_planes(ctx, dir);
    if (rc) return rc;
    const Shape s = shape_of(ctx->cfg);
    if (ctx->cfg.flags & SCAN3D_FLAG_MODULATION_MASK) {
        CK(ctx->roi_eff.ensure(npix(ctx)));
        CK(launch_modulation_roi(s, fringe_dev, roi_dev, ctx->roi_eff, ctx->stream));
        ctx->launches++;
        roi_dev = ctx->roi_eff;
    }
    CK(launch_wrapped(s, ctx->cfg.N, fringe_dev, roi_dev, ctx->wrapped[dir], ctx->atan_tab, ctx->nstep_w, false, ctx->stream));
    CK(launch_mask(s, roi_dev, ctx->mask[dir], ctx->stream));
    ctx->launches += 2;
    ctx->results.produce(dir == 0 ? WRAPPED_V : WRAPPED_H);
    return SCAN3D_OK;
}

int scan3d_compute_wrapped_phase_dev(scan3d_ctx* ctx, int dir, const uint8_t* fringe_dev, const uint8_t* roi_dev)
{
    if (!ctx || !fringe_dev || !roi_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (dir < 0 || dir >= ctx->cfg.dirs) return fail(ctx, SCAN3D_ERR_ARG, "bad pattern_type");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(dir == 0 ? WRAPPED_V : WRAPPED_H);
    const int rc = strict_roi(ctx, &roi_dev);
    if (rc) return rc;
    return wrapped_phase(ctx, dir, fringe_dev, roi_dev);
}

// The host-pointer entries stage their inputs in the context's own buffers (allocated on first use, sized for a whole
// capture stack, kept until scan3d_destroy): no allocation or free per call.
static int ensure_staging(scan3d_ctx* ctx)
{
    const size_t sb = (size_t)scan3d_stack_bytes(&ctx->cfg);
    size_t rb;
    roi_bytes(ctx, &rb);
    CK(ctx->d_stack.ensure(sb));
    CK(ctx->d_roi.ensure(rb));
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
    if (!ctx->results.has(dir == 0 ? WRAPPED_V : WRAPPED_H))
        return fail(ctx, SCAN3D_ERR_STATE, "unwrap_phase before compute_wrapped_phase");
    CK(cudaSetDevice(ctx->device));
    const Result unwrapped = dir == 0 ? UNWRAPPED_V : UNWRAPPED_H;
    ctx->results.drop(unwrapped);
    const Shape s = shape_of(ctx->cfg);
    const int M = dir == 0 ? ctx->cfg.M_v : ctx->cfg.M_h;
    CK(launch_unwrap(s, dir, M, gray_dev, inv_dev, ctx->wrapped[dir], ctx->mask[dir], ctx->code[dir],
                     ctx->unwrapped[dir], ctx->stream));
    ctx->launches++;
    ctx->results.produce(unwrapped);
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
    if (!ctx->results.has(UNWRAPPED_V) || !ctx->results.has(UNWRAPPED_H))
        return fail(ctx, SCAN3D_ERR_STATE, "compute_c_p_map before unwrap_phase(0) and (1)");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(CPMAP);
    ctx->results.drop(VALID);
    const Shape s = shape_of(ctx->cfg);
    CK(launch_cpmap(s, ctx->cfg.fw_v, ctx->cfg.fw_h, ctx->unwrapped[0], ctx->unwrapped[1], ctx->mask[0],
                    ctx->mask[1], ctx->cpmap, ctx->valid, ctx->stream));
    ctx->launches++;
    ctx->results.produce(CPMAP);
    ctx->results.produce(VALID);
    return SCAN3D_OK;
}

int scan3d_triangulate(scan3d_ctx* ctx)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->has_calib) return fail(ctx, SCAN3D_ERR_STATE, "triangulate before set_calibration");
    if (!ctx->results.has(CPMAP)) return fail(ctx, SCAN3D_ERR_STATE, "triangulate before compute_c_p_map");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(XYZ);
    CK(ctx->xyz.ensure(3 * npix(ctx)));
    const Shape s = shape_of(ctx->cfg);
    CK(launch_triangulate(s, ctx->dcal, ctx->cam_lut, ctx->proj_lut, ctx->cpmap, ctx->valid, ctx->xyz, ctx->stream));
    ctx->launches++;
    ctx->results.produce(XYZ);
    return SCAN3D_OK;
}

// the compacted points, and their colours when a texture is set
static void produce_points(scan3d_ctx* ctx)
{
    ctx->results.produce(POINTS);
    if (ctx->texture) ctx->results.produce(POINT_COLOURS);
}

int scan3d_compact_points(scan3d_ctx* ctx, int64_t* count_out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->results.has(XYZ)) return fail(ctx, SCAN3D_ERR_STATE, "compact_points before triangulate");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(POINTS);
    const size_t n = npix(ctx);
    CK(ctx->block_counts.ensure((n + 1023) / 1024 + 1));
    CK(ctx->pix.ensure(n));
    if (ctx->texture) CK(ctx->rgb.ensure(3 * n));
    const Shape s = shape_of(ctx->cfg);
    int nl = 0;
    CK(launch_compact(s, ctx->xyz, ctx->valid, ctx->texture, ctx->block_counts, points_of(ctx), ctx->pix,
                      ctx->texture ? ctx->rgb.get() : nullptr, ctx->d_count, ctx->stream, &nl));
    ctx->launches += nl;
    produce_points(ctx);
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
        int rc = wrapped_phase(ctx, d, p, roi);
        if (rc) return rc;
        p += (size_t)c.N * n;
        rc = scan3d_unwrap_phase_dev(ctx, d, p, p + (size_t)M * n);
        if (rc) return rc;
        p += 2 * (size_t)M * n;
    }
    if (c.dirs == 1) {
        CK(cudaMemcpyAsync(ctx->valid, ctx->mask[0], n, cudaMemcpyDeviceToDevice, ctx->stream));
        ctx->results.produce(VALID);
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
    ctx->results.drop(WRAPPED_V);     // every pixel result is computed from the wrapped phases
    ctx->results.drop(WRAPPED_H);
    {
        const int rc = strict_roi(ctx, &roi_dev);
        if (rc) return rc;
    }
    if (!ctx->fast_div_ok || !fused7_supported(ctx->cfg)) return reconstruct_stagewise(ctx, stack_dev, roi_dev);
    const scan3d_config& c = ctx->cfg;
    FusedArgs a{};
    a.stack = stack_dev; a.roi = roi_dev;
    if (c.flags & SCAN3D_FLAG_MODULATION_MASK) {
        // check_I_mod_criteria's modulation criterion (3/wrapped_phase.cpp:84-104): one effective ROI plane per
        // direction from that direction's three fringe images (a pre-pass: the mask recurrence needs it two rows up)
        const Shape s = shape_of(c);
        const size_t n = npix(ctx);
        CK(ctx->roi_eff.ensure(n));
        CK(launch_modulation_roi(s, stack_dev, roi_dev, ctx->roi_eff, ctx->stream));
        ctx->launches++;
        a.roi = ctx->roi_eff;
        a.roi2 = ctx->roi_eff;
        a.roi_list = roi_dev;
        if (c.dirs == 2) {
            CK(ctx->roi_eff_h.ensure(n));
            CK(launch_modulation_roi(s, stack_dev + (size_t)(c.N + 2 * c.M_v) * n, roi_dev, ctx->roi_eff_h, ctx->stream));
            ctx->launches++;
            a.roi2 = ctx->roi_eff_h;
        }
    }
    a.unw_v = ctx->unwrapped[0]; a.unw_h = ctx->unwrapped[1];
    a.code_v = ctx->code[0]; a.code_h = ctx->code[1];
    a.valid = ctx->valid; a.cpmap = ctx->cpmap;
    a.pts = points_of(ctx); a.pix = ctx->pix;
    a.rgb = ctx->texture ? ctx->rgb.get() : nullptr; a.texture = ctx->texture;
    a.d_count = ctx->d_count; a.tile_state = ctx->tile_state; a.trace = ctx->trace; a.tile_flags = ctx->tile_flags; a.tile_list = ctx->tile_list + 1; a.n_list = ctx->tile_list;
    a.cam_lut = ctx->cam_lut; a.proj_lut = ctx->proj_lut; a.atan_tab = ctx->atan_tab; a.code_term = ctx->code_term;
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
    CK(launch_fused7(c, a, ctx->dcal, ctx->sm_count, ctx->stream));
    ctx->launches += 3;   // work-list flags, work-list scan, persistent fused kernel
    if (ctx->reg_on && !fold_reg && c.dirs == 2) {
        // shapes without the folding variant: the same transform as one more pass over the compacted points
        CK(launch_register_points(points_of(ctx), points_of(ctx), (long long)npix(ctx), ctx->reg_R, ctx->reg_t[0], ctx->reg_t[1],
                                  ctx->reg_t[2], ctx->sm_count, ctx->stream));
        ctx->launches++;
    }
    // inputs before what is computed from them: producing a result drops what was computed from its old value
    ctx->results.produce(UNWRAPPED_V);
    if (c.dirs == 2) ctx->results.produce(UNWRAPPED_H);
    ctx->results.produce(VALID);
    if (c.dirs == 2) {
        ctx->results.produce(CPMAP);
        produce_points(ctx);
    }
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
    CK(ctx->d_undist.ensure(sb));
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
// a plane id's buffer, its element size and the result that holds it
struct Plane {
    void* buf;
    size_t elt;
    Result result;
};

static Plane plane_of(const scan3d_ctx* ctx, int plane)
{
    switch (plane) {
        case SCAN3D_PLANE_WRAPPED_V: return {ctx->wrapped[0], 4, WRAPPED_V};
        case SCAN3D_PLANE_WRAPPED_H: return {ctx->wrapped[1], 4, WRAPPED_H};
        case SCAN3D_PLANE_UNWRAPPED_V: return {ctx->unwrapped[0], 4, UNWRAPPED_V};
        case SCAN3D_PLANE_UNWRAPPED_H: return {ctx->unwrapped[1], 4, UNWRAPPED_H};
        case SCAN3D_PLANE_CODE_V: return {ctx->code[0], 2, UNWRAPPED_V};
        case SCAN3D_PLANE_CODE_H: return {ctx->code[1], 2, UNWRAPPED_H};
        case SCAN3D_PLANE_MASK: return {ctx->mask[0], 1, WRAPPED_V};
        case S3D_PLANE_MASK_H: return {ctx->mask[1], 1, WRAPPED_H};
        case SCAN3D_PLANE_VALID: return {ctx->valid, 1, VALID};
        case SCAN3D_PLANE_CPMAP: return {ctx->cpmap, 8, CPMAP};
        case SCAN3D_PLANE_XYZ: return {ctx->xyz, 24, XYZ};
        default: return {nullptr, 0, RESULT_COUNT};
    }
}

int64_t scan3d_plane_bytes(const scan3d_ctx* ctx, int plane)
{
    if (!ctx) return 0;
    return (int64_t)(plane_of(ctx, plane).elt * npix(ctx));
}

void* scan3d_device_plane(scan3d_ctx* ctx, int plane)
{
    if (!ctx) return nullptr;
    const Plane p = plane_of(ctx, plane);
    return ctx->results.has(p.result) ? p.buf : nullptr;     // (a plane nothing has written is not handed out)
}

int scan3d_get_plane(scan3d_ctx* ctx, int plane, void* dst_host)
{
    if (!ctx || !dst_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    const Plane p = plane_of(ctx, plane);
    if (!p.buf || !ctx->results.has(p.result))
        return fail(ctx, SCAN3D_ERR_STATE, "plane not available: no compute entry has produced it (the single-pass entry "
                                           "keeps wrapped phases and per-direction masks in registers)");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dst_host, p.buf, p.elt * npix(ctx), cudaMemcpyDeviceToHost, ctx->stream));
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
    if (!ctx->results.has(POINTS)) return fail(ctx, SCAN3D_ERR_STATE, "no compacted points yet");
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
        if (ctx->results.has(POINT_COLOURS)) CK(cudaMemcpyAsync(rgb_host, ctx->rgb, (size_t)n * 3, cudaMemcpyDeviceToHost, ctx->stream));
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
    ctx->results.drop(POINTS);
    ctx->pts_ext = (float*)points_dev;
    return SCAN3D_OK;
}
void* scan3d_device_point_pixels(scan3d_ctx* ctx) { return ctx ? ctx->pix.get() : nullptr; }
void* scan3d_device_point_count(scan3d_ctx* ctx) { return ctx ? ctx->d_count.get() : nullptr; }

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

// The vertex element of write_ply_with_normals and the face element "vertex_indices" (uchar count, int indices) of
// scan3d_write_mesh_ply and scan3d_write_voxel_surface_ply.
static void write_ply_with_faces(FILE* f, int binary, int64_t nv, const float* xyz, const float* nrm, const uint8_t* rgb,
                                 int64_t nf, const int32_t* faces)
{
    char face_header[96];
    snprintf(face_header, sizeof(face_header), "element face %lld\nproperty list uchar int vertex_indices\n", (long long)nf);
    write_ply_with_normals(f, binary, nv, xyz, nrm, rgb, face_header);
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
    if (!ctx->results.has(POINTS)) return fail(ctx, SCAN3D_ERR_STATE, "build_mesh before the points are computed");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(MESH);
    const size_t n = npix(ctx);
    const size_t nb = (n + POINT_BLOCK - 1) / POINT_BLOCK;
    const size_t max_faces = 2 * (size_t)(c.W - 1) * (size_t)(c.H - 1);
    CK(ctx->block_counts.ensure(nb + 1));
    CK(ctx->mesh_idx.ensure(n));
    CK(ctx->mesh_counts.ensure(nb));
    CK(ctx->mesh_totals.ensure(2));
    CK(ctx->mesh_faces.ensure(3 * std::max(max_faces, (size_t)1)));
    CK(ctx->mesh_normals.ensure(3 * n));
    CK(launch_mesh(ctx->valid, points_of(ctx), c.W, c.H, max_edge, ctx->mesh_idx, ctx->block_counts, ctx->mesh_counts,
                   ctx->mesh_totals, ctx->mesh_faces, ctx->mesh_normals, ctx->stream, &ctx->launches));
    ctx->results.produce(MESH);
    return SCAN3D_OK;
}

int scan3d_mesh_face_count(scan3d_ctx* ctx, int64_t* count_out)
{
    if (!ctx || !count_out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!ctx->results.has(MESH)) return fail(ctx, SCAN3D_ERR_STATE, "no mesh of the current points: call scan3d_build_mesh");
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

void* scan3d_device_mesh_faces(scan3d_ctx* ctx) { return ctx && ctx->results.has(MESH) ? ctx->mesh_faces.get() : nullptr; }
void* scan3d_device_point_normals(scan3d_ctx* ctx)
{
    return ctx && ctx->results.has(MESH) ? ctx->mesh_normals.get() : nullptr;
}

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
    write_ply_with_faces(f, binary, np, xyz.data(), nrm.data(), rgb.data(), nf, faces.data());
    const bool ok = fclose(f) == 0;
    return ok ? SCAN3D_OK : fail(ctx, SCAN3D_ERR_IO, "PLY write failed");
}

// ------------------------------------------------------------------------------------------
// voxel-grid merge of registered views (include/scan3d.h and common/scan3d_voxel_math.h have the exact rules)
// ------------------------------------------------------------------------------------------
int scan3d_voxel_begin(scan3d_ctx* ctx, float voxel_size, int64_t max_voxels)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!(voxel_size > 0.0f && voxel_size - voxel_size == 0.0f))
        return fail(ctx, SCAN3D_ERR_ARG, "voxel_size must be finite and > 0");
    if (max_voxels < 1 || max_voxels >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_ARG, "max_voxels must be in [1, 2^31)");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(ACCUMULATOR);
    CK(ctx->vox.reset((uint32_t)max_voxels, (double)voxel_size, ctx->sm_count, ctx->stream));
    const size_t m = (size_t)max_voxels, n = npix(ctx);
    CK(grow_group(Grow(ctx->vox_xyz, 3 * m), Grow(ctx->vox_nrm, 3 * m), Grow(ctx->vox_rgb, 3 * m),
                  Grow(ctx->vox_cnt, m)));
    CK(ctx->vox_point_slot.ensure(n));
    CK(ctx->vox_flags.ensure(n));
    CK(ctx->block_counts.ensure((n + POINT_BLOCK - 1) / POINT_BLOCK + 1));
    ctx->vox_bound = 0;
    ctx->vox_chunks = 0;
    ctx->results.produce(ACCUMULATOR);
    return SCAN3D_OK;
}

// one add of <= W*H points (n_dev: the count is on the device)
static int voxel_add(scan3d_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgb, const uint32_t* n_dev,
                     uint32_t plane)
{
    CK(launch_voxel_add(ctx->vox.view, xyz, nrm, rgb, n_dev, plane, ctx->vox_point_slot, ctx->vox_flags,
                        ctx->block_counts, (int)(ctx->vox_chunks & 1), ctx->stream, &ctx->launches));
    ctx->vox_chunks++;
    return SCAN3D_OK;
}

static const uint64_t VOXEL_MAX_POINTS = 0xffffffffull;   // point indices since begin are uint32

int scan3d_voxel_add_points(scan3d_ctx* ctx)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->results.has(ACCUMULATOR)) return fail(ctx, SCAN3D_ERR_STATE, "voxel add before scan3d_voxel_begin");
    if (ctx->cfg.dirs != 2) return fail(ctx, SCAN3D_ERR_STATE, "no point cloud in a one-direction configuration");
    if (!ctx->results.has(POINTS)) return fail(ctx, SCAN3D_ERR_STATE, "voxel add before the points are computed");
    const uint64_t ub = npix(ctx);
    if (ctx->vox_bound + ub > VOXEL_MAX_POINTS)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more than 2^32 - 1 points since scan3d_voxel_begin (W*H counted per ctx add)");
    CK(cudaSetDevice(ctx->device));
    ctx->vox_bound += ub;
    ctx->results.drop(VOXELS);
    return voxel_add(ctx, points_of(ctx), ctx->results.has(MESH) ? ctx->mesh_normals.get() : nullptr,
                     ctx->results.has(POINT_COLOURS) ? ctx->rgb.get() : nullptr, ctx->d_count, (uint32_t)ub);
}

int scan3d_voxel_add_points_dev(scan3d_ctx* ctx, const float* xyz_dev, const float* normals_dev, const uint8_t* rgb_dev,
                                int64_t n)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (n < 0) return fail(ctx, SCAN3D_ERR_ARG, "n < 0");
    if (!xyz_dev && n > 0) return fail(ctx, SCAN3D_ERR_ARG, "null xyz_dev");
    if (((uintptr_t)xyz_dev & 3) || ((uintptr_t)normals_dev & 3))
        return fail(ctx, SCAN3D_ERR_ARG, "xyz_dev and normals_dev must be 4-byte aligned");
    if (!ctx->results.has(ACCUMULATOR)) return fail(ctx, SCAN3D_ERR_STATE, "voxel add before scan3d_voxel_begin");
    if (ctx->vox_bound + (uint64_t)n > VOXEL_MAX_POINTS)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more than 2^32 - 1 points since scan3d_voxel_begin");
    CK(cudaSetDevice(ctx->device));
    ctx->vox_bound += (uint64_t)n;
    ctx->results.drop(VOXELS);
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
    if (!ctx->results.has(ACCUMULATOR)) return fail(ctx, SCAN3D_ERR_STATE, "voxel finish before scan3d_voxel_begin");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(VOXELS);
    CK(launch_voxel_finish(ctx->vox.view, (int)(ctx->vox_chunks & 1), ctx->vox_xyz, ctx->vox_nrm, ctx->vox_rgb,
                           ctx->vox_cnt, ctx->sm_count, ctx->stream));
    ctx->launches += 1;
    ctx->results.produce(VOXELS);
    return SCAN3D_OK;
}

int scan3d_voxel_count(scan3d_ctx* ctx, int64_t* voxels_out, int64_t* dropped_out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->results.has(VOXELS))
        return fail(ctx, SCAN3D_ERR_STATE, "no voxel outputs of the current adds: call scan3d_voxel_finish");
    CK(cudaSetDevice(ctx->device));
    VoxelState st;
    CK(cudaMemcpyAsync(&st, ctx->vox.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st.overflow || st.occupied > ctx->vox.view.max_voxels)
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
// scan-to-model alignment (include/scan3d.h and common/scan3d_align_math.h have the exact rules)
// ------------------------------------------------------------------------------------------
static bool finite_d(double v) { return v - v == 0.0; }

// T_init: finite, last row (0, 0, 0, 1), R^T R - I and det R - 1 within 1e-6
static bool rigid_4x4(const double* T)
{
    for (int k = 0; k < 16; k++)
        if (!finite_d(T[k])) return false;
    if (T[12] != 0.0 || T[13] != 0.0 || T[14] != 0.0 || T[15] != 1.0) return false;
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            const double d = T[i] * T[j] + T[4 + i] * T[4 + j] + T[8 + i] * T[8 + j] - (i == j ? 1.0 : 0.0);
            if (!(fabs(d) <= 1e-6)) return false;
        }
    const double det = T[0] * (T[5] * T[10] - T[6] * T[9]) - T[1] * (T[4] * T[10] - T[6] * T[8]) +
                       T[2] * (T[4] * T[9] - T[5] * T[8]);
    return fabs(det - 1.0) <= 1e-6;
}

static int check_align_args(scan3d_ctx* ctx, const scan3d_align_params* p, scan3d_align_result* out)
{
    if (!p || !out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!(p->max_distance > 0.0f && p->max_distance - p->max_distance == 0.0f))
        return fail(ctx, SCAN3D_ERR_ARG, "max_distance must be finite and > 0");
    if (p->max_iterations < 1 || p->max_iterations > 64) return fail(ctx, SCAN3D_ERR_ARG, "max_iterations must be in 1..64");
    if (p->stride < 1) return fail(ctx, SCAN3D_ERR_ARG, "stride must be >= 1");
    if (!(p->stop_rotation >= 0.0) || !(p->stop_translation >= 0.0))
        return fail(ctx, SCAN3D_ERR_ARG, "stop thresholds must be >= 0");
    if (!rigid_4x4(p->T_init)) return fail(ctx, SCAN3D_ERR_ARG, "T_init must be a finite rigid transform (rotation within 1e-6)");
    if (!ctx->results.has(VOXELS))
        return fail(ctx, SCAN3D_ERR_STATE, "no voxel outputs of the current adds to align to: call scan3d_voxel_finish");
    return SCAN3D_OK;
}

// the whole run on the source xyz (n_dev: its count is on the device, <= n_max)
static int align_run(scan3d_ctx* ctx, float* xyz, const uint32_t* n_dev, long long n_max, const scan3d_align_params* p,
                     scan3d_align_result* out)
{
    CK(cudaSetDevice(ctx->device));
    AlignRun run;
    for (int k = 0; k < 12; k++) run.T0[k] = p->T_init[k];
    run.S = s3l::cell_edge(p->max_distance);
    run.r2 = (double)p->max_distance * (double)p->max_distance;   // host TU: -ffp-contract=off
    run.stop_rotation = p->stop_rotation;
    run.stop_translation = p->stop_translation;
    run.max_iterations = p->max_iterations;
    CK(ctx->aln.align(ctx->vox.view, (int)(ctx->vox_chunks & 1), ctx->vox_xyz, ctx->vox_nrm, run, xyz, n_dev, n_max,
                      p->stride, ctx->sm_count, ctx->stream, &ctx->launches));
    AlignState st;
    CK(cudaMemcpyAsync(&st, ctx->aln.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st.overflow)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more distinct voxels than max_voxels: begin again with a larger max_voxels");
    for (int k = 0; k < 12; k++) out->T[k] = st.T[k];
    out->T[12] = out->T[13] = out->T[14] = 0.0;
    out->T[15] = 1.0;
    out->iterations = st.iterations;
    out->status = st.status;
    out->pairs_first = st.pairs_first;
    out->pairs_last = st.pairs_last;
    out->rms_first = st.rms_first;
    out->rms_last = st.rms_last;
    const long long n = n_dev ? std::min((long long)st.n_src, n_max) : n_max;
    if (p->apply && n > 0) {
        float R[16];
        for (int k = 0; k < 16; k++) R[k] = (float)out->T[k];
        CK(launch_register_points(xyz, xyz, n, R, 0.0f, 0.0f, 0.0f, ctx->sm_count, ctx->stream));
        ctx->launches += 1;
    }
    return SCAN3D_OK;
}

int scan3d_align_to_voxels(scan3d_ctx* ctx, const scan3d_align_params* p, scan3d_align_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    int rc = check_align_args(ctx, p, out);
    if (rc) return rc;
    if (ctx->cfg.dirs != 2) return fail(ctx, SCAN3D_ERR_STATE, "no point cloud in a one-direction configuration");
    if (!ctx->results.has(POINTS)) return fail(ctx, SCAN3D_ERR_STATE, "align before the points are computed");
    if (p->apply) ctx->results.drop(MESH);   // the points move; their colours stay theirs
    return align_run(ctx, points_of(ctx), ctx->d_count, (long long)npix(ctx), p, out);
}

int scan3d_align_to_voxels_dev(scan3d_ctx* ctx, float* xyz_dev, int64_t n, const scan3d_align_params* p,
                               scan3d_align_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (n < 0) return fail(ctx, SCAN3D_ERR_ARG, "n < 0");
    if (!xyz_dev && n > 0) return fail(ctx, SCAN3D_ERR_ARG, "null xyz_dev");
    if ((uintptr_t)xyz_dev & 3) return fail(ctx, SCAN3D_ERR_ARG, "xyz_dev must be 4-byte aligned");
    const int rc = check_align_args(ctx, p, out);
    if (rc) return rc;
    return align_run(ctx, xyz_dev, nullptr, (long long)n, p, out);
}

// ------------------------------------------------------------------------------------------
// triangle surface of the merged voxels (include/scan3d.h and common/scan3d_surface_math.h have the exact rules)
// ------------------------------------------------------------------------------------------
int scan3d_voxel_surface(scan3d_ctx* ctx, const scan3d_surface_params* p, scan3d_surface_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!p || !out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!(p->max_distance > 0.0f && p->max_distance - p->max_distance == 0.0f))
        return fail(ctx, SCAN3D_ERR_ARG, "max_distance must be finite and > 0");
    if (p->max_points < 1 || p->max_points >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_ARG, "max_points must be in [1, 2^31)");
    if (!ctx->results.has(VOXELS))
        return fail(ctx, SCAN3D_ERR_STATE, "no voxel outputs of the current adds to mesh: call scan3d_voxel_finish");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(SURFACE);
    ctx->srf_repaired = ctx->srf_filled_after_repair = false;
    AlignRun run{};                                      // the index only; T0 = I for the state it initialises
    run.T0[0] = run.T0[5] = run.T0[10] = 1.0;
    run.S = s3l::cell_edge(p->max_distance);
    const int par = (int)(ctx->vox_chunks & 1);
    const uint32_t maxp = (uint32_t)p->max_points;
    CK(ctx->aln.index(ctx->vox.view, par, ctx->vox_xyz, ctx->vox_nrm, run, nullptr, ctx->sm_count, ctx->stream,
                      &ctx->launches));
    CK(ctx->lattice.count(ctx->aln.view, ctx->vox.view, par, ctx->vox_nrm, p->max_distance, maxp, ctx->sm_count,
                          ctx->stream, &ctx->launches));
    SurfaceState st;
    int vox_overflow = 0;
    CK(cudaMemcpyAsync(&st, ctx->lattice.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&vox_overflow, &ctx->aln.state.get()->overflow, sizeof(int), cudaMemcpyDeviceToHost,
                       ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (vox_overflow)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more distinct voxels than max_voxels: begin again with a larger max_voxels");
    if (st.overflow || st.occupied > maxp)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more distinct lattice points than max_points: extract again with a larger max_points");
    if ((uint64_t)st.vertices * 6 > 0xffffffffull)   // the face count is a 32-bit sum of <= 6 per vertex
        return fail(ctx, SCAN3D_ERR_CONFIG, "more than (2^32 - 1) / 6 surface vertices");
    CK(ctx->surface.grow(st.vertices, st.faces));
    CK(ctx->lattice.emit(ctx->vox_rgb, st.vertices, ctx->surface, ctx->stream, &ctx->launches));
    ctx->surface.vertices = st.vertices;
    ctx->surface.faces = st.faces;
    ctx->results.produce(SURFACE);
    out->vertices = st.vertices;
    out->faces = st.faces;
    out->lattice_points = st.occupied;
    out->undefined_points = (int64_t)st.undefined;
    return SCAN3D_OK;
}

int scan3d_get_voxel_surface(scan3d_ctx* ctx, float* xyz, float* normals, uint8_t* rgb, int32_t* faces,
                             int64_t max_vertices, int64_t max_faces)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    CK(cudaSetDevice(ctx->device));
    const SurfaceMesh& s = ctx->surface;
    const int64_t nv = std::max<int64_t>(0, std::min(s.vertices, max_vertices));
    const int64_t nf = std::max<int64_t>(0, std::min(s.faces, max_faces));
    if (xyz && nv) CK(cudaMemcpyAsync(xyz, s.xyz, (size_t)nv * 12, cudaMemcpyDeviceToHost, ctx->stream));
    if (normals && nv) CK(cudaMemcpyAsync(normals, s.nrm, (size_t)nv * 12, cudaMemcpyDeviceToHost, ctx->stream));
    if (rgb && nv) CK(cudaMemcpyAsync(rgb, s.rgb, (size_t)nv * 3, cudaMemcpyDeviceToHost, ctx->stream));
    if (faces && nf) CK(cudaMemcpyAsync(faces, s.tri, (size_t)nf * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

int scan3d_write_voxel_surface_ply(scan3d_ctx* ctx, const char* path, int binary)
{
    if (!ctx || !path) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    const int64_t nv = ctx->surface.vertices, nf = ctx->surface.faces;
    std::vector<float> xyz((size_t)nv * 3), nrm((size_t)nv * 3);
    std::vector<uint8_t> rgb((size_t)nv * 3);
    std::vector<int32_t> faces((size_t)nf * 3);
    const int rc = scan3d_get_voxel_surface(ctx, xyz.data(), nrm.data(), rgb.data(), faces.data(), nv, nf);
    if (rc) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ctx, SCAN3D_ERR_IO, "cannot open PLY for writing");
    write_ply_with_faces(f, binary, nv, xyz.data(), nrm.data(), rgb.data(), nf, faces.data());
    const bool ok = fclose(f) == 0;
    return ok ? SCAN3D_OK : fail(ctx, SCAN3D_ERR_IO, "PLY write failed");
}

// ------------------------------------------------------------------------------------------
// connected components of a triangle mesh (include/scan3d.h has the exact rules)
// ------------------------------------------------------------------------------------------
int scan3d_voxel_surface_components(scan3d_ctx* ctx, const scan3d_components_params* p, scan3d_components_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!p || !out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (p->min_faces < 0 || p->max_components < 0) return fail(ctx, SCAN3D_ERR_ARG, "min_faces and max_components must be >= 0");
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(COMPONENTS);
    CK(ctx->cc.select(ctx->surface, (unsigned long long)p->min_faces, (unsigned long long)p->max_components,
                      ctx->stream, &ctx->launches));
    ComponentsState st;
    CK(cudaMemcpyAsync(&st, ctx->cc.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(ctx->spare.grow(st.vertices, st.faces));
    CK(ctx->cc.emit(ctx->surface, ctx->spare, ctx->stream, &ctx->launches));
    // the compacted set becomes the held surface; the old one is the next compaction's destination
    std::swap(ctx->surface, ctx->spare);
    ctx->surface.vertices = st.vertices;
    ctx->surface.faces = st.faces;
    ctx->cc_components = st.components;
    ctx->results.produce(COMPONENTS);
    out->components = st.components;
    out->kept = st.kept;
    out->vertices = st.vertices;
    out->faces = st.faces;
    out->largest_faces = st.largest;
    return SCAN3D_OK;
}

int scan3d_get_surface_components(scan3d_ctx* ctx, int64_t* vertices, int64_t* faces, uint8_t* kept,
                                  int64_t max_components)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!ctx->results.has(COMPONENTS))
        return fail(ctx, SCAN3D_ERR_STATE, "no component table of the held surface: call scan3d_voxel_surface_components");
    CK(cudaSetDevice(ctx->device));
    const int64_t n = std::max<int64_t>(0, std::min(ctx->cc_components, max_components));
    std::vector<uint32_t> v(vertices ? n : 0), f(faces ? n : 0);
    if (vertices && n) CK(cudaMemcpyAsync(v.data(), ctx->cc.comp_v, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (faces && n) CK(cudaMemcpyAsync(f.data(), ctx->cc.comp_f, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (kept && n) CK(cudaMemcpyAsync(kept, ctx->cc.kept, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int64_t c = 0; vertices && c < n; c++) vertices[c] = v[c];
    for (int64_t c = 0; faces && c < n; c++) faces[c] = f[c];
    return SCAN3D_OK;
}

int scan3d_mesh_components_dev(scan3d_ctx* ctx, const int32_t* faces_dev, int64_t n_faces, int64_t n_vertices,
                               int32_t* label_dev, int64_t* components_out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!components_out) return fail(ctx, SCAN3D_ERR_ARG, "null components_out");
    if (n_faces < 0 || n_faces >= (1LL << 31) || n_vertices < 0 || n_vertices >= (1LL << 31))
        return fail(ctx, SCAN3D_ERR_ARG, "n_faces and n_vertices must be in [0, 2^31)");
    if ((!faces_dev && n_faces > 0) || (!label_dev && n_vertices > 0)) return fail(ctx, SCAN3D_ERR_ARG, "null device pointer");
    if (((uintptr_t)faces_dev & 3) || ((uintptr_t)label_dev & 3))
        return fail(ctx, SCAN3D_ERR_ARG, "faces_dev and label_dev must be 4-byte aligned");
    CK(cudaSetDevice(ctx->device));
    CK(ctx->cc.labels(faces_dev, (uint32_t)n_faces, (uint32_t)n_vertices, label_dev, ctx->stream, &ctx->launches));
    ComponentsState st;
    CK(cudaMemcpyAsync(&st, ctx->cc.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st.bad) return fail(ctx, SCAN3D_ERR_ARG, "a face index outside [0, n_vertices)");
    *components_out = st.components;
    return SCAN3D_OK;
}

// ------------------------------------------------------------------------------------------
// simplification of the voxel surface (include/scan3d.h and common/scan3d_decimate_math.h have the exact rules)
// ------------------------------------------------------------------------------------------
int scan3d_voxel_surface_decimate(scan3d_ctx* ctx, float cell_size, scan3d_decimate_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!(cell_size - cell_size == 0.0f)) return fail(ctx, SCAN3D_ERR_ARG, "cell_size must be finite");
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    const double H = (double)cell_size, s = ctx->vox.view.S;
    if (!(H >= s && H <= s3q::RATIO_MAX * s))
        return fail(ctx, SCAN3D_ERR_ARG, "cell_size must be in [voxel_size, 256 voxel_size]");
    if (ctx->results.has(SIMPLIFIED))
        return fail(ctx, SCAN3D_ERR_STATE, "the held surface is already simplified: extract it again first");
    if (ctx->results.has(SMOOTHED))
        return fail(ctx, SCAN3D_ERR_STATE, "the held surface is smoothed: extract it again to simplify it");
    if (ctx->srf_filled_after_repair)
        return fail(ctx, SCAN3D_ERR_STATE, "the held surface was filled after a repair changed it: extract it again to "
                                           "simplify it");
    const int64_t nv = ctx->surface.vertices, nf = ctx->surface.faces;
    if (nf >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_CONFIG, "more than 2^31 - 1 surface faces");
    CK(cudaSetDevice(ctx->device));
    ctx->results.drop(COMPONENTS);
    // the emission runs before the synchronisation, so the spare set holds the whole input
    CK(ctx->spare.grow(std::max<int64_t>(nv, 1), std::max<int64_t>(nf, 1)));
    CK(ctx->dec.run(ctx->surface, H, ctx->spare, ctx->sm_count, ctx->stream, &ctx->launches));
    DecimateState st;
    VoxelState vst;
    CK(cudaMemcpyAsync(&st, ctx->dec.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&vst, ctx->dec.clusters.state, sizeof(vst), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // the simplified set becomes the held surface; the old one is the next compaction's destination
    std::swap(ctx->surface, ctx->spare);
    ctx->surface.vertices = vst.total[1];
    ctx->surface.faces = st.faces;
    ctx->results.produce(SIMPLIFIED);
    out->vertices = vst.total[1];
    out->faces = st.faces;
    out->collapsed_faces = st.collapsed;
    out->duplicate_faces = nf - st.collapsed - st.faces;
    out->mean_fallbacks = st.fallbacks;
    return SCAN3D_OK;
}

// ------------------------------------------------------------------------------------------
// smoothing of the voxel surface and of device meshes (include/scan3d.h and common/scan3d_smooth_math.h have the exact
// rules)
// ------------------------------------------------------------------------------------------
static int check_smooth_args(scan3d_ctx* ctx, const scan3d_smooth_params* p, scan3d_smooth_result* out)
{
    if (!p || !out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (p->iterations < 0 || p->iterations > SCAN3D_SMOOTH_MAX_ITERATIONS)
        return fail(ctx, SCAN3D_ERR_ARG, "iterations must be in [0, 4096]");
    if (!(p->lambda > 0.0f && p->lambda <= 1.0f)) return fail(ctx, SCAN3D_ERR_ARG, "lambda must be in (0, 1]");
    if (!(p->mu >= -1.0f && p->mu <= 0.0f)) return fail(ctx, SCAN3D_ERR_ARG, "mu must be in [-1, 0]");
    return SCAN3D_OK;
}

// smooths the mesh (xyz, nrm, faces) into xyz_out / nrm_out (the same buffers or others; nrm and nrm_out may be null);
// one synchronisation; on an error found on the device nothing is written
static int smooth_run(scan3d_ctx* ctx, const float* xyz, const float* nrm, const int32_t* faces, int64_t nv, int64_t nf,
                      const scan3d_smooth_params* p, float* xyz_out, float* nrm_out, scan3d_smooth_result* out)
{
    if (6 * nf >= (1LL << 32)) return fail(ctx, SCAN3D_ERR_CONFIG, "more than (2^32 - 1) / 6 faces");
    const int passes = p->iterations * (p->mu == 0.0f ? 1 : 2);
    CK(ctx->smooth.run(xyz, nrm, faces, (uint32_t)nv, (uint32_t)nf, passes, (double)p->lambda, (double)p->mu, xyz_out,
                       nrm_out, ctx->stream, &ctx->launches));
    SmoothState st;
    CK(cudaMemcpyAsync(&st, ctx->smooth.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st.bad) return fail(ctx, SCAN3D_ERR_ARG, "a coordinate that is not finite or a face index outside [0, n_vertices)");
    if (st.overflow)
        return fail(ctx, SCAN3D_ERR_CONFIG,
                    "a free vertex with more than 2^20 neighbours, or moved beyond the fixed-point limit");
    out->vertices = nv;
    out->faces = nf;
    out->held_vertices = st.held;
    out->isolated_vertices = st.isolated;
    out->passes = passes;
    double move;
    memcpy(&move, &st.max_move, sizeof(move));
    out->max_displacement = move;
    return SCAN3D_OK;
}

int scan3d_voxel_surface_smooth(scan3d_ctx* ctx, const scan3d_smooth_params* p, scan3d_smooth_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    int rc = check_smooth_args(ctx, p, out);
    if (rc) return rc;
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    CK(cudaSetDevice(ctx->device));
    SurfaceMesh &s = ctx->surface, &spare = ctx->spare;
    CK(spare.grow_positions(std::max<int64_t>(s.vertices, 1)));
    rc = smooth_run(ctx, s.xyz, s.nrm, s.tri, s.vertices, s.faces, p, spare.xyz, spare.nrm, out);
    if (rc) return rc;
    // the smoothed positions and normals become the held surface; faces, colours and the vertex order are unchanged
    std::swap(s.xyz, spare.xyz);
    std::swap(s.nrm, spare.nrm);
    ctx->results.produce(SMOOTHED);
    return SCAN3D_OK;
}

int scan3d_mesh_smooth_dev(scan3d_ctx* ctx, float* xyz_dev, float* normals_dev, int64_t n_vertices,
                           const int32_t* faces_dev, int64_t n_faces, const scan3d_smooth_params* p,
                           scan3d_smooth_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    const int rc = check_smooth_args(ctx, p, out);
    if (rc) return rc;
    if (n_faces < 0 || n_faces >= (1LL << 31) || n_vertices < 0 || n_vertices >= (1LL << 31))
        return fail(ctx, SCAN3D_ERR_ARG, "n_faces and n_vertices must be in [0, 2^31)");
    if ((!xyz_dev && n_vertices > 0) || (!faces_dev && n_faces > 0)) return fail(ctx, SCAN3D_ERR_ARG, "null device pointer");
    if (((uintptr_t)xyz_dev & 3) || ((uintptr_t)normals_dev & 3) || ((uintptr_t)faces_dev & 3))
        return fail(ctx, SCAN3D_ERR_ARG, "xyz_dev, normals_dev and faces_dev must be 4-byte aligned");
    CK(cudaSetDevice(ctx->device));
    return smooth_run(ctx, xyz_dev, normals_dev, faces_dev, n_vertices, n_faces, p, xyz_dev, normals_dev, out);
}

// ------------------------------------------------------------------------------------------
// hole filling of the voxel surface and of device meshes (include/scan3d.h and common/scan3d_fill_math.h have the
// exact rules)
// ------------------------------------------------------------------------------------------
// finds the holes of the mesh (the first synchronisation) into *st; the faces the holes can add into *most
static int fill_count(scan3d_ctx* ctx, const float* xyz, const int32_t* faces, int64_t nv, int64_t nf,
                      int32_t max_edges, FillState* st, int64_t* most)
{
    if (6 * nf >= (1LL << 32)) return fail(ctx, SCAN3D_ERR_CONFIG, "more than (2^32 - 1) / 6 faces");
    CK(ctx->fill.count(xyz, faces, (uint32_t)nv, (uint32_t)nf, (uint32_t)max_edges, ctx->stream, &ctx->launches));
    CK(cudaMemcpyAsync(st, ctx->fill.state, sizeof(*st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st->bad) return fail(ctx, SCAN3D_ERR_ARG, "a coordinate that is not finite or a face index outside [0, n_vertices)");
    if (st->cells64 >= (1ULL << 32)) return fail(ctx, SCAN3D_ERR_CONFIG, "the holes need 2^32 DP cells or more");
    *most = (int64_t)st->loop_edges - 2 * (int64_t)st->holes;
    if (nf + *most >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_CONFIG, "the filled mesh could have 2^31 faces or more");
    return SCAN3D_OK;
}

// triangulates the holes found by fill_count and writes the added faces to faces_out unless there are more than
// capacity (the second synchronisation); fills *out
static int fill_finish(scan3d_ctx* ctx, const FillState& counts, const float* xyz, const int32_t* faces, int64_t nv,
                       int64_t nf, int32_t* faces_out, int64_t capacity, scan3d_fill_result* out)
{
    CK(ctx->fill.fill(counts, xyz, faces, (uint32_t)nv, faces_out, (uint64_t)capacity, ctx->stream, &ctx->launches));
    FillState st;
    CK(cudaMemcpyAsync(&st, ctx->fill.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const bool fits = st.added <= (uint64_t)capacity;
    out->vertices = nv;
    out->faces = nf + (fits ? st.added : 0);
    out->boundary_edges = st.boundary;
    out->holes = st.holes;
    out->filled = st.filled;
    out->faces_added = st.added;
    // a filled hole of n edges adds n - 2 faces and closes its n hole edges
    out->open_edges = (int64_t)st.boundary - (fits ? (int64_t)st.added + 2 * (int64_t)st.filled : 0);
    if (!fits) return fail(ctx, SCAN3D_ERR_CONFIG, "more added faces than max_faces_out: call again with faces_added");
    return SCAN3D_OK;
}

int scan3d_voxel_surface_fill_holes(scan3d_ctx* ctx, int32_t max_edges, scan3d_fill_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    // an unrefined surface stays decimatable only with holes of at most SCAN3D_FILL_NETS_MAX_EDGES edges
    const bool refined = ctx->results.has(SIMPLIFIED) || ctx->results.has(SMOOTHED);
    const int32_t cap = refined ? SCAN3D_FILL_MAX_EDGES : SCAN3D_FILL_NETS_MAX_EDGES;
    if (max_edges < 3 || max_edges > cap)
        return fail(ctx, SCAN3D_ERR_ARG, refined ? "max_edges must be in [3, 1024]"
                                                 : "max_edges must be in [3, 22] on a surface that is neither "
                                                   "simplified nor smoothed");
    CK(cudaSetDevice(ctx->device));
    SurfaceMesh &s = ctx->surface, &spare = ctx->spare;
    const int64_t nv = s.vertices, nf = s.faces;
    ctx->results.drop(COMPONENTS);
    FillState counts;
    int64_t most = 0;
    int rc = fill_count(ctx, s.xyz, s.tri, nv, nf, max_edges, &counts, &most);
    if (rc) return rc;
    // the held faces, then the added ones, into the spare face set, which becomes the held one
    CK(spare.tri.ensure(3 * (size_t)std::max<int64_t>(nf + most, 1)));
    if (nf) CK(cudaMemcpyAsync(spare.tri, s.tri, (size_t)nf * 12, cudaMemcpyDeviceToDevice, ctx->stream));
    rc = fill_finish(ctx, counts, s.xyz, s.tri, nv, nf, spare.tri.get() + 3 * nf, most, out);
    if (rc) return rc;
    std::swap(s.tri, spare.tri);
    s.faces = out->faces;
    if (out->faces_added && ctx->srf_repaired) ctx->srf_filled_after_repair = true;
    return SCAN3D_OK;
}

int scan3d_mesh_fill_holes_dev(scan3d_ctx* ctx, const float* xyz_dev, int64_t n_vertices, const int32_t* faces_dev,
                               int64_t n_faces, int32_t max_edges, int32_t* faces_out_dev, int64_t max_faces_out,
                               scan3d_fill_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (max_edges < 3 || max_edges > SCAN3D_FILL_MAX_EDGES) return fail(ctx, SCAN3D_ERR_ARG, "max_edges must be in [3, 1024]");
    if (n_faces < 0 || n_faces >= (1LL << 31) || n_vertices < 0 || n_vertices >= (1LL << 31) || max_faces_out < 0 ||
        max_faces_out >= (1LL << 31))
        return fail(ctx, SCAN3D_ERR_ARG, "n_vertices, n_faces and max_faces_out must be in [0, 2^31)");
    if ((!xyz_dev && n_vertices > 0) || (!faces_dev && n_faces > 0) || (!faces_out_dev && max_faces_out > 0))
        return fail(ctx, SCAN3D_ERR_ARG, "null device pointer");
    if (((uintptr_t)xyz_dev & 3) || ((uintptr_t)faces_dev & 3) || ((uintptr_t)faces_out_dev & 3))
        return fail(ctx, SCAN3D_ERR_ARG, "xyz_dev, faces_dev and faces_out_dev must be 4-byte aligned");
    CK(cudaSetDevice(ctx->device));
    FillState counts;
    int64_t most = 0;
    const int rc = fill_count(ctx, xyz_dev, faces_dev, n_vertices, n_faces, max_edges, &counts, &most);
    if (rc) return rc;
    return fill_finish(ctx, counts, xyz_dev, faces_dev, n_vertices, n_faces, faces_out_dev, max_faces_out, out);
}

// ------------------------------------------------------------------------------------------
// repair of the non-manifold edges and vertices of the voxel surface and of device meshes (include/scan3d.h and
// common/scan3d_repair_math.h have the exact rules)
// ------------------------------------------------------------------------------------------
static int check_repair_flags(scan3d_ctx* ctx, int32_t flags, scan3d_repair_result* out)
{
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (flags <= 0 || (flags & ~(SCAN3D_REPAIR_FACES | SCAN3D_REPAIR_VERTICES)))
        return fail(ctx, SCAN3D_ERR_ARG, "flags must be a non-empty combination of SCAN3D_REPAIR_FACES and "
                                         "SCAN3D_REPAIR_VERTICES");
    return SCAN3D_OK;
}

// finds the drops and the fans of the mesh (the first synchronisation) and fills *out
static int repair_count(scan3d_ctx* ctx, const float* xyz, const int32_t* faces, int64_t nv, int64_t nf, int32_t flags,
                        scan3d_repair_result* out)
{
    if (3 * nf >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_CONFIG, "3 n_faces must be below 2^31");
    CK(ctx->repair.count(xyz, faces, (uint32_t)nv, (uint32_t)nf, flags, ctx->stream, &ctx->launches));
    RepairState st;
    CK(cudaMemcpyAsync(&st, ctx->repair.state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st.bad) return fail(ctx, SCAN3D_ERR_ARG, "a coordinate that is not finite or a face index outside [0, n_vertices)");
    out->vertices = nv + st.added;
    out->faces = st.faces;
    out->degenerate_faces = st.degenerate;
    out->duplicate_faces = st.duplicate;
    out->nonmanifold_edges = st.nonmanifold_edges;
    out->nonmanifold_faces = st.nonmanifold_faces;
    out->split_vertices = st.split;
    out->vertices_added = st.added;
    out->boundary_edges = st.boundary;
    out->inconsistent_edges = st.inconsistent;
    if (out->vertices >= (1LL << 31)) return fail(ctx, SCAN3D_ERR_CONFIG, "the repaired mesh would have 2^31 vertices or more");
    return SCAN3D_OK;
}

int scan3d_voxel_surface_repair(scan3d_ctx* ctx, int32_t flags, scan3d_repair_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    int rc = check_repair_flags(ctx, flags, out);
    if (rc) return rc;
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    CK(cudaSetDevice(ctx->device));
    SurfaceMesh &s = ctx->surface, &spare = ctx->spare;
    const int64_t nv = s.vertices, nf = s.faces;
    ctx->results.drop(COMPONENTS);
    rc = repair_count(ctx, s.xyz, s.tri, nv, nf, flags, out);
    if (rc) return rc;
    // the held vertices, the copies after them and the kept faces into the spare set, which becomes the held one
    const int64_t added = out->vertices_added;
    CK(spare.grow(std::max<int64_t>(nv + added, 1), std::max<int64_t>(out->faces, 1)));
    CK(ctx->repair.source.ensure(std::max<int64_t>(added, 1)));
    if (nv) {
        CK(cudaMemcpyAsync(spare.xyz, s.xyz, (size_t)nv * 12, cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaMemcpyAsync(spare.nrm, s.nrm, (size_t)nv * 12, cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaMemcpyAsync(spare.rgb, s.rgb, (size_t)nv * 3, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    CK(ctx->repair.emit(s.tri, (uint32_t)nv, (uint32_t)nf, flags, spare.tri, ctx->repair.source, s.xyz,
                        s.nrm, s.rgb, spare.xyz, spare.nrm, spare.rgb, ctx->stream, &ctx->launches));
    CK(cudaStreamSynchronize(ctx->stream));
    std::swap(s, spare);
    s.vertices = out->vertices;
    s.faces = out->faces;
    if (out->faces < nf || added) ctx->srf_repaired = true;
    return SCAN3D_OK;
}

int scan3d_mesh_repair_dev(scan3d_ctx* ctx, const float* xyz_dev, int64_t n_vertices, const int32_t* faces_dev,
                           int64_t n_faces, int32_t flags, int32_t* faces_out_dev, int32_t* source_out_dev,
                           int64_t max_source_out, scan3d_repair_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    int rc = check_repair_flags(ctx, flags, out);
    if (rc) return rc;
    if (n_faces < 0 || n_faces >= (1LL << 31) || n_vertices < 0 || n_vertices >= (1LL << 31) || max_source_out < 0 ||
        max_source_out >= (1LL << 31))
        return fail(ctx, SCAN3D_ERR_ARG, "n_vertices, n_faces and max_source_out must be in [0, 2^31)");
    if ((!xyz_dev && n_vertices > 0) || (!faces_dev && n_faces > 0) || (!faces_out_dev && n_faces > 0) ||
        (!source_out_dev && max_source_out > 0))
        return fail(ctx, SCAN3D_ERR_ARG, "null device pointer");
    if (((uintptr_t)xyz_dev & 3) || ((uintptr_t)faces_dev & 3) || ((uintptr_t)faces_out_dev & 3) ||
        ((uintptr_t)source_out_dev & 3))
        return fail(ctx, SCAN3D_ERR_ARG, "xyz_dev, faces_dev, faces_out_dev and source_out_dev must be 4-byte aligned");
    if (faces_out_dev && faces_out_dev == faces_dev) return fail(ctx, SCAN3D_ERR_ARG, "faces_out_dev must not be faces_dev");
    CK(cudaSetDevice(ctx->device));
    rc = repair_count(ctx, xyz_dev, faces_dev, n_vertices, n_faces, flags, out);
    if (rc) return rc;
    if (out->vertices_added > max_source_out)
        return fail(ctx, SCAN3D_ERR_CONFIG, "more added vertices than max_source_out: call again with vertices_added");
    CK(ctx->repair.emit(faces_dev, (uint32_t)n_vertices, (uint32_t)n_faces, flags, faces_out_dev, source_out_dev,
                        nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, ctx->stream, &ctx->launches));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

// ------------------------------------------------------------------------------------------
// coherent orientation and measures of the voxel surface and of device meshes (include/scan3d.h and
// common/scan3d_orient_math.h have the exact rules)
// ------------------------------------------------------------------------------------------
static int check_mesh_args(scan3d_ctx* ctx, const float* xyz, const float* nrm, int64_t nv, const int32_t* faces,
                           int64_t nf)
{
    if (nf < 0 || nf >= (1LL << 31) || nv < 0 || nv >= (1LL << 31))
        return fail(ctx, SCAN3D_ERR_ARG, "n_vertices and n_faces must be in [0, 2^31)");
    if ((!xyz && nv > 0) || (!faces && nf > 0)) return fail(ctx, SCAN3D_ERR_ARG, "null device pointer");
    if (((uintptr_t)xyz & 3) || ((uintptr_t)nrm & 3) || ((uintptr_t)faces & 3))
        return fail(ctx, SCAN3D_ERR_ARG, "xyz_dev, normals_dev and faces_dev must be 4-byte aligned");
    return SCAN3D_OK;
}

// the counting pass over the mesh and, with apply, the flips into faces_out and nrm; one synchronisation
static int orient_run(scan3d_ctx* ctx, const float* xyz, float* nrm, const int32_t* faces, bool apply,
                      int32_t* faces_out, int64_t nv, int64_t nf, OrientState* st)
{
    if (6 * nf >= (1LL << 32)) return fail(ctx, SCAN3D_ERR_CONFIG, "more than (2^32 - 1) / 6 faces");
    CK(ctx->orient.count(xyz, faces, (uint32_t)nv, (uint32_t)nf, ctx->stream, &ctx->launches));
    if (apply) CK(ctx->orient.apply(faces_out, nrm, (uint32_t)nv, (uint32_t)nf, ctx->stream, &ctx->launches));
    CK(cudaMemcpyAsync(st, ctx->orient.state, sizeof(*st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st->bad) return fail(ctx, SCAN3D_ERR_ARG, "a coordinate that is not finite or a face index outside [0, n_vertices)");
    return SCAN3D_OK;
}

static int orient_mesh(scan3d_ctx* ctx, const float* xyz, float* nrm, int32_t* faces, int64_t nv, int64_t nf,
                       scan3d_orient_result* out)
{
    OrientState st;
    const int rc = orient_run(ctx, xyz, nrm, faces, true, faces, nv, nf, &st);
    if (rc) return rc;
    out->vertices = nv;
    out->faces = nf;
    out->degenerate_faces = st.degenerate;
    out->patches = st.patches;
    out->closed_patches = st.closed;
    out->nonorientable_patches = st.nonorientable;
    out->flipped_faces = st.flipped;
    out->flipped_normals = st.flipped_normals;
    out->inconsistent_edges_before = st.inconsistent;
    out->inconsistent_edges = st.inconsistent_after;
    return SCAN3D_OK;
}

static int measure_mesh(scan3d_ctx* ctx, const float* xyz, const int32_t* faces, int64_t nv, int64_t nf,
                        scan3d_measure_result* out)
{
    OrientState st;
    const int rc = orient_run(ctx, xyz, nullptr, faces, false, nullptr, nv, nf, &st);
    if (rc) return rc;
    const int64_t live = nf - (int64_t)st.degenerate;
    out->vertices = nv;
    out->faces = nf;
    out->degenerate_faces = st.degenerate;
    out->patches = st.patches;
    out->closed_patches = st.closed;
    out->nonorientable_patches = st.nonorientable;
    out->unreferenced_vertices = nv - (int64_t)st.referenced;
    out->edges = st.edges;
    out->boundary_edges = st.boundary;
    out->nonmanifold_edges = st.nonmanifold;
    out->inconsistent_edges = st.inconsistent;
    out->euler_characteristic = (int64_t)st.referenced - (int64_t)st.edges + live;
    out->watertight = live > 0 && st.boundary == 0 && st.nonmanifold == 0 && st.inconsistent == 0;
    const int E = s3o::exponent(st.exp_field);
    out->area = s3o::area(st.area[0], st.area[1], E);
    out->volume = s3o::volume(st.volume[0], st.volume[1], E);
    for (int k = 0; k < 3; k++) {
        uint32_t lo = 0, hi = 0;                         // +0.0f without a referenced vertex
        if (st.referenced) {
            lo = s3o::key_bits(st.box_lo[k]);
            hi = s3o::key_bits(st.box_hi[k]);
        }
        memcpy(&out->bbox_min[k], &lo, 4);
        memcpy(&out->bbox_max[k], &hi, 4);
    }
    return SCAN3D_OK;
}

int scan3d_voxel_surface_orient(scan3d_ctx* ctx, scan3d_orient_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    CK(cudaSetDevice(ctx->device));
    SurfaceMesh& s = ctx->surface;
    // faces and normals change in place; the vertex and face sets, and so every result, stay current
    const int rc = orient_mesh(ctx, s.xyz, s.nrm, s.tri, s.vertices, s.faces, out);
    if (rc) return rc;
    if (out->flipped_faces) ctx->srf_repaired = true;
    return SCAN3D_OK;
}

int scan3d_mesh_orient_dev(scan3d_ctx* ctx, const float* xyz_dev, float* normals_dev, int64_t n_vertices,
                           int32_t* faces_dev, int64_t n_faces, scan3d_orient_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    const int rc = check_mesh_args(ctx, xyz_dev, normals_dev, n_vertices, faces_dev, n_faces);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    return orient_mesh(ctx, xyz_dev, normals_dev, faces_dev, n_vertices, n_faces, out);
}

int scan3d_voxel_surface_measure(scan3d_ctx* ctx, scan3d_measure_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (!ctx->results.has(SURFACE))
        return fail(ctx, SCAN3D_ERR_STATE, "no surface of the current voxel outputs: call scan3d_voxel_surface");
    CK(cudaSetDevice(ctx->device));
    const SurfaceMesh& s = ctx->surface;
    return measure_mesh(ctx, s.xyz, s.tri, s.vertices, s.faces, out);
}

int scan3d_mesh_measure_dev(scan3d_ctx* ctx, const float* xyz_dev, int64_t n_vertices, const int32_t* faces_dev,
                            int64_t n_faces, scan3d_measure_result* out)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    if (!out) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    const int rc = check_mesh_args(ctx, xyz_dev, nullptr, n_vertices, faces_dev, n_faces);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    return measure_mesh(ctx, xyz_dev, faces_dev, n_vertices, n_faces, out);
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
    CK(ctx->pattern_profiles.ensure(2 * max_prof));
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
    DeviceBuffer<uint8_t> d;
    CK(d.ensure((size_t)bytes));
    const int rc = scan3d_generate_patterns_dev(ctx, dir, d);
    if (rc) return rc;
    CK(cudaMemcpyAsync(patterns_host, d, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
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
    DeviceBuffer<double> dy, dx;
    DeviceBuffer<float> dout;
    CK(dy.ensure((size_t)n));
    CK(dx.ensure((size_t)n));
    CK(dout.ensure((size_t)n));
    CK(cudaMemcpyAsync(dy, y_host, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dx, x_host, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_debug_atan2(dy, dx, dout, n, mode, ctx->atan_tab, ctx->stream));
    ctx->launches++;
    CK(cudaMemcpyAsync(out_host, dout, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
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
    DeviceBuffer<unsigned long long> d;
    CK(d.ensure(1));
    unsigned long long h = 0;
    CK(cudaMemsetAsync(d, 0, 8, ctx->stream));
    CK(launch_debug_divcheck(d, ctx->stream));
    ctx->launches++;
    CK(cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *mismatches = h;
    return SCAN3D_OK;
}

}  // extern "C"
