// scan3d_aux_api.cu -- C ABI entries for the steps either side of the reconstruction path
// (include/scan3d.h, "either side of the path"): capture-side cvUndistort2, image_scissor's ROI fill,
// register_point_clouds' transform.  GPU only, like the rest of the library.
#include <stdlib.h>
#include <string.h>

#include <string>
#include <utility>

#include "scan3d_internal.h"
#include "../common/scan3d_aux_math.h"

using namespace s3d;

// frame shape of the device whose images are undistorted: 0 = camera, 1 = projector
static int kind_shape(scan3d_ctx* ctx, int kind, int* W, int* H)
{
    if (kind != 0 && kind != 1) return fail(ctx, SCAN3D_ERR_ARG, "device_kind must be 0 (camera) or 1 (projector)");
    if (!ctx->has_calib) return fail(ctx, SCAN3D_ERR_STATE, "calibration not set");
    if (kind == 0) {
        if (ctx->cfg.row0 != 0 || ctx->cfg.H_total != ctx->cfg.H)
            return fail(ctx, SCAN3D_ERR_CONFIG, "capture-side undistortion needs the whole frame (row-sharded ctx)");
        *W = ctx->cfg.W; *H = ctx->cfg.H;
    } else {
        if (ctx->cfg.PW < 1 || ctx->cfg.PH < 1) return fail(ctx, SCAN3D_ERR_CONFIG, "projector size not configured");
        *W = ctx->cfg.PW; *H = ctx->cfg.PH;
    }
    return SCAN3D_OK;
}

static int ensure_map(scan3d_ctx* ctx, int kind, int W, int H)
{
    if (ctx->undist_xy[kind]) return SCAN3D_OK;
    const size_t n = (size_t)W * H;
    DeviceBuffer<short2> xy;
    DeviceBuffer<uint16_t> frac;
    const double* K = kind == 0 ? ctx->hcal.Kc : ctx->hcal.Kp;
    const double* d = kind == 0 ? ctx->hcal.dc : ctx->hcal.dp;
    cudaError_t e = xy.ensure(n);
    if (e == cudaSuccess) e = frac.ensure(n);
    if (e == cudaSuccess) e = launch_undistort_map(K, d, W, H, xy, frac, ctx->stream);
    if (e != cudaSuccess) {      // both maps or none: a half-built pair must never look usable
        cudaGetLastError();
        ctx->err = std::string("undistortion map: ") + cudaGetErrorString(e);
        return SCAN3D_ERR_CUDA;
    }
    ctx->undist_xy[kind] = std::move(xy);
    ctx->undist_frac[kind] = std::move(frac);
    ctx->launches++;
    return SCAN3D_OK;
}

extern "C" {

int scan3d_undistort_frames_dev(scan3d_ctx* ctx, int device_kind, const uint8_t* src_dev, int n_frames, uint8_t* dst_dev)
{
    if (!ctx || !src_dev || !dst_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (n_frames < 0) return fail(ctx, SCAN3D_ERR_ARG, "negative frame count");
    if (src_dev == dst_dev) return fail(ctx, SCAN3D_ERR_ARG, "undistortion cannot run in place");
    int W, H;
    int rc = kind_shape(ctx, device_kind, &W, &H);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ensure_map(ctx, device_kind, W, H);
    if (rc) return rc;
    if (n_frames == 0) return SCAN3D_OK;
    CK(launch_remap_frames(src_dev, dst_dev, ctx->undist_xy[device_kind], ctx->undist_frac[device_kind], W, H, n_frames,
                           ctx->sm_count, ctx->stream));
    ctx->launches++;
    return SCAN3D_OK;
}

int scan3d_undistort_frames(scan3d_ctx* ctx, int device_kind, const uint8_t* src_host, int n_frames, uint8_t* dst_host)
{
    if (!ctx || !src_host || !dst_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (n_frames < 0) return fail(ctx, SCAN3D_ERR_ARG, "negative frame count");
    int W, H;
    int rc = kind_shape(ctx, device_kind, &W, &H);
    if (rc) return rc;
    if (n_frames == 0) return SCAN3D_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)W * H * n_frames;
    DeviceBuffer<uint8_t> buf;
    CK(buf.ensure(2 * bytes));
    CK(cudaMemcpyAsync(buf, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    rc = scan3d_undistort_frames_dev(ctx, device_kind, buf, n_frames, buf + bytes);
    if (rc) return rc;
    CK(cudaMemcpyAsync(dst_host, buf + bytes, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

int scan3d_get_undistort_map(scan3d_ctx* ctx, int device_kind, int16_t* xy_host, uint16_t* frac_host)
{
    if (!ctx) return SCAN3D_ERR_ARG;
    int W, H;
    int rc = kind_shape(ctx, device_kind, &W, &H);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ensure_map(ctx, device_kind, W, H);
    if (rc) return rc;
    const size_t n = (size_t)W * H;
    if (xy_host) CK(cudaMemcpyAsync(xy_host, ctx->undist_xy[device_kind], n * sizeof(short2), cudaMemcpyDeviceToHost, ctx->stream));
    if (frac_host) CK(cudaMemcpyAsync(frac_host, ctx->undist_frac[device_kind], n * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

int scan3d_roi_fill_dev(scan3d_ctx* ctx, const uint8_t* outline_dev, uint8_t* roi_dev, uint8_t* filled_dev)
{
    if (!ctx || !outline_dev || !roi_dev) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (roi_dev == outline_dev || (filled_dev && filled_dev == roi_dev))
        return fail(ctx, SCAN3D_ERR_ARG, "the ROI plane must be a separate buffer");
    CK(cudaSetDevice(ctx->device));
    CK(launch_roi_fill(outline_dev, ctx->cfg.W, ctx->cfg.H_total, roi_dev, filled_dev, ctx->stream));
    ctx->launches++;
    return SCAN3D_OK;
}

int scan3d_roi_fill(scan3d_ctx* ctx, const uint8_t* outline_host, uint8_t* roi_host, uint8_t* filled_host)
{
    if (!ctx || !outline_host || !roi_host) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->cfg.W * ctx->cfg.H_total;
    DeviceBuffer<uint8_t> buf;
    CK(buf.ensure(2 * n));
    CK(cudaMemcpyAsync(buf, outline_host, n, cudaMemcpyHostToDevice, ctx->stream));
    const int rc = scan3d_roi_fill_dev(ctx, buf, buf + n, filled_host ? buf.get() : nullptr);   // outline filled in place, like the reference
    if (rc) return rc;
    CK(cudaMemcpyAsync(roi_host, buf + n, n, cudaMemcpyDeviceToHost, ctx->stream));
    if (filled_host) CK(cudaMemcpyAsync(filled_host, buf, n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

int scan3d_register_rotation(float theta_deg, float R[16])
{
    if (!R) return SCAN3D_ERR_ARG;
    s3a::register_rotation(theta_deg, R);
    return SCAN3D_OK;
}

int scan3d_register_points_dev(scan3d_ctx* ctx, const float* src_dev, float* dst_dev, int64_t n, float theta_deg, float tx,
                               float ty, float tz)
{
    if (!ctx || (n > 0 && (!src_dev || !dst_dev))) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (n < 0) return fail(ctx, SCAN3D_ERR_ARG, "negative point count");
    if (n == 0) return SCAN3D_OK;
    CK(cudaSetDevice(ctx->device));
    float R[16];
    s3a::register_rotation(theta_deg, R);
    CK(launch_register_points(src_dev, dst_dev, (long long)n, R, tx, ty, tz, ctx->sm_count, ctx->stream));
    ctx->launches++;
    return SCAN3D_OK;
}

int scan3d_register_points(scan3d_ctx* ctx, const float* src_host, float* dst_host, int64_t n, float theta_deg, float tx,
                           float ty, float tz)
{
    if (!ctx || (n > 0 && (!src_host || !dst_host))) return fail(ctx, SCAN3D_ERR_ARG, "null argument");
    if (n < 0) return fail(ctx, SCAN3D_ERR_ARG, "negative point count");
    if (n == 0) return SCAN3D_OK;
    CK(cudaSetDevice(ctx->device));
    DeviceBuffer<float> buf;
    CK(buf.ensure(3 * (size_t)n));
    CK(cudaMemcpyAsync(buf, src_host, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    const int rc = scan3d_register_points_dev(ctx, buf, buf, n, theta_deg, tx, ty, tz);   // element-wise: in place is fine
    if (rc) return rc;
    CK(cudaMemcpyAsync(dst_host, buf, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SCAN3D_OK;
}

}  // extern "C"
