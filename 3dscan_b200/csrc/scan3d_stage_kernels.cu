// scan3d_stage_kernels.cu -- one plain kernel per reference stage (any frame shape).  These back
// the stage-by-stage C ABI (scan3d_compute_wrapped_phase ... scan3d_compact_points) and are the
// shape-generic path; the benchmarked single-pass kernel lives in scan3d_fused_kernel7.cu.
#include <math.h>

#include "scan3d_internal.h"

namespace s3d {

static inline unsigned cdiv(long a, long b) { return (unsigned)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------
// mask: ROI -> valid after the raster recurrence (3/wrapped_phase.cpp:106-115 + :266-279)
// ------------------------------------------------------------------------------------------
__global__ void k_mask(const uint8_t* __restrict__ roi, uint8_t* __restrict__ mask, int W, int H,
                       int row0, int H_total)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int yl = blockIdx.y;
    if (x >= W || yl >= H) return;
    const int y = row0 + yl;
    auto inv = [&](int qx, int qy) { return roi[(size_t)qy * W + qx] == 0; };
    bool v = !inv(x, y);
    const bool border = x == 0 || y == 0 || x == W - 1 || y == H_total - 1;
    if (v && !border) v = !mask_trigger(x, y, W, H_total, inv);
    mask[(size_t)yl * W + x] = v ? 1 : 0;
}

// ------------------------------------------------------------------------------------------
// optional modulation criterion (3/wrapped_phase.cpp:84-104, disabled in the reference):
// roi_eff = roi && gamma > 0.01, arithmetic as written there (see oracle/scan3d_oracle.c)
// ------------------------------------------------------------------------------------------
__global__ void k_modulation_roi(const uint8_t* __restrict__ fringe, const uint8_t* __restrict__ roi,
                                 uint8_t* __restrict__ roi_eff, size_t n)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int i0 = fringe[i], i1 = fringe[n + i], i2 = fringe[2 * n + i];
    const int d = i0 - i2, e = 2 * i1 - i0 - i2;
    const float t1 = __fsqrt_rn((float)(3 * d * d + e * e));      // exact integer below 2^24
    const float t2 = (float)(i0 + i1 + i2);
    const float t3 = __fdiv_rn(t1, t2);                            // 0/0 -> NaN -> rejected
    roi_eff[i] = ((double)t3 > 0.01 && roi[i] != 0) ? 1 : 0;
}

// SCAN3D_FLAG_STRICT_REFERENCE: the ROI as check_I_mod_criteria reads it as committed (3/wrapped_phase.cpp:106-115)
__global__ void k_strict_roi(const uint8_t* __restrict__ roi, uint8_t* __restrict__ roi_eff, size_t n, int n_is_3_or_4)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) roi_eff[i] = (n_is_3_or_4 && roi[i] == 1) ? 1 : 0;
}

cudaError_t launch_strict_roi(const uint8_t* roi, uint8_t* roi_eff, size_t n, int N, cudaStream_t st)
{
    k_strict_roi<<<(unsigned)cdiv((long long)n, 256), 256, 0, st>>>(roi, roi_eff, n, N == 3 || N == 4);
    return cudaGetLastError();
}

cudaError_t launch_modulation_roi(const Shape& s, const uint8_t* fringe, const uint8_t* roi, uint8_t* roi_eff, cudaStream_t st)
{
    const size_t n = (size_t)s.W * s.H;
    k_modulation_roi<<<(unsigned)cdiv((long long)n, 256), 256, 0, st>>>(fringe, roi, roi_eff, n);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// projector patterns (1/pattern_generator.cpp): a pattern is constant along its stripes, so each
// image is its 1-D profile (host, exact libm: common/scan3d_pattern_profile.h) expanded across
// the other axis.  Pure write stream: 16 bytes per thread, PW % 16 == 0.
// ------------------------------------------------------------------------------------------
constexpr int PATTERN_ROWS_PER_BLOCK = 32;
__global__ void k_expand_patterns(const uint8_t* __restrict__ profiles, int profile_len, int n_patterns,
                                  uint8_t* __restrict__ out, int PW, int PH, int dir)
{
    const int x16 = blockIdx.x * blockDim.x + threadIdx.x;       // 16-pixel group along the row
    const int p = blockIdx.z;
    if (x16 * 16 >= PW) return;
    const uint8_t* prof = profiles + (size_t)p * profile_len;
    const int y0 = blockIdx.y * PATTERN_ROWS_PER_BLOCK, y1 = min(PH, y0 + PATTERN_ROWS_PER_BLOCK);
    uint4* dst = reinterpret_cast<uint4*>(out + ((size_t)p * PH + y0) * PW + 16 * x16);
    const int pitch = PW / 16;
    if (dir == 0) {
        const uint4 v = *reinterpret_cast<const uint4*>(prof + 16 * x16);    // vertical stripes: value = f(column)
        for (int y = y0; y < y1; y++, dst += pitch) __stcs(dst, v);
    } else {
        for (int y = y0; y < y1; y++, dst += pitch) {
            const uint32_t b = prof[y] * 0x01010101u;                        // horizontal stripes: value = f(row)
            __stcs(dst, make_uint4(b, b, b, b));
        }
    }
}

cudaError_t launch_expand_patterns(const uint8_t* profiles, int profile_len, int n_patterns, uint8_t* out, int PW, int PH,
                                   int dir, cudaStream_t st)
{
    dim3 grid(cdiv(PW / 16, 128), cdiv(PH, PATTERN_ROWS_PER_BLOCK), n_patterns);
    k_expand_patterns<<<grid, 128, 0, st>>>(profiles, profile_len, n_patterns, out, PW, PH, dir);
    return cudaGetLastError();
}

cudaError_t launch_mask(const Shape& s, const uint8_t* roi_full, uint8_t* mask, cudaStream_t st)
{
    dim3 grid(cdiv(s.W, 256), s.H);
    k_mask<<<grid, 256, 0, st>>>(roi_full, mask, s.W, s.H, s.row0, s.H_total);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// wrapped phase (3/wrapped_phase.cpp:151-238): computed where the ROI is set (valid0), i.e.
// BEFORE the mask recurrence, exactly like create_wrapped_phase(); 0 elsewhere.
// ------------------------------------------------------------------------------------------
template <int N, bool LIBDEV>
__global__ void k_wrapped(const uint8_t* __restrict__ fringe, const uint8_t* __restrict__ roi,
                          float* __restrict__ wrapped, int W, int H, int row0, int n_runtime,
                          const double* __restrict__ tab, const double* __restrict__ nw)
{
    const size_t plane = (size_t)W * H;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < plane;
         p += (size_t)gridDim.x * blockDim.x) {
        float out = 0.0f;
        if (roi[(size_t)row0 * W + p] != 0) {
            int I[N > 0 ? N : 16];
            const int n = N > 0 ? N : n_runtime;
#pragma unroll
            for (int k = 0; k < (N > 0 ? N : 16); k++)
                if (k < n) I[k] = fringe[(size_t)k * plane + p];
            out = wrapped_phase<N, LIBDEV>(I, nw, nw + 64, n, tab, tab + 33);
        }
        wrapped[p] = out;
    }
}

cudaError_t launch_wrapped(const Shape& s, int N, const uint8_t* fringe, const uint8_t* roi_full,
                           float* wrapped, const double* tab, const double* nw, bool libdevice,
                           cudaStream_t st)
{
    const size_t plane = (size_t)s.W * s.H;
    const unsigned grid = (unsigned)min((size_t)148 * 16, (plane + 255) / 256);
#define S3D_W(NN)                                                                                 \
    do {                                                                                          \
        if (libdevice)                                                                            \
            k_wrapped<NN, true><<<grid, 256, 0, st>>>(fringe, roi_full, wrapped, s.W, s.H, s.row0, N, tab, nw); \
        else                                                                                      \
            k_wrapped<NN, false><<<grid, 256, 0, st>>>(fringe, roi_full, wrapped, s.W, s.H, s.row0, N, tab, nw); \
    } while (0)
    switch (N) {
        case 3: S3D_W(3); break;
        case 4: S3D_W(4); break;
        case 5: S3D_W(5); break;
        case 8: S3D_W(8); break;
        default: S3D_W(0); break;
    }
#undef S3D_W
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Gray decode + unwrap (4/phase_unwrap.cpp:134-316)
// ------------------------------------------------------------------------------------------
__global__ void k_unwrap(int dir, int M, const uint8_t* __restrict__ gray,
                         const uint8_t* __restrict__ inv, float* __restrict__ wrapped,
                         const uint8_t* __restrict__ mask, int16_t* __restrict__ code,
                         float* __restrict__ unwrapped, int W, int H, int row0, int H_total)
{
    const size_t plane = (size_t)W * H;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < plane;
         p += (size_t)gridDim.x * blockDim.x) {
        if (!mask[p]) {
            code[p] = -1;          // :141-143
            unwrapped[p] = 0.0f;   // zero-fill policy for planes the reference leaves unwritten
            continue;
        }
        int c = 0, b = 0;
        for (int i = 0; i < M; i++) {
            const int g = (int)gray[(size_t)i * plane + p] - (int)inv[(size_t)i * plane + p] >= 0;  // :183
            b = (i == 0) ? g : (b ^ g);                                                             // :187-191
            c += b << (M - 1 - i);                                                                  // :193
        }
        code[p] = (int16_t)c;
        const int x = (int)(p % W), y = row0 + (int)(p / W);
        const bool skipped = dir == 0 ? (x == 0 || x == W - 1) : (y == 0 || y == H_total - 1);  // :285 / :304
        if (skipped) {
            unwrapped[p] = 0.0f;
        } else {
            const float w = add_pi(wrapped[p]);   // :290, stored back
            wrapped[p] = w;
            unwrapped[p] = unwrap_abs(w, c);      // :291
        }
    }
}

cudaError_t launch_unwrap(const Shape& s, int dir, int M, const uint8_t* gray, const uint8_t* inv,
                          float* wrapped, const uint8_t* mask, int16_t* code, float* unwrapped,
                          cudaStream_t st)
{
    const size_t plane = (size_t)s.W * s.H;
    const unsigned grid = (unsigned)min((size_t)148 * 16, (plane + 255) / 256);
    k_unwrap<<<grid, 256, 0, st>>>(dir, M, gray, inv, wrapped, mask, code, unwrapped, s.W, s.H, s.row0,
                                   s.H_total);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// correspondence (5/compute_correspondance.cpp:60-77, 642-679)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int sat_i32(long long v)
{
    return v > 2147483647LL ? 2147483647 : (v < -2147483648LL ? (int)-2147483648LL : (int)v);
}

__global__ void k_cpmap(int fw_v, int fw_h, const float* __restrict__ unw_v,
                        const float* __restrict__ unw_h, const uint8_t* __restrict__ mask_v,
                        const uint8_t* __restrict__ mask_h, int2* __restrict__ cpmap,
                        uint8_t* __restrict__ valid, size_t plane, int PW, int PH)
{
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < plane;
         p += (size_t)gridDim.x * blockDim.x) {
        int2 cp = make_int2(0, 0);
        bool v = mask_v[p] == 1 && mask_h[p] == 1;
        if (v) {
            long long x = 0, y = 0;
            if (!correspond(unw_v[p], fw_v, &x)) {
                v = false;
            } else if (!correspond(unw_h[p], fw_h, &y)) {
                v = false;
                cp.x = sat_i32(x);
            } else {
                cp = make_int2(sat_i32(x), sat_i32(y));
                if (x > PW - 1 || y > PH - 1 || x < 0 || y < 0) v = false;  // :671-675
            }
        }
        cpmap[p] = cp;
        valid[p] = v ? 1 : 0;
    }
}

cudaError_t launch_cpmap(const Shape& s, int fw_v, int fw_h, const float* unw_v, const float* unw_h,
                         const uint8_t* mask_v, const uint8_t* mask_h, int2* cpmap, uint8_t* valid,
                         cudaStream_t st)
{
    const size_t plane = (size_t)s.W * s.H;
    const unsigned grid = (unsigned)min((size_t)148 * 16, (plane + 255) / 256);
    k_cpmap<<<grid, 256, 0, st>>>(fw_v, fw_h, unw_v, unw_h, mask_v, mask_h, cpmap, valid, plane, s.PW,
                                  s.PH);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// undistorted-pixel tables (7/triangulation.cpp:262-307, 352-378), built once per calibration
// ------------------------------------------------------------------------------------------
__global__ void k_undistort_lut(const __grid_constant__ DeviceCalib cal, int projector, int W, int H,
                                int row0, double2* __restrict__ lut)
{
    const size_t plane = (size_t)W * H;
    const double* K = projector ? cal.Kp : cal.Kc;
    const double* k = projector ? cal.dp : cal.dc;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < plane;
         p += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(p % W), y = row0 + (int)(p / W);
        double u, v;
        undistorted_pixel(K, k, (double)x, (double)y, &u, &v);
        lut[p] = make_double2(u, v);
    }
}

cudaError_t launch_undistort_lut(const double*, const DeviceCalib& cal, bool projector, int W, int H,
                                 int row0, double2* lut, cudaStream_t st)
{
    const size_t plane = (size_t)W * H;
    const unsigned grid = (unsigned)min((size_t)148 * 8, (plane + 127) / 128);
    k_undistort_lut<<<grid, 128, 0, st>>>(cal, projector ? 1 : 0, W, H, row0, lut);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// triangulation (7/triangulation.cpp:1223-1247), dense f64 output like intersection_points
// ------------------------------------------------------------------------------------------
__global__ void k_triangulate(const __grid_constant__ DeviceCalib cal,
                              const double2* __restrict__ cam_lut,
                              const double2* __restrict__ proj_lut, const int2* __restrict__ cpmap,
                              const uint8_t* __restrict__ valid, double* __restrict__ xyz, int W, int H,
                              int row0, int PW)
{
    const size_t plane = (size_t)W * H;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < plane;
         p += (size_t)gridDim.x * blockDim.x) {
        double X[3] = {0.0, 0.0, 0.0};
        if (valid[p]) {
            const int x = (int)(p % W), y = row0 + (int)(p / W);
            double uc, vc, up, vp;
            if (cam_lut) {
                const double2 t = cam_lut[p];
                uc = t.x; vc = t.y;
            } else {
                undistorted_pixel_nodist(cal.Kc, cal.ifx_c, cal.ify_c, cal.cam_std != 0, (double)x, (double)y, &uc, &vc);
            }
            const int2 cp = cpmap[p];
            if (proj_lut) {
                const double2 t = proj_lut[(size_t)cp.y * PW + cp.x];
                up = t.x; vp = t.y;
            } else {
                undistorted_pixel_nodist(cal.Kp, cal.ifx_p, cal.ify_p, cal.proj_std != 0, (double)cp.x, (double)cp.y, &up, &vp);
            }
            triangulate_point(cal.Ac, cal.Ap, uc, vc, up, vp, X);
        }
        xyz[3 * p + 0] = X[0];
        xyz[3 * p + 1] = X[1];
        xyz[3 * p + 2] = X[2];
    }
}

cudaError_t launch_triangulate(const Shape& s, const DeviceCalib& cal, const double2* cam_lut,
                               const double2* proj_lut, const int2* cpmap, const uint8_t* valid,
                               double* xyz, cudaStream_t st)
{
    const size_t plane = (size_t)s.W * s.H;
    const unsigned grid = (unsigned)min((size_t)148 * 8, (plane + 127) / 128);
    k_triangulate<<<grid, 128, 0, st>>>(cal, cam_lut, proj_lut, cpmap, valid, xyz, s.W, s.H, s.row0,
                                        s.PW);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// raster-order compaction (8/save_point_cloud.cpp:33-39, 85-136): count / scan / scatter
// ------------------------------------------------------------------------------------------
constexpr int CB = POINT_BLOCK;  // pixels per compaction block

__global__ void k_count(const uint8_t* __restrict__ valid, uint32_t* __restrict__ counts, size_t plane)
{
    __shared__ uint32_t wsum[CB / 32];
    const size_t p = (size_t)blockIdx.x * CB + threadIdx.x;
    const bool v = p < plane && valid[p] != 0;
    const unsigned b = __ballot_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = __popc(b);
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t s = wsum[threadIdx.x];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (threadIdx.x == 0) counts[blockIdx.x] = s;
    }
}

// exclusive scan of n block counts in place by one CTA; writes the total to *total
__global__ void k_scan(uint32_t* __restrict__ counts, int n, uint32_t* __restrict__ total)
{
    __shared__ uint32_t wsum[32];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < n ? counts[i] : 0;
        uint32_t s = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, s, o);
            if ((threadIdx.x & 31) >= o) s += t;
        }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t w = wsum[threadIdx.x];
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, w, o);
                if (threadIdx.x >= o) w += t;
            }
            wsum[threadIdx.x] = w;
        }
        __syncthreads();
        const uint32_t warp_off = (threadIdx.x >> 5) ? wsum[(threadIdx.x >> 5) - 1] : 0;
        const uint32_t c = carry;
        if (i < n) counts[i] = c + warp_off + s - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + warp_off + s;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void k_scatter(const double* __restrict__ xyz, const uint8_t* __restrict__ valid,
                          const uint8_t* __restrict__ texture, const uint32_t* __restrict__ offsets,
                          float* __restrict__ pts, uint32_t* __restrict__ pix, uint8_t* __restrict__ rgb,
                          size_t plane, unsigned pix_base)
{
    __shared__ uint32_t wsum[CB / 32];
    const size_t p = (size_t)blockIdx.x * CB + threadIdx.x;
    const bool v = p < plane && valid[p] != 0;
    const unsigned b = __ballot_sync(0xffffffffu, v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) wsum[w] = __popc(b);
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t s = wsum[threadIdx.x];
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, s, o);
            if (threadIdx.x >= o) s += t;
        }
        wsum[threadIdx.x] = s;  // inclusive
    }
    __syncthreads();
    if (!v) return;
    const uint32_t dst = offsets[blockIdx.x] + (w ? wsum[w - 1] : 0) + __popc(b & ((1u << lane) - 1));
    pts[3 * (size_t)dst + 0] = (float)xyz[3 * p + 0];   // :94-96 (float) casts
    pts[3 * (size_t)dst + 1] = (float)xyz[3 * p + 1];
    pts[3 * (size_t)dst + 2] = (float)xyz[3 * p + 2];
    if (pix) pix[dst] = pix_base + (unsigned)p;
    if (rgb) {                                          // :91-93, cvSplit(BGR)
        rgb[3 * (size_t)dst + 0] = texture ? texture[3 * p + 2] : 0;
        rgb[3 * (size_t)dst + 1] = texture ? texture[3 * p + 1] : 0;
        rgb[3 * (size_t)dst + 2] = texture ? texture[3 * p + 0] : 0;
    }
}

cudaError_t launch_point_offsets(const uint8_t* valid, size_t plane, uint32_t* block_counts, uint32_t* total,
                                 cudaStream_t st)
{
    const int nb = plane ? (int)cdiv((long)plane, CB) : 1;
    k_count<<<nb, CB, 0, st>>>(valid, block_counts, plane);
    k_scan<<<1, 1024, 0, st>>>(block_counts, nb, total);
    return cudaGetLastError();
}

cudaError_t launch_block_scan(uint32_t* counts, int n, uint32_t* total, cudaStream_t st)
{
    k_scan<<<1, 1024, 0, st>>>(counts, n, total);
    return cudaGetLastError();
}

cudaError_t launch_compact(const Shape& s, const double* xyz, const uint8_t* valid,
                           const uint8_t* texture, uint32_t* block_counts, float* pts, uint32_t* pix,
                           uint8_t* rgb, uint32_t* d_count, cudaStream_t st, int* n_launches)
{
    const size_t plane = (size_t)s.W * s.H;
    const int nb = (int)cdiv((long)plane, CB);
    launch_point_offsets(valid, plane, block_counts, d_count, st);
    k_scatter<<<nb, CB, 0, st>>>(xyz, valid, texture, block_counts, pts, pix, rgb, plane,
                                 (unsigned)((size_t)s.row0 * s.W));
    if (n_launches) *n_launches = 3;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// self-test: (float)atan2(y, x) with CUDA's libdevice (mode 0) or the in-house evaluation (1)
// ------------------------------------------------------------------------------------------
__global__ void k_debug_atan2(const double* __restrict__ y, const double* __restrict__ x,
                              float* __restrict__ out, int n, int mode, const double* __restrict__ tab)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = mode == 0 ? __double2float_rn(atan2(y[i], x[i]))
                       : atan2_to_float(y[i], x[i], (float)y[i], (float)x[i], tab);
}

cudaError_t launch_debug_atan2(const double* y, const double* x, float* out, int n, int mode,
                               const double* tab, cudaStream_t st)
{
    k_debug_atan2<<<cdiv(n, 256), 256, 0, st>>>(y, x, out, n, mode, tab);
    return cudaGetLastError();
}


// self-test: the 3-operation exact quotient Phi/(2.0*Pi) against IEEE division on EVERY finite
// non-negative float phase (the only operands 5/compute_correspondance.cpp:648 can see).
__global__ void k_debug_divcheck(unsigned long long* __restrict__ bad)
{
    unsigned long long local = 0;
    for (unsigned long long b = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; b < 0x7f800000ull;
         b += (unsigned long long)gridDim.x * blockDim.x) {
        const double a = (double)__uint_as_float((unsigned)b);
        const double q1 = ddiv(a, S3D_TWO_PI_REF);
        const double q2 = div_const(a, S3D_TWO_PI_REF, 1.0 / (S3D_TWO_PI_REF), true);
        local += q1 != q2;
    }
    if (local) atomicAdd(bad, local);
}

cudaError_t launch_debug_divcheck(unsigned long long* bad, cudaStream_t st)
{
    k_debug_divcheck<<<148 * 16, 256, 0, st>>>(bad);
    return cudaGetLastError();
}

}  // namespace s3d
