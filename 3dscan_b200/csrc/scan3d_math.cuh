// scan3d_math.cuh -- per-pixel arithmetic of the 3dscan reconstruction path, written so that
// every value that feeds an integer decision (fringe order, lrint correspondence, validity)
// follows the reference's IEEE operation sequence exactly.  All double arithmetic that must
// match goes through __dmul_rn/__dadd_rn/__dsub_rn/__ddiv_rn so nvcc never contracts it to FMA
// (the reference was an SSE2 build: separate multiply and add roundings).
//
// Reference expressions (paths relative to the reference tree):
//   3/wrapped_phase.cpp:171-175,195-198,217-220   wrapped phase
//   4/phase_unwrap.cpp:183-193                    Gray threshold / Gray->binary / code
//   4/phase_unwrap.cpp:290-291                    += Pi ; + code*2.0*Pi
//   5/compute_correspondance.cpp:648,659,671      lrint correspondences + bounds
//   7/triangulation.cpp:290-307,1152-1211         undistorted pixel, P, F, (P^T P)^-1 P^T F
//   PROJECT_GLOBAL/global_cv.h:62                 #define Pi 22.0/7.0 (textual)
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#if !defined(__CUDACC__)
// host build of this header (CPU tests only): the including translation unit provides the CUDA
// intrinsics used below as plain IEEE host functions (tests/cuda_host_shim.h)
double s3d_host_rcp_seed(double x);
#endif

namespace s3d {

// Double constants of the hot loops live in the constant bank (the FP64 pipe takes a constant-bank operand directly;
// as literals each one costs two moves per use at 80 registers per thread).  Host builds see plain constants.
#if defined(__CUDACC__)
#define S3D_KCONST static __constant__ double
#else
#define S3D_KCONST static const double
#endif
S3D_KCONST K_ATAN_P9 = 1.0 / 9.0;
S3D_KCONST K_ATAN_P7 = -1.0 / 7.0;
S3D_KCONST K_ATAN_P5 = 1.0 / 5.0;
S3D_KCONST K_ATAN_P3 = -1.0 / 3.0;
S3D_KCONST K_SQRT_HALF = 0.70710678118654752440;
S3D_KCONST K_2P52_512 = 4503599627370496.0 + 512.0;
S3D_KCONST K_2P52_1024 = 4503599627370496.0 + 1024.0;
S3D_KCONST K_PI_REF = 22.0 / 7.0;
S3D_KCONST K_TWO_PI_REF = 2.0 * 22.0 / 7.0;
S3D_KCONST K_RCP_TWO_PI_REF = 1.0 / (2.0 * 22.0 / 7.0);
S3D_KCONST K_RCP_7 = 1.0 / 7.0;

// "Pi" as the reference's macro expands inside each expression.
#define S3D_PI_REF (22.0 / 7.0)              // x += Pi            -> x + 22.0/7.0
#define S3D_TWO_PI_REF (2.0 * 22.0 / 7.0)    // (2.0*Pi)           -> (2.0*22.0)/7.0

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

// ---------------------------------------------------------------------------------------
// atan2 evaluated in double and rounded to float: (float)atan2((double)t1,(double)t2) of
// 3/wrapped_phase.cpp:175.  Accuracy ~1 double ulp, so the float result differs from a
// correctly rounded libm only when the true value lies within ~2^-52 of a float rounding
// boundary (probability ~1e-8 per pixel; tests count and bound these).
//
// Method: reduce to a = min/max in [0,1]; pick c = i/32 nearest to a (float estimate);
// atan(a) = atan(c) + atan(t), t = (mn - c*mx)/(mx + c*mn), |t| <= 1/64, so a degree-9 odd
// polynomial is exact to 2^-60; one division (reciprocal seed + Newton) instead of libm's two
// range-reduction divisions and degree-19 polynomial.
// ---------------------------------------------------------------------------------------
// Table layout (66 + 6 doubles, built on the host by fill_atan_table with long-double atanl):
//   [0..32]  hi(atan(i/32))      [33..65] lo(atan(i/32))
//   [66..71] quadrant constants {K_hi, K_lo} for k = 0 (none), 1 (pi/2), 2 (pi)
constexpr int ATAN_TAB_DOUBLES = 72;

// host side: fills that table (long-double atanl split into hi + lo)
inline void fill_atan_table(double* t)
{
    for (int i = 0; i <= 32; i++) {
        const long double c = (long double)i / 32.0L;
        const long double a = atanl(c);
        const double hi = (double)a;
        t[i] = hi;
        t[33 + i] = (double)(a - (long double)hi);
    }
    // quadrant constants {hi, lo}: 0, pi/2, pi
    t[66] = 0.0; t[67] = 0.0;
    t[68] = 1.57079632679489655800e+00; t[69] = 6.12323399573676603587e-17;
    t[70] = 3.14159265358979311600e+00; t[71] = 1.22464679914735317720e-16;
}

// rcp.approx.ftz.f64: a ~20-bit reciprocal seed (only the high word of the operand is looked at, the
// low word of the result is zero).  The host build (tests/fused_math_host.cpp) substitutes a seed
// of the same quality; after the corrections below the seed's low bits do not reach the result.
__device__ __forceinline__ double rcp_seed(double x)
{
#if defined(__CUDA_ARCH__)
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
#elif !defined(__CUDACC__)
    return s3d_host_rcp_seed(x);
#else
    return x;   // nvcc's host pass only parses this function, nothing calls it there
#endif
}

__device__ __forceinline__ double fast_div(double num, double den)
{
    double r = rcp_seed(den);                                  // ~20 good bits
    r = fma(r, fma(-den, r, 1.0), r);                          // ~40
    const double t = num * r;
    return fma(fma(-den, t, num), r, t);                       // residual correction: ~1 ulp
}

// y, x: exact doubles; yf, xf: any float approximations of them (only select the table row).
// Branch-free on purpose: the two directions' evaluations interleave in one basic block.
//   atan2 = K + s*atan(mn/mx):  (|y|<=|x|, x>=0): K=0, s=+   (|y|>|x|, x>=0): K=pi/2, s=-
//                               (|y|<=|x|, x<0):  K=pi, s=-  (|y|>|x|, x<0):  K=pi/2, s=+
// then the sign of y.
// mx and mn are selected from the words of x and y; the high word goes through a float select with |.| operands, which
// clears its sign bit in the same instruction (fabs of a double in a register costs a DADD on the FP64 pipe).  Read as
// a float, a high word is never NaN or subnormal here (|x|, |y| lie in [2^-1000, 2^1000] or are 0).  The sign of x is
// its high word's: x is never -0 (every caller passes an integer, or a round-to-nearest sum that starts from one, and
// such a sum is -0 only when both of its operands are).
__device__ __forceinline__ float atan2_to_float(double y, double x, float yf, float xf,
                                                const double* __restrict__ tab)
{
    const bool swap = fabs(y) > fabs(x);
    const int xh = __double2hiint(x), xl = __double2loint(x), yh = __double2hiint(y), yl = __double2loint(y);
    const bool xneg = xh < 0;
    const float axh = fabsf(__int_as_float(xh)), ayh = fabsf(__int_as_float(yh));
    const double mx = __hiloint2double(__float_as_int(swap ? ayh : axh), swap ? yl : xl);
    const double mn = __hiloint2double(__float_as_int(swap ? axh : ayh), swap ? xl : yl);
    (void)yf; (void)xf;
    // Table row i = round(32 * mn / mx) and c = i / 32, both out of ONE double: 2^47 + q has an ulp of exactly 1/32,
    // so adding q = mn * (reciprocal seed of mx) to 2^47 rounds it to a multiple of 1/32, leaves i in the low word of
    // the sum and c after subtracting 2^47 again (a 20-bit seed is plenty: the row only has to be near, the degree-9
    // polynomial has 2^-60 head-room).  mx == 0: seed = inf, 0 * inf = NaN, whose low word is 0 -> row 0, and the
    // result is forced to 0 below.
    const double s47 = fma(mn, rcp_seed(mx), 140737488355328.0);
    const int i = __double2loint(s47) & 63;
    const double c = s47 - 140737488355328.0;
    const double num = fma(-c, mx, mn);
    const double den = fma(c, mn, mx);
    const double t = fast_div(num, den);
    const double s = t * t;
    double p = fma(s, K_ATAN_P9, K_ATAN_P7);
    p = fma(s, p, K_ATAN_P5);
    p = fma(s, p, K_ATAN_P3);
    p = fma(t * s, p, t);
    double res = tab[i] + (tab[33 + i] + p);
    // s*res: flip the sign when exactly one of (swap, xneg) holds
    res = __hiloint2double(__double2hiint(res) ^ ((swap != xneg) ? 0x80000000 : 0), __double2loint(res));
    const int k = swap ? 1 : (xneg ? 2 : 0);
    res = tab[66 + 2 * k] + (tab[67 + 2 * k] + res);
    float out = __double2float_rn(res);
    out = mx == 0.0 ? 0.0f : out;
    // copy the sign of y (y is never -0 here: it is a difference of non-negative samples)
    return __int_as_float(__float_as_int(out) ^ (__double2hiint(y) & 0x80000000));
}

// ---------------------------------------------------------------------------------------
// The 5-step formula calls the FLOAT atan2f (3/wrapped_phase.cpp:220).  glibc's atan2f is the
// fdlibm routine (sysdeps/ieee754/flt-32/e_atan2f.c + s_atanf.c, unchanged from the eglibc 2.15
// the reference ran on to the glibc 2.39 of this image): a fixed sequence of float operations.
// Restated here with explicitly rounded float intrinsics so the result is bit-identical
// (tests/test_oracle_golden.py pins the same restatement against libm on the CPU).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float fm(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fa(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fs(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fd(float a, float b) { return __fdiv_rn(a, b); }

__device__ __forceinline__ float atanf_fdlibm(float x)
{
    const float atanhi[4] = {4.6364760399e-01f, 7.8539812565e-01f, 9.8279368877e-01f, 1.5707962513e+00f};
    const float atanlo[4] = {5.0121582440e-09f, 3.7748947079e-08f, 3.4473217170e-08f, 7.5497894159e-08f};
    const int hx = __float_as_int(x), ix = hx & 0x7fffffff;
    int id;
    if (ix >= 0x4c000000) {
        if (ix > 0x7f800000) return fa(x, x);
        return hx > 0 ? fa(atanhi[3], atanlo[3]) : fs(-atanhi[3], atanlo[3]);
    }
    if (ix < 0x3ee00000) {
        if (ix < 0x31000000) return x;
        id = -1;
    } else {
        x = fabsf(x);
        if (ix < 0x3f980000) {
            if (ix < 0x3f300000) { id = 0; x = fd(fs(fm(2.0f, x), 1.0f), fa(2.0f, x)); }
            else { id = 1; x = fd(fs(x, 1.0f), fa(x, 1.0f)); }
        } else {
            if (ix < 0x401c0000) { id = 2; x = fd(fs(x, 1.5f), fa(1.0f, fm(1.5f, x))); }
            else { id = 3; x = fd(-1.0f, x); }
        }
    }
    const float z = fm(x, x), w = fm(z, z);
    const float s1 = fm(z, fa(3.3333334327e-01f, fm(w, fa(1.4285714924e-01f, fm(w, fa(9.0908870101e-02f,
                     fm(w, fa(6.6610731184e-02f, fm(w, fa(4.9768779427e-02f, fm(w, 1.6285819933e-02f)))))))))));
    const float s2 = fm(w, fa(-2.0000000298e-01f, fm(w, fa(-1.1111110449e-01f, fm(w, fa(-7.6918758452e-02f,
                     fm(w, fa(-5.8335702866e-02f, fm(w, -3.6531571299e-02f)))))))));
    if (id < 0) return fs(x, fm(x, fa(s1, s2)));
    const float hi = id == 0 ? atanhi[0] : id == 1 ? atanhi[1] : id == 2 ? atanhi[2] : atanhi[3];
    const float lo = id == 0 ? atanlo[0] : id == 1 ? atanlo[1] : id == 2 ? atanlo[2] : atanlo[3];
    const float r = fs(hi, fs(fs(fm(x, fa(s1, s2)), lo), x));
    return hx < 0 ? -r : r;
}

__device__ __forceinline__ float atan2f_fdlibm(float y, float x)
{
    const float tiny = 1.0e-30f, pi_o_2 = 1.5707963705e+00f, pi = 3.1415927410e+00f, pi_lo = -8.7422776573e-08f;
    const int hx = __float_as_int(x), ix = hx & 0x7fffffff, hy = __float_as_int(y), iy = hy & 0x7fffffff;
    if (ix > 0x7f800000 || iy > 0x7f800000) return fa(x, y);
    if (hx == 0x3f800000) return atanf_fdlibm(y);
    const int m = ((hy >> 31) & 1) | ((hx >> 30) & 2);
    if (iy == 0) return m == 0 || m == 1 ? y : (m == 2 ? fa(pi, tiny) : fs(-pi, tiny));
    if (ix == 0) return hy < 0 ? fs(-pi_o_2, tiny) : fa(pi_o_2, tiny);
    // (infinite operands cannot occur: the inputs are differences of 8-bit samples)
    const int k = (iy - ix) >> 23;
    float z;
    if (k > 60) z = fa(pi_o_2, fm(0.5f, pi_lo));
    else if (hx < 0 && k < -60) z = 0.0f;
    else z = atanf_fdlibm(fabsf(fd(y, x)));
    if (m == 0) return z;
    if (m == 1) return __int_as_float(__float_as_int(z) ^ 0x80000000);
    if (m == 2) return fs(pi, fs(z, pi_lo));
    return fs(fs(z, pi_lo), pi);
}

// ---------------------------------------------------------------------------------------
// wrapped phase (3/wrapped_phase.cpp:151-238).  I[k] are the pixel's N fringe samples.
// USE_LIBDEVICE selects CUDA's own double atan2 (reference implementation for A/B tests).
// ---------------------------------------------------------------------------------------
template <bool USE_LIBDEVICE>
__device__ __forceinline__ float phase_from_terms(double d1, double d2, float f1, float f2,
                                                  const double* tab_hi, const double* /*tab_lo*/)
{
    if (USE_LIBDEVICE) return __double2float_rn(atan2(d1, d2));
    return atan2_to_float(d1, d2, f1, f2, tab_hi);
}

template <int N, bool USE_LIBDEVICE>
__device__ __forceinline__ float wrapped_phase(const int* I, const double* __restrict__ wsin,
                                               const double* __restrict__ wcos, int n_runtime,
                                               const double* tab_hi, const double* tab_lo)
{
    if (N == 3) {            // :171-175   t1 = I0 - I2 ; t2 = 2*I1 - I0 - I2   (exact)
        const int t1 = I[0] - I[2], t2 = 2 * I[1] - I[0] - I[2];
        return phase_from_terms<USE_LIBDEVICE>((double)t1, (double)t2, (float)t1, (float)t2, tab_hi, tab_lo);
    } else if (N == 4) {     // :195-198   t1 = I3 - I1 ; t2 = I0 - I2
        const int t1 = I[3] - I[1], t2 = I[0] - I[2];
        return phase_from_terms<USE_LIBDEVICE>((double)t1, (double)t2, (float)t1, (float)t2, tab_hi, tab_lo);
    } else if (N == 5) {     // :217-220   t1 = 2(I1 - I3) ; t2 = 2*I2 - I0 - I4 ; atan2f
        const int t1 = 2 * (I[1] - I[3]), t2 = 2 * I[2] - I[0] - I[4];
        return atan2f_fdlibm((float)t1, (float)t2);
    } else if (N == 8) {     // extension: shifts k*pi/4, phase origin of the 4-step formula
        const int a1 = I[6] - I[2], b1 = I[5] + I[7] - I[1] - I[3];
        const int a2 = I[0] - I[4], b2 = I[1] + I[7] - I[3] - I[5];
        const double r = 0.70710678118654752440;
        const double d1 = dadd((double)a1, dmul((double)b1, r));
        const double d2 = dadd((double)a2, dmul((double)b2, r));
        const float f1 = fmaf((float)b1, 0.70710678f, (float)a1);
        const float f2 = fmaf((float)b2, 0.70710678f, (float)a2);
        return phase_from_terms<USE_LIBDEVICE>(d1, d2, f1, f2, tab_hi, tab_lo);
    } else {                 // extension: generic N, sequential double sums (k ascending)
        double S = 0.0, C = 0.0;
        for (int k = 0; k < n_runtime; k++) {
            const double v = (double)I[k];
            S = dadd(S, dmul(v, wsin[k]));
            C = dadd(C, dmul(v, wcos[k]));
        }
        const double d1 = dsub(0.0, S);
        return phase_from_terms<USE_LIBDEVICE>(d1, C, (float)d1, (float)C, tab_hi, tab_lo);
    }
}

// Correctly rounded a/b for a constant divisor b in 3 operations (Markstein): with y = RN(1/b),
// q0 = RN(a*y), r = a - q0*b (exact in one FMA), q = RN(q0 + r*y).  The host verifies the
// identity against IEEE division on every fringe order (a = code*44, b = 7) at context creation
// and the GPU tests verify it on every float phase (b = 44/7); `exact == false` selects the
// plain IEEE division.
__device__ __forceinline__ double div_const(double a, double b, double rcp_b, bool exact)
{
    if (!exact) return ddiv(a, b);
    const double q0 = dmul(a, rcp_b);
    const double r = fma(-q0, b, a);
    return fma(r, rcp_b, q0);
}

// 4/phase_unwrap.cpp:290 :  wrapped += Pi          (float <- double sum)
__device__ __forceinline__ float add_pi(float wrapped)
{
    return __double2float_rn(dadd((double)wrapped, K_PI_REF));
}
// 4/phase_unwrap.cpp:291 :  unwrapped = wrapped + code*2.0*Pi   == w + ((code*2.0)*22.0)/7.0
__device__ __forceinline__ float unwrap_abs(float wrapped_plus_pi, int code, bool fast = false)
{
    // (code*2.0)*22.0 is an exact integer, so only the division rounds
    const double k = div_const((double)(code * 44), 7.0, K_RCP_7, fast);   // code*44 < 2^21: exact
    return __double2float_rn(dadd((double)wrapped_plus_pi, k));
}
// the same with k = code*2.0*Pi looked up (fill_code_term_table)
__device__ __forceinline__ float unwrap_abs_k(float wrapped_plus_pi, double k)
{
    return __double2float_rn(dadd((double)wrapped_plus_pi, k));
}
// host side: code*2.0*Pi of every fringe order below n, in the reference's IEEE order.  The single-pass kernel loads
// it (one cached load per pixel and direction) instead of converting the order and dividing (4 FP64 instructions).
inline void fill_code_term_table(double* t, int n)
{
    for (int code = 0; code < n; code++) t[code] = (((double)code * 2.0) * 22.0) / 7.0;
}
// 5/compute_correspondance.cpp:648 : lrint(fw * (Phi / (2.0*Pi))), round-half-even; FE_INVALID
// (NaN/inf/out of range) rejects the pixel.  Returns false on FE_INVALID.
__device__ __forceinline__ bool correspond(float phi_abs, int fw, long long* out, bool fast = false)
{
    const double v = dmul((double)fw, div_const((double)phi_abs, S3D_TWO_PI_REF, 1.0 / (S3D_TWO_PI_REF), fast));
    *out = __double2ll_rn(v);
    return (v == v) && v < 9223372036854775808.0 && v >= -9223372036854775808.0;
}
// Same decision in 32 bits for the fused kernels: cvt.rni.s32.f64 saturates exactly like the
// clamp of the 64-bit lrint to int, NaN converts to 0 and fails the |v| < 2^63 test (FE_INVALID).
// (fw as a double: the caller converts the fringe width once, not per pixel)
__device__ __forceinline__ bool correspond32(float phi_abs, double fw, int* out)
{
    const double v = dmul(fw, div_const((double)phi_abs, K_TWO_PI_REF, K_RCP_TWO_PI_REF, true));
    *out = __double2int_rn(v);
    return fabs(v) < 9223372036854775808.0;
}
// correspond32 for a phase that is known to be finite and below 2^18 in magnitude (k_fused7: 0, or
// RN(RN(w + 22/7) + code*44/7) with w in [-pi, pi] and code < 2^15): with fw < 2^31, |v| < 2^47, so the
// FE_INVALID test always passes and is left out.  An out-of-range v still saturates, and the caller's unsigned
// bounds compare rejects both saturated values.
__device__ __forceinline__ int correspond32_finite(float phi_abs, double fw)
{
    return __double2int_rn(dmul(fw, div_const((double)phi_abs, K_TWO_PI_REF, K_RCP_TWO_PI_REF, true)));
}

// ---------------------------------------------------------------------------------------
// calibration algebra on the device
// ---------------------------------------------------------------------------------------
struct DeviceCalib {
    double Ac[12];      // K_cam * [R|t]   (3x4 row-major)   7/triangulation.cpp:1090-1101
    double Ap[12];      // K_proj * [R|t]                     :1104-1116
    double Kc[9], dc[5], Kp[9], dp[5];
    double ifx_c, ify_c, ifx_p, ify_p;   // 1./fx, 1./fy exactly as cvUndistortPoints computes them (host IEEE division)
    int cam_distorted;  // any camera distortion coefficient non-zero
    int proj_distorted; // any projector distortion coefficient non-zero
    int cam_std;        // Kc == [fx 0 cx; 0 fy cy; 0 0 1]: the K*[x;y;1] product has exact shortcuts
    int proj_std;
    int fast_div_ok;    // host verified: the 3-operation exact quotients below equal IEEE division
    // the fast solve in the camera's frame (triangulate_point_camframe; filled by camera_frame_calib)
    double Apc[12];     // Ap * [Rc|tc]^-1: the projector's matrix for camera-frame points
    double Rct[9];      // Rc^T (row-major): camera frame -> world
    double oc[3];       // -Rc^T tc: the camera centre in the world
    double fx2, fy2;    // Kc[0]^2, Kc[4]^2
};

// Host side: the camera-frame set-up from the camera's rotation Rc (row-major), translation tc and intrinsics Kc and
// the projector's world matrix Ap.
inline void camera_frame_calib(const double Kc[9], const double Rc[9], const double tc[3], const double Ap[12],
                               DeviceCalib* d)
{
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) d->Rct[i * 3 + j] = Rc[j * 3 + i];
    for (int i = 0; i < 3; i++) {
        long double s = 0.0L;
        for (int k = 0; k < 3; k++) s -= (long double)Rc[k * 3 + i] * tc[k];
        d->oc[i] = (double)s;
    }
    // [Rc|tc]^-1 = [Rc^T | -Rc^T tc]
    for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) {
            long double s = 0.0L;
            for (int k = 0; k < 3; k++) s += (long double)Ap[i * 4 + k] * Rc[j * 3 + k];
            d->Apc[i * 4 + j] = (double)s;
        }
        long double s = Ap[i * 4 + 3];
        for (int k = 0; k < 3; k++) s += (long double)Ap[i * 4 + k] * d->oc[k];
        d->Apc[i * 4 + 3] = (double)s;
    }
    d->fx2 = Kc[0] * Kc[0];
    d->fy2 = Kc[4] * Kc[4];
}

// One pixel of cvUndistortPoints (5 fixed iterations, 5-coefficient model) followed by
// K*[xn;yn;1] and the divide by the third row (7/triangulation.cpp:290-307 / :363-378).
__device__ __forceinline__ void undistorted_pixel(const double* __restrict__ K,
                                                  const double* __restrict__ k, double u, double v,
                                                  double* ou, double* ov)
{
    const double cx = K[2], cy = K[5];
    const double ifx = ddiv(1.0, K[0]), ify = ddiv(1.0, K[4]);
    double x, y, x0, y0;
    x0 = x = dmul(dsub(u, cx), ifx);
    y0 = y = dmul(dsub(v, cy), ify);
#pragma unroll 1
    for (int j = 0; j < 5; j++) {
        const double r2 = dadd(dmul(x, x), dmul(y, y));
        const double poly = dmul(dadd(dmul(dadd(dmul(k[4], r2), k[1]), r2), k[0]), r2);
        const double icdist = ddiv(1.0, dadd(1.0, poly));
        // deltaX = 2*k[2]*x*y + k[3]*(r2 + 2*x*x)
        const double dX = dadd(dmul(dmul(dmul(2.0, k[2]), x), y), dmul(k[3], dadd(r2, dmul(dmul(2.0, x), x))));
        // deltaY = k[2]*(r2 + 2*y*y) + 2*k[3]*x*y
        const double dY = dadd(dmul(k[2], dadd(r2, dmul(dmul(2.0, y), y))), dmul(dmul(dmul(2.0, k[3]), x), y));
        x = dmul(dsub(x0, dX), icdist);
        y = dmul(dsub(y0, dY), icdist);
    }
    // cvMatMul(K, [x;y;1]) with sums k ascending from 0, then rows 0,1 divided by row 2
    const double m0 = dadd(dadd(dadd(0.0, dmul(K[0], x)), dmul(K[1], y)), dmul(K[2], 1.0));
    const double m1 = dadd(dadd(dadd(0.0, dmul(K[3], x)), dmul(K[4], y)), dmul(K[5], 1.0));
    const double m2 = dadd(dadd(dadd(0.0, dmul(K[6], x)), dmul(K[7], y)), dmul(K[8], 1.0));
    *ou = ddiv(m0, m2);
    *ov = ddiv(m1, m2);
}

// Zero distortion: the 5 iterations are the exact identity (icdist == 1, deltas == 0), so only
// the normalise / re-project round trip remains.  Bit-identical to undistorted_pixel() then.
// With K in the standard form [fx 0 cx; 0 fy cy; 0 0 1] the GEMM row ((0 + fx*x) + 0*y) + cx*1
// equals fx*x + cx exactly (adding +-0 and multiplying by 1 are exact) and the third row is
// exactly 1, so the divide by it is the identity: 4 operations per coordinate.
__device__ __forceinline__ double undist_coord_std(double u, double c, double inv_f, double f)
{
    return dadd(dmul(f, dmul(dsub(u, c), inv_f)), c);
}
// the same for callers that only run without a table when K has the standard form (the host builds a table otherwise)
__device__ __forceinline__ void undistorted_pixel_std(const double* __restrict__ K, double ifx, double ify, double u, double v,
                                                      double* ou, double* ov)
{
    *ou = undist_coord_std(u, K[2], ifx, K[0]);
    *ov = undist_coord_std(v, K[5], ify, K[4]);
}
__device__ __forceinline__ void undistorted_pixel_nodist(const double* __restrict__ K, double ifx,
                                                         double ify, bool std_form, double u,
                                                         double v, double* ou, double* ov)
{
    if (std_form) {
        *ou = undist_coord_std(u, K[2], ifx, K[0]);
        *ov = undist_coord_std(v, K[5], ify, K[4]);
        return;
    }
    const double x = dmul(dsub(u, K[2]), ifx);
    const double y = dmul(dsub(v, K[5]), ify);
    const double m0 = dadd(dadd(dadd(0.0, dmul(K[0], x)), dmul(K[1], y)), dmul(K[2], 1.0));
    const double m1 = dadd(dadd(dadd(0.0, dmul(K[3], x)), dmul(K[4], y)), dmul(K[5], 1.0));
    const double m2 = dadd(dadd(dadd(0.0, dmul(K[6], x)), dmul(K[7], y)), dmul(K[8], 1.0));
    *ou = ddiv(m0, m2);
    *ov = ddiv(m1, m2);
}

// sum_k a_k*b_k, k ascending, accumulator starts at 0 (OpenCV GEMM order)
__device__ __forceinline__ double dot4(double a0, double b0, double a1, double b1, double a2,
                                       double b2, double a3, double b3)
{
    return dadd(dadd(dadd(dmul(a0, b0), dmul(a1, b1)), dmul(a2, b2)), dmul(a3, b3));
}
__device__ __forceinline__ double dot3(double a0, double b0, double a1, double b1, double a2,
                                       double b2)
{
    return dadd(dadd(dmul(a0, b0), dmul(a1, b1)), dmul(a2, b2));
}

// compute_P / compute_F / compute_X_Y_Z (7/triangulation.cpp:1134-1218) for one correspondence:
// V = ((P^T P)^-1 P^T) F with cvInvert's closed-form 3x3 and the reference's product order.
__device__ __forceinline__ void triangulate_point(const double* __restrict__ Ac,
                                                  const double* __restrict__ Ap, double uc,
                                                  double vc, double up, double vp, double* X)
{
    double P[4][3], F[4];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        P[0][j] = dsub(Ac[0 * 4 + j], dmul(uc, Ac[2 * 4 + j]));
        P[1][j] = dsub(Ac[1 * 4 + j], dmul(vc, Ac[2 * 4 + j]));
        P[2][j] = dsub(Ap[0 * 4 + j], dmul(up, Ap[2 * 4 + j]));
        P[3][j] = dsub(Ap[1 * 4 + j], dmul(vp, Ap[2 * 4 + j]));
    }
    F[0] = dsub(dmul(Ac[11], uc), Ac[3]);
    F[1] = dsub(dmul(Ac[11], vc), Ac[7]);
    F[2] = dsub(dmul(Ap[11], up), Ap[3]);
    F[3] = dsub(dmul(Ap[11], vp), Ap[7]);
    // S = P^T P (symmetric bit-for-bit: products commute, same summation order)
    const double S00 = dot4(P[0][0], P[0][0], P[1][0], P[1][0], P[2][0], P[2][0], P[3][0], P[3][0]);
    const double S01 = dot4(P[0][0], P[0][1], P[1][0], P[1][1], P[2][0], P[2][1], P[3][0], P[3][1]);
    const double S02 = dot4(P[0][0], P[0][2], P[1][0], P[1][2], P[2][0], P[2][2], P[3][0], P[3][2]);
    const double S11 = dot4(P[0][1], P[0][1], P[1][1], P[1][1], P[2][1], P[2][1], P[3][1], P[3][1]);
    const double S12 = dot4(P[0][1], P[0][2], P[1][1], P[1][2], P[2][1], P[2][2], P[3][1], P[3][2]);
    const double S22 = dot4(P[0][2], P[0][2], P[1][2], P[1][2], P[2][2], P[2][2], P[3][2], P[3][2]);
    const double S10 = S01, S20 = S02, S21 = S12;
    // cvInvert, n == 3, CV_64F: det3 then cofactors times 1/det
    const double c00 = dsub(dmul(S11, S22), dmul(S12, S21));
    const double c01 = dsub(dmul(S10, S22), dmul(S12, S20));
    const double c02 = dsub(dmul(S10, S21), dmul(S11, S20));
    double d = dadd(dsub(dmul(S00, c00), dmul(S01, c01)), dmul(S02, c02));
    // the cofactor matrix of a symmetric S is symmetric bit-for-bit (the mirrored entries are the
    // same two products in the other operand order), so 6 of cvInvert's 9 entries are computed
    double T[3][3];
    if (d != 0.0) {
        d = ddiv(1.0, d);
        T[0][0] = dmul(c00, d);
        T[0][1] = dmul(dsub(dmul(S02, S21), dmul(S01, S22)), d);
        T[0][2] = dmul(dsub(dmul(S01, S12), dmul(S02, S11)), d);
        T[1][1] = dmul(dsub(dmul(S00, S22), dmul(S02, S20)), d);
        T[1][2] = dmul(dsub(dmul(S02, S10), dmul(S00, S12)), d);
        T[2][2] = dmul(dsub(dmul(S00, S11), dmul(S01, S10)), d);
        T[1][0] = T[0][1];
        T[2][0] = T[0][2];
        T[2][1] = T[1][2];
    } else {
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
            for (int j = 0; j < 3; j++) T[i][j] = 0.0;
    }
    // I2 = T * P^T (3x4), V = I2 * F
#pragma unroll
    for (int i = 0; i < 3; i++) {
        double I2[4];
#pragma unroll
        for (int j = 0; j < 4; j++) I2[j] = dot3(T[i][0], P[j][0], T[i][1], P[j][1], T[i][2], P[j][2]);
        X[i] = dot4(I2[0], F[0], I2[1], F[1], I2[2], F[2], I2[3], F[3]);
    }
}

// Same least-squares solution with fused multiply-adds and the right-hand side reduced first:
// x = adj(S) (P^T F) / det(S), S = P^T P.  ~90 FP64 operations instead of ~220; differs from the
// reference's operation order by rounding only (<= 1e-10 relative, against the 1e-5 bar), so the
// float point cloud is identical except for last-bit ties.  Selected by SCAN3D_FLAG_FAST_TRIANGULATION.
__device__ __forceinline__ void triangulate_point_fast(const double* __restrict__ Ac,
                                                       const double* __restrict__ Ap, double uc,
                                                       double vc, double up, double vp, double* X)
{
    double P[4][3], F[4];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        P[0][j] = fma(-uc, Ac[8 + j], Ac[0 + j]);
        P[1][j] = fma(-vc, Ac[8 + j], Ac[4 + j]);
        P[2][j] = fma(-up, Ap[8 + j], Ap[0 + j]);
        P[3][j] = fma(-vp, Ap[8 + j], Ap[4 + j]);
    }
    F[0] = fma(Ac[11], uc, -Ac[3]);
    F[1] = fma(Ac[11], vc, -Ac[7]);
    F[2] = fma(Ap[11], up, -Ap[3]);
    F[3] = fma(Ap[11], vp, -Ap[7]);
#define S3D_DOT4(a, b) fma(P[3][a], P[3][b], fma(P[2][a], P[2][b], fma(P[1][a], P[1][b], P[0][a] * P[0][b])))
    const double S00 = S3D_DOT4(0, 0), S01 = S3D_DOT4(0, 1), S02 = S3D_DOT4(0, 2);
    const double S11 = S3D_DOT4(1, 1), S12 = S3D_DOT4(1, 2), S22 = S3D_DOT4(2, 2);
#undef S3D_DOT4
    double b[3];
#pragma unroll
    for (int j = 0; j < 3; j++) b[j] = fma(P[3][j], F[3], fma(P[2][j], F[2], fma(P[1][j], F[1], P[0][j] * F[0])));
    const double c00 = fma(S11, S22, -S12 * S12);
    const double c01 = fma(S02, S12, -S01 * S22);
    const double c02 = fma(S01, S12, -S02 * S11);
    const double c11 = fma(S00, S22, -S02 * S02);
    const double c12 = fma(S01, S02, -S00 * S12);
    const double c22 = fma(S00, S11, -S01 * S01);
    const double det = fma(S02, c02, fma(S01, c01, S00 * c00));
    double r = rcp_seed(det);
    r = fma(r, fma(-det, r, 1.0), r);
    r = fma(r, fma(-det, r, 1.0), r);
    r = det != 0.0 ? r : 0.0;   // cvInvert returns a zero matrix for a singular input
    X[0] = fma(c02, b[2], fma(c01, b[1], c00 * b[0])) * r;
    X[1] = fma(c12, b[2], fma(c11, b[1], c01 * b[0])) * r;
    X[2] = fma(c22, b[2], fma(c12, b[1], c02 * b[0])) * r;
}

// triangulate_point_fast solved in the camera's frame, for a camera matrix in the standard form (cam_std).  The
// residuals P_i X - F_i are the same functions of the point in any frame reached by a rigid motion, so the
// least-squares point is the same and so is the conditioning of the normal equations.  With the camera at the
// origin, its rows become [fx, 0, cx - uc] and [0, fy, cy - vc] with F = 0: 73 FP64 operations instead of 84,
// including the 9 that take the point back to the world frame.
__device__ __forceinline__ void triangulate_point_camframe(const DeviceCalib& cal, double uc, double vc, double up,
                                                           double vp, double* X)
{
    const double* __restrict__ A = cal.Apc;
    const double du = cal.Kc[2] - uc, dv = cal.Kc[5] - vc;
    double P2[3], P3[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        P2[j] = fma(-up, A[8 + j], A[0 + j]);
        P3[j] = fma(-vp, A[8 + j], A[4 + j]);
    }
    const double F2 = fma(A[11], up, -A[3]);
    const double F3 = fma(A[11], vp, -A[7]);
#define S3D_DOT2(a, b, c0) fma(P3[a], P3[b], fma(P2[a], P2[b], c0))
    const double S00 = S3D_DOT2(0, 0, cal.fx2), S01 = fma(P3[0], P3[1], P2[0] * P2[1]);
    const double S02 = S3D_DOT2(0, 2, cal.Kc[0] * du);
    const double S11 = S3D_DOT2(1, 1, cal.fy2), S12 = S3D_DOT2(1, 2, cal.Kc[4] * dv);
    const double S22 = S3D_DOT2(2, 2, fma(dv, dv, du * du));
#undef S3D_DOT2
    double b[3];
#pragma unroll
    for (int j = 0; j < 3; j++) b[j] = fma(P3[j], F3, P2[j] * F2);
    const double c00 = fma(S11, S22, -S12 * S12);
    const double c01 = fma(S02, S12, -S01 * S22);
    const double c02 = fma(S01, S12, -S02 * S11);
    const double c11 = fma(S00, S22, -S02 * S02);
    const double c12 = fma(S01, S02, -S00 * S12);
    const double c22 = fma(S00, S11, -S01 * S01);
    const double det = fma(S02, c02, fma(S01, c01, S00 * c00));
    // one Newton step on the 20-bit seed leaves 1/det within ~2^-40 relative, far inside the mode's 1e-6 bound
    // against the reference order (the world-frame solve above takes two)
    double r = rcp_seed(det);
    r = fma(r, fma(-det, r, 1.0), r);
    const double x0 = fma(c02, b[2], fma(c01, b[1], c00 * b[0])) * r;
    const double x1 = fma(c12, b[2], fma(c11, b[1], c01 * b[0])) * r;
    const double x2 = fma(c22, b[2], fma(c12, b[1], c02 * b[0])) * r;
    if (det == 0.0) {   // cvInvert returns a zero matrix for a singular input: the world origin
        X[0] = X[1] = X[2] = 0.0;
        return;
    }
#pragma unroll
    for (int i = 0; i < 3; i++) X[i] = fma(cal.Rct[3 * i + 2], x2, fma(cal.Rct[3 * i + 1], x1, fma(cal.Rct[3 * i], x0, cal.oc[i])));
}

// ---------------------------------------------------------------------------------------
// closed form of the raster mask recurrence (3/wrapped_phase.cpp:266-279); see DESIGN.md.
// inv(x,y) must return true for a pixel whose ROI flag != 1; coordinates are GLOBAL.
// ---------------------------------------------------------------------------------------
template <class InvFn>
__device__ __forceinline__ bool mask_trigger(int x, int y, int W, int H, InvFn inv)
{
    auto border = [&](int qx, int qy) { return qx == 0 || qy == 0 || qx == W - 1 || qy == H - 1; };
    // LATE = {R, DL, D, DR}; EARLY = {UL, U, UR, L}
    auto late_any = [&](int qx, int qy) {
        return inv(qx + 1, qy) || inv(qx - 1, qy + 1) || inv(qx, qy + 1) || inv(qx + 1, qy + 1);
    };
    if (late_any(x, y)) return true;
    const int ex[4] = {-1, 0, 1, -1}, ey[4] = {-1, -1, -1, 0};
    bool trig = false;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int qx = x + ex[k], qy = y + ey[k];
        if (!inv(qx, qy)) continue;
        if (border(qx, qy)) { trig = true; continue; }
        bool E = late_any(qx, qy);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int rx = qx + ex[j], ry = qy + ey[j];
            E = E || (border(rx, ry) && inv(rx, ry));
        }
        trig = trig || !E;
    }
    return trig;
}

}  // namespace s3d
