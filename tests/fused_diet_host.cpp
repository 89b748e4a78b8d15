// fused_diet_host.cpp -- HOST build of the identities that let k_fused7 drop FP64 work, for the CPU test suite
// (tests/test_fused_diet_host.py):
//   * the fast triangulation solved in the camera's frame (triangulate_point_camframe) against the world-frame
//     fast solve (triangulate_point_fast);
//   * correspond32_finite against correspond32 on the phases the single-pass kernel can produce;
//   * the table of unwrap terms code*2.0*Pi against the exact quotient it replaces.
// Built like tests/fused_math_host.cpp: g++ -O2 -std=c++17 -ffp-contract=off -I/usr/local/cuda/include -shared -fPIC
#include "cuda_host_shim.h"

#include "../3dscan_b200/csrc/scan3d_math.cuh"

using namespace s3d;

extern "C" {

// n correspondences (uc, vc) <-> (up, vp); Kc row-major, Rc row-major rotation, tc, and the world matrices
// Ac = Kc[Rc|tc], Ap (3x4 row-major).  Writes both solves' points (n x 3) and returns cam_std.
int s3d_host_camframe(const double* Kc, const double* Rc, const double* tc, const double* Ac, const double* Ap, int n,
                      const double* uc, const double* vc, const double* up, const double* vp, double* x_fast,
                      double* x_cam)
{
    DeviceCalib cal{};
    memcpy(cal.Ac, Ac, sizeof(cal.Ac));
    memcpy(cal.Ap, Ap, sizeof(cal.Ap));
    memcpy(cal.Kc, Kc, sizeof(cal.Kc));
    camera_frame_calib(Kc, Rc, tc, Ap, &cal);
    for (int i = 0; i < n; i++) {
        triangulate_point_fast(cal.Ac, cal.Ap, uc[i], vc[i], up[i], vp[i], x_fast + 3 * i);
        triangulate_point_camframe(cal, uc[i], vc[i], up[i], vp[i], x_cam + 3 * i);
    }
    return Kc[1] == 0.0 && Kc[3] == 0.0 && Kc[6] == 0.0 && Kc[7] == 0.0 && Kc[8] == 1.0;
}

// The unwrap term table against the 3-operation exact quotient it replaces: n fringe orders, n_w wrapped phases each.
// Returns the number of (code, w) pairs whose unwrapped phases differ, or -1 if a table entry differs.
int s3d_host_code_term(int n, const float* w, int n_w)
{
    double* t = new double[n];
    fill_code_term_table(t, n);
    int bad = 0;
    for (int code = 0; code < n && bad >= 0; code++) {
        if (t[code] != div_const((double)(code * 44), 7.0, K_RCP_7, true)) bad = -1;
        for (int i = 0; i < n_w && bad >= 0; i++) {
            const float a = unwrap_abs(w[i], code, true), b = unwrap_abs_k(w[i], t[code]);
            if (memcmp(&a, &b, 4) != 0) bad++;
        }
    }
    delete[] t;
    return bad;
}

// The single-pass kernel's unwrapped phase for wrapped phase w and fringe order code (add_pi, unwrap_abs with the
// exact quotient), then correspond32 and correspond32_finite on it.  ok[i] = correspond32's FE_INVALID test.
void s3d_host_correspond(const float* w, const int* code, int n, double fw, float* phi, int* px_old, int* ok,
                         int* px_new)
{
    for (int i = 0; i < n; i++) {
        phi[i] = unwrap_abs(add_pi(w[i]), code[i], true);
        ok[i] = correspond32(phi[i], fw, &px_old[i]);
        px_new[i] = correspond32_finite(phi[i], fw);
    }
}
}
