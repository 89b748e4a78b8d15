// scan3d_align_math.h -- the arithmetic of the scan-to-model alignment (scan3d_align_to_voxels*): point-to-plane ICP of
// a source cloud against the merged voxel cloud.  Written once for the CUDA kernels (scan3d_align_kernels.cu) and for
// a host build of the very same expressions that the CPU tests compare with an independent numpy restatement
// (tests/test_align_math_host.py compiles this header with g++ -ffp-contract=off).
//
// T is the row-major 3x4 block [R | t] of the 4x4 estimate, p_model = T p_source.  Every double operation below is one
// correctly rounded IEEE operation (S3A_*), in this order, no FMA:
//
//   transform   p'_i = ((T[4i] x + T[4i+1] y) + T[4i+2] z) + T[4i+3], x, y, z the float coordinates as doubles
//   cell        S = (double)max_distance * (1 + 2^-20); per axis c = floor(v / S) in [-2^20, 2^20), else no cell
//               (the margin makes every point within max_distance of p' lie in the 27 cells around p''s cell)
//   distance    d = ((dx dx + dy dy) + dz dz), dx = p'_x - (double)q_x, ...; pair when d <= r2 = md * md, md =
//               (double)max_distance; the candidate with the smaller d wins, a tie goes to the smaller voxel ordinal
//   row         J = [p' x n, n] with (p' x n)_0 = p'_y n_z - p'_z n_y, _1 = p'_z n_x - p'_x n_z, _2 = p'_x n_y - p'_y n_x;
//               r = (dx n_x + dy n_y) + dz n_z
//   sums        s[0..20] = J_i J_j (i <= j, row-major upper triangle), s[21..26] = J_i r, s[27] = r r; per sample the
//               products are added to running sums that start at +0
//   solve       mu = 1e-6 * (trace(A) / 6), trace summed in index order; M = A + mu I; LDL^T: for column j,
//               D_j = M_jj - sum_k<j (L_jk L_jk) D_k, L_ij = (M_ij - sum_k<j (L_ik L_jk) D_k) / D_j (sums in k order);
//               the pivot test fails unless mu is finite and > 0 and every D_j > mu / 2; then y = -b - L y (forward),
//               z = y / D, x = z - L^T x (backward, k ascending); x = (omega, v) must be finite
//   rotation    th2 = (w0 w0 + w1 w1) + w2 w2; th2 == 0: dR = I; th2 not finite: failure; th = sqrt(th2), k = w / th;
//               sin and cos of h = th / 2 by halving h (exactly) to <= 1/8, Taylor polynomials in nested form
//               (sin: t (1 - t2/6 (1 - t2/20 (1 - t2/42 (1 - t2/72 (1 - t2/110))))), cos: 1 - t2/2 (1 - t2/12 (1 -
//               t2/30 (1 - t2/56 (1 - t2/90)))), t2 = t t, each t2/m one division), then the same number of doublings
//               s' = (2 s) c, c' = 1 - (2 s) s; s = (2 sh) ch, c1 = (2 sh) sh, c = 1 - c1;
//               dR_ij = ((i == j ? c : 0) + (c1 k_i) k_j) + s K_ij, K = [[0, -k2, k1], [k2, 0, -k0], [-k1, k0, 0]]
//   update      T'_ij = ((dR_i0 T_0j + dR_i1 T_1j) + dR_i2 T_2j) (+ v_i for j = 3)
//   stop        |v| = sqrt((v0 v0 + v1 v1) + v2 v2); converged when (stop_rotation > 0 or stop_translation > 0) and
//               th <= stop_rotation and |v| <= stop_translation
//   rms         sqrt(s[27] / pairs), 0 without pairs
// Transcendental functions are avoided on purpose: the device's and the host's sin / cos are not the same function.
#pragma once
#include "scan3d_aux_math.h"
#include "scan3d_voxel_math.h"

#if defined(__CUDA_ARCH__)
#define S3L_SQRT(a) __dsqrt_rn(a)
#define S3L_UNROLL _Pragma("unroll")   // constant indices keep the small matrices in registers
#else
#define S3L_SQRT(a) sqrt((double)(a))
#define S3L_UNROLL
#endif

namespace s3l {

constexpr int NSUM = 28;                    // 21 of J^T J, 6 of J^T r, r^2
constexpr double CELL_MARGIN = 1.0 + 1.0 / 1048576.0;
constexpr double DAMPING = 1e-6;

// p' = T p
S3A_HD void transform(const double* T, float x, float y, float z, double p[3])
{
    S3L_UNROLL
    for (int i = 0; i < 3; i++)
        p[i] = S3A_ADD(S3A_ADD(S3A_ADD(S3A_MUL(T[4 * i], (double)x), S3A_MUL(T[4 * i + 1], (double)y)),
                               S3A_MUL(T[4 * i + 2], (double)z)),
                       T[4 * i + 3]);
}

S3A_HD double cell_edge(float max_distance) { return S3A_MUL((double)max_distance, CELL_MARGIN); }

// the cell of v along one axis; false when v is not finite or the cell is outside [-2^20, 2^20)
S3A_HD bool cell_axis(double v, double S, long long* c)
{
    if (!(v - v == 0.0)) return false;
    const double f = floor(S3A_DIV(v, S));
    if (!(f >= (double)s3v::I_MIN && f < (double)s3v::I_MAX)) return false;
    *c = (long long)f;
    return true;
}

S3A_HD bool cell_of(const double p[3], double S, long long c[3])
{
    return cell_axis(p[0], S, &c[0]) && cell_axis(p[1], S, &c[1]) && cell_axis(p[2], S, &c[2]);
}

S3A_HD double dist2(const double p[3], float qx, float qy, float qz)
{
    const double dx = S3A_SUB(p[0], (double)qx), dy = S3A_SUB(p[1], (double)qy), dz = S3A_SUB(p[2], (double)qz);
    return S3A_ADD(S3A_ADD(S3A_MUL(dx, dx), S3A_MUL(dy, dy)), S3A_MUL(dz, dz));
}

// candidate (d, ord) beats the best so far
S3A_HD bool closer(double d, uint32_t ord, double best_d, uint32_t best_ord)
{
    return d < best_d || (d == best_d && ord < best_ord);
}

// the point-to-plane residual (p' - q) . n_q of a pair
S3A_HD double residual(const double p[3], float qx, float qy, float qz, float nx, float ny, float nz)
{
    const double dx = S3A_SUB(p[0], (double)qx), dy = S3A_SUB(p[1], (double)qy), dz = S3A_SUB(p[2], (double)qz);
    return S3A_ADD(S3A_ADD(S3A_MUL(dx, (double)nx), S3A_MUL(dy, (double)ny)), S3A_MUL(dz, (double)nz));
}

// the Jacobian row and the residual of a pair (p', q, n_q)
S3A_HD void row(const double p[3], float qx, float qy, float qz, float nx, float ny, float nz, double J[6], double* r)
{
    const double n0 = nx, n1 = ny, n2 = nz;
    J[0] = S3A_SUB(S3A_MUL(p[1], n2), S3A_MUL(p[2], n1));
    J[1] = S3A_SUB(S3A_MUL(p[2], n0), S3A_MUL(p[0], n2));
    J[2] = S3A_SUB(S3A_MUL(p[0], n1), S3A_MUL(p[1], n0));
    J[3] = n0;
    J[4] = n1;
    J[5] = n2;
    *r = residual(p, qx, qy, qz, nx, ny, nz);
}

// s += the products of one pair
S3A_HD void accumulate(const double J[6], double r, double s[NSUM])
{
    int k = 0;
    S3L_UNROLL
    for (int i = 0; i < 6; i++)
        S3L_UNROLL
        for (int j = i; j < 6; j++, k++) s[k] = S3A_ADD(s[k], S3A_MUL(J[i], J[j]));
    S3L_UNROLL
    for (int i = 0; i < 6; i++) s[21 + i] = S3A_ADD(s[21 + i], S3A_MUL(J[i], r));
    s[27] = S3A_ADD(s[27], S3A_MUL(r, r));
}

// position of A_ij (i <= j) in the upper-triangle sums
S3A_HD int upper(int i, int j) { return i * 6 - (i * (i - 1)) / 2 + (j - i); }

// (A + mu I) x = -b by LDL^T; false when the pivot test fails or x is not finite
S3A_HD bool solve6(const double s[NSUM], double x[6])
{
    double tr = s[upper(0, 0)];
    S3L_UNROLL
    for (int i = 1; i < 6; i++) tr = S3A_ADD(tr, s[upper(i, i)]);
    const double mu = S3A_MUL(DAMPING, S3A_DIV(tr, 6.0));
    if (!(mu > 0.0 && mu - mu == 0.0)) return false;
    const double half_mu = S3A_MUL(mu, 0.5);
    double L[6][6], D[6];
    S3L_UNROLL
    for (int j = 0; j < 6; j++) {
        double d = S3A_ADD(s[upper(j, j)], mu);
        S3L_UNROLL
        for (int k = 0; k < j; k++) d = S3A_SUB(d, S3A_MUL(S3A_MUL(L[j][k], L[j][k]), D[k]));
        if (!(d > half_mu)) return false;
        D[j] = d;
        S3L_UNROLL
        for (int i = j + 1; i < 6; i++) {
            double v = s[upper(j, i)];
            S3L_UNROLL
            for (int k = 0; k < j; k++) v = S3A_SUB(v, S3A_MUL(S3A_MUL(L[i][k], L[j][k]), D[k]));
            L[i][j] = S3A_DIV(v, d);
        }
    }
    double y[6];
    S3L_UNROLL
    for (int i = 0; i < 6; i++) {
        double v = -s[21 + i];
        S3L_UNROLL
        for (int k = 0; k < i; k++) v = S3A_SUB(v, S3A_MUL(L[i][k], y[k]));
        y[i] = v;
    }
    S3L_UNROLL
    for (int i = 5; i >= 0; i--) {
        double v = S3A_DIV(y[i], D[i]);
        S3L_UNROLL
        for (int k = i + 1; k < 6; k++) v = S3A_SUB(v, S3A_MUL(L[k][i], x[k]));
        x[i] = v;
    }
    S3L_UNROLL
    for (int i = 0; i < 6; i++)
        if (!(x[i] - x[i] == 0.0)) return false;
    return true;
}

// sin and cos of h >= 0 (finite)
S3A_HD void sincos_halving(double h, double* sn, double* cs)
{
    double t = h;
    int m = 0;
    while (t > 0.125) {
        t = S3A_MUL(t, 0.5);
        m++;
    }
    const double t2 = S3A_MUL(t, t);
    double a = S3A_SUB(1.0, S3A_DIV(t2, 110.0));
    a = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 72.0), a));
    a = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 42.0), a));
    a = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 20.0), a));
    a = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 6.0), a));
    double s = S3A_MUL(t, a);
    double b = S3A_SUB(1.0, S3A_DIV(t2, 90.0));
    b = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 56.0), b));
    b = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 30.0), b));
    b = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 12.0), b));
    double c = S3A_SUB(1.0, S3A_MUL(S3A_DIV(t2, 2.0), b));
    for (; m > 0; m--) {
        const double s2 = S3A_MUL(2.0, s);
        const double ns = S3A_MUL(s2, c);
        c = S3A_SUB(1.0, S3A_MUL(s2, s));
        s = ns;
    }
    *sn = s;
    *cs = c;
}

// dR = Rodrigues(w) (row-major 3x3), *th = |w|; false when |w|^2 is not finite
S3A_HD bool rodrigues(const double w[3], double dR[9], double* th)
{
    const double th2 = S3A_ADD(S3A_ADD(S3A_MUL(w[0], w[0]), S3A_MUL(w[1], w[1])), S3A_MUL(w[2], w[2]));
    if (!(th2 - th2 == 0.0)) return false;
    if (th2 == 0.0) {
        S3L_UNROLL
        for (int k = 0; k < 9; k++) dR[k] = k % 4 == 0 ? 1.0 : 0.0;
        *th = 0.0;
        return true;
    }
    const double t = S3L_SQRT(th2);
    const double k[3] = {S3A_DIV(w[0], t), S3A_DIV(w[1], t), S3A_DIV(w[2], t)};
    double sh, ch;
    sincos_halving(S3A_MUL(t, 0.5), &sh, &ch);
    const double sh2 = S3A_MUL(2.0, sh);
    const double s = S3A_MUL(sh2, ch), c1 = S3A_MUL(sh2, sh), c = S3A_SUB(1.0, c1);
    const double K[9] = {0.0, -k[2], k[1], k[2], 0.0, -k[0], -k[1], k[0], 0.0};
    S3L_UNROLL
    for (int i = 0; i < 3; i++)
        S3L_UNROLL
        for (int j = 0; j < 3; j++)
            dR[3 * i + j] = S3A_ADD(S3A_ADD(i == j ? c : 0.0, S3A_MUL(S3A_MUL(c1, k[i]), k[j])), S3A_MUL(s, K[3 * i + j]));
    *th = t;
    return true;
}

// T <- [dR | v] T
S3A_HD void compose(const double dR[9], const double v[3], double T[12])
{
    double o[12];
    S3L_UNROLL
    for (int i = 0; i < 3; i++)
        S3L_UNROLL
        for (int j = 0; j < 4; j++) {
            double e = S3A_ADD(S3A_ADD(S3A_MUL(dR[3 * i], T[j]), S3A_MUL(dR[3 * i + 1], T[4 + j])),
                               S3A_MUL(dR[3 * i + 2], T[8 + j]));
            o[4 * i + j] = j == 3 ? S3A_ADD(e, v[i]) : e;
        }
    S3L_UNROLL
    for (int k = 0; k < 12; k++) T[k] = o[k];
}

S3A_HD bool converged(double th, const double v[3], double stop_rotation, double stop_translation)
{
    const double tn = S3L_SQRT(S3A_ADD(S3A_ADD(S3A_MUL(v[0], v[0]), S3A_MUL(v[1], v[1])), S3A_MUL(v[2], v[2])));
    return (stop_rotation > 0.0 || stop_translation > 0.0) && th <= stop_rotation && tn <= stop_translation;
}

S3A_HD double rms(double sum_r2, long long pairs)
{
    return pairs > 0 ? S3L_SQRT(S3A_DIV(sum_r2, (double)pairs)) : 0.0;
}

}  // namespace s3l
