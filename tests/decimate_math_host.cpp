// Host build of 3dscan_b200/common/scan3d_decimate_math.h for tests/test_decimate_math_host.py (g++ -ffp-contract=off):
// every function over arrays, so numpy can compare whole batches bit for bit.
#include <math.h>
#include <stdint.h>

#include "../3dscan_b200/common/scan3d_decimate_math.h"

extern "C" {

// faces [n][3][3] float (corners a, b, c): u [n][3], w [n], ok [n]
void s3q_host_face_planes(const float* p, long long n, double H, double* u, double* w, int32_t* ok)
{
    for (long long i = 0; i < n; i++) {
        const float* f = p + 9 * i;
        u[3 * i] = u[3 * i + 1] = u[3 * i + 2] = w[i] = 0.0;
        ok[i] = s3q::face_plane(f, f + 3, f + 6, H, u + 3 * i, w + i);
    }
}

void s3q_host_corner_coeffs(const double* u, const double* w, const double* f, long long n, long long* q)
{
    for (long long i = 0; i < n; i++) s3q::corner_coeffs(u + 3 * i, w[i], f + 3 * i, q + s3q::NQ * i);
}

void s3q_host_fractions(const float* x, long long n, double H, double* f)
{
    for (long long i = 0; i < n; i++) f[i] = s3q::fraction(x[i], H);
}

void s3q_host_to_fixed(const double* v, long long n, long long* q)
{
    for (long long i = 0; i < n; i++) q[i] = s3q::to_fixed(v[i]);
}

void s3q_host_place(const long long* qs, const unsigned long long* sq, const uint32_t* cnt, long long n, double* y,
                    int32_t* status)
{
    for (long long i = 0; i < n; i++) status[i] = s3q::place(qs + s3q::NQ * i, sq + 3 * i, cnt[i], y + 3 * i);
}

void s3q_host_coords(const long long* ijk, const double* y, long long n, double H, float* out)
{
    for (long long i = 0; i < 3 * n; i++) out[i] = s3q::coord(ijk[i], y[i], H);
}

void s3q_host_canonical(const int32_t* t, long long n, int32_t* out, uint8_t* col)
{
    for (long long i = 0; i < n; i++) {
        col[i] = s3q::collapsed(t[3 * i], t[3 * i + 1], t[3 * i + 2]);
        s3q::canonical(t[3 * i], t[3 * i + 1], t[3 * i + 2], out + 3 * i);
    }
}

double s3q_host_face_bound(double r) { return s3q::face_bound(r); }
double s3q_host_sum_bound(double r) { return s3q::sum_bound(r); }
int s3q_host_p() { return s3q::P; }
double s3q_host_damping() { return s3q::DAMPING; }
}
