// Host build of 3dscan_b200/common/scan3d_smooth_math.h for tests/test_smooth_math_host.py (g++ -ffp-contract=off):
// every function over arrays, so numpy can compare whole batches bit for bit.
#include <math.h>
#include <stdint.h>

#include "../3dscan_b200/common/scan3d_smooth_math.h"

extern "C" {

int s3t_host_exponent(const float* x, long long n)
{
    unsigned int field = 0;
    for (long long i = 0; i < n; i++) {
        const unsigned int f = s3t::exponent_field(x[i]);
        field = f > field ? f : field;
    }
    return s3t::exponent(field);
}

void s3t_host_quantise(const float* x, long long n, int E, long long* q)
{
    for (long long i = 0; i < n; i++) q[i] = s3t::quantise(x[i], E);
}

void s3t_host_dequantise(const long long* q, long long n, int E, float* x)
{
    for (long long i = 0; i < n; i++) x[i] = s3t::dequantise(q[i], E);
}

void s3t_host_update(const long long* q, const long long* s, const uint32_t* d, long long n, double k, long long* out,
                     uint8_t* over)
{
    for (long long i = 0; i < n; i++) {
        out[i] = s3t::update(q[i], s[i], d[i], k);
        over[i] = s3t::over_limit(out[i]);
    }
}

// faces [n][3][3] float (corners a, b, c): m [n][3], ok [n]
void s3t_host_face_normals(const float* p, long long n, long long* m, uint8_t* ok)
{
    for (long long i = 0; i < n; i++) {
        const float* f = p + 9 * i;
        m[3 * i] = m[3 * i + 1] = m[3 * i + 2] = 0;
        ok[i] = s3t::face_normal(f, f + 3, f + 6, m + 3 * i);
    }
}

void s3t_host_normal_out(const long long* s, long long n, float* out)
{
    for (long long i = 0; i < n; i++) s3v::normal_out(s[3 * i], s[3 * i + 1], s[3 * i + 2], out + 3 * i);
}

void s3t_host_displacement(const float* a, const float* b, long long n, double* out)
{
    for (long long i = 0; i < n; i++) out[i] = s3t::displacement(a + 3 * i, b + 3 * i);
}

void s3t_host_limits(long long* out)
{
    out[0] = s3t::P;
    out[1] = s3t::Q_LIMIT;
    out[2] = s3t::DEGREE_LIMIT;
    out[3] = s3t::E_MIN;
}
}
