// Host build of 3dscan_b200/common/scan3d_orient_math.h for tests/test_orient_math_host.py (g++ -ffp-contract=off):
// the centre, the exponent, the per-face volume and area terms and the int128 sum over arrays, so numpy can compare
// them bit for bit.
#include <stdint.h>

#include "../3dscan_b200/common/scan3d_orient_math.h"

extern "C" {

// the centre c [3] of the box lo, hi [3] and the exponent of the points p [m][3] about it
int s3o_host_frame(const float* lo, const float* hi, const float* p, long long m, float* c)
{
    unsigned int field = 0;
    for (int k = 0; k < 3; k++) c[k] = s3o::centre(lo[k], hi[k]);
    for (long long i = 0; i < 3 * m; i++) {
        const unsigned int f = s3o::offset_field(p[i], c[i % 3]);
        field = f > field ? f : field;
    }
    return s3o::exponent(field);
}

// faces [n][3][3] float (corners a, b, c): the volume and area terms [n] about c with exponent E
void s3o_host_terms(const float* p, long long n, const float* c, int E, long long* vol, long long* area)
{
    for (long long i = 0; i < n; i++) {
        vol[i] = s3o::volume_term(p + 9 * i, p + 9 * i + 3, p + 9 * i + 6, c, E);
        area[i] = s3o::area_term(p + 9 * i, p + 9 * i + 3, p + 9 * i + 6, E);
    }
}

// the int128 sum of t [n] as (lo, hi), its sign, and it scaled as a volume and an area with exponent E
int s3o_host_sum(const long long* t, long long n, int E, unsigned long long* lohi, double* va)
{
    unsigned long long lo = 0, hi = 0;
    for (long long i = 0; i < n; i++) s3o::add128(&lo, &hi, t[i]);
    lohi[0] = lo;
    lohi[1] = hi;
    va[0] = s3o::volume(lo, hi, E);
    va[1] = s3o::area(lo, hi, E);
    return s3o::sign128(lo, hi);
}
}
