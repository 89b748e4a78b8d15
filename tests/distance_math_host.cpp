// Host build of 3dscan_b200/common/scan3d_distance_math.h for tests/test_distance_math_host.py (g++ -ffp-contract=off):
// the squared distance and the side of point-face pairs, the signed distance, and the cell box and entry count of
// faces, over arrays, so numpy can compare them bit for bit.
#include <stdint.h>

#include "../3dscan_b200/common/scan3d_distance_math.h"

extern "C" {

// p [n][3] float, corners [n][3][3] float: d2 and s [n], the signed distance [n]
void s3p_host_pairs(const float* p, const float* corners, long long n, double* d2, double* s, float* sd)
{
    for (long long i = 0; i < n; i++) {
        const double q[3] = {p[3 * i], p[3 * i + 1], p[3 * i + 2]};
        d2[i] = s3p::face_distance(q, corners + 9 * i, corners + 9 * i + 3, corners + 9 * i + 6, &s[i]);
        sd[i] = s3p::signed_distance(d2[i], s[i]);
    }
}

// corners [n][3][3] float, R: the cell boxes lo, hi [n][3], ok [n], entries [n] (clamped at 2^32)
void s3p_host_cells(const float* corners, long long n, float R, long long* lo, long long* hi, int* ok,
                    unsigned long long* entries)
{
    const double S = s3l::cell_edge(R);
    for (long long i = 0; i < n; i++) {
        ok[i] = s3p::face_cells(corners + 9 * i, corners + 9 * i + 3, corners + 9 * i + 6, S, lo + 3 * i, hi + 3 * i);
        entries[i] = ok[i] ? s3p::face_entries(lo + 3 * i, hi + 3 * i) : 0;
    }
}
}
