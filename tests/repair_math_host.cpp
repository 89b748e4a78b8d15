// Host build of 3dscan_b200/common/scan3d_repair_math.h for tests/test_repair_math_host.py (g++ -ffp-contract=off):
// the face key and the per-edge keep rule over arrays, so numpy can compare them bit for bit.
#include <stdint.h>

#include "../3dscan_b200/common/scan3d_repair_math.h"

extern "C" {

// faces [n][3][3] float (corners a, b, c) with face indices idx [n]: keys [n]
void s3r_host_face_key(const float* p, const uint32_t* idx, long long n, unsigned long long* keys)
{
    for (long long i = 0; i < n; i++) keys[i] = s3r::face_key(p + 9 * i, p + 9 * i + 3, p + 9 * i + 6, idx[i]);
}

// kept [n] = the edge rule for key k with the edge's m0, m1 and second
void s3r_host_kept(const unsigned long long* k, const unsigned long long* m0, const unsigned long long* m1,
                   const unsigned long long* second, long long n, uint8_t* kept)
{
    for (long long i = 0; i < n; i++) kept[i] = s3r::kept_on_edge(k[i], m0[i], m1[i], second[i]);
}
}
