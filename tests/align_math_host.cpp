// Host build of 3dscan_b200/common/scan3d_align_math.h (the very expressions the CUDA kernels of
// scan3d_align_kernels.cu evaluate): the per-element functions, and a sequential point-to-plane ICP built from them --
// a cell map of the model and a 27-cell search -- so that the CPU test suite can compare both with numpy without a GPU.
// Built by tests/test_align_math_host.py with g++ -O2 -ffp-contract=off.
#include <stddef.h>
#include <stdint.h>

#include <unordered_map>
#include <vector>

#include "../3dscan_b200/common/scan3d_align_math.h"
#include "../include/scan3d.h"

extern "C" {

void s3l_host_transform(const double* T, const float* xyz, long long n, double* out)
{
    for (long long i = 0; i < n; i++) s3l::transform(T, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], out + 3 * i);
}

// cells [n][3] of points p [n][3]; ok[n]
void s3l_host_cells(const double* p, long long n, float max_distance, long long* cells, uint8_t* ok)
{
    const double S = s3l::cell_edge(max_distance);
    for (long long i = 0; i < n; i++) ok[i] = s3l::cell_of(p + 3 * i, S, cells + 3 * i);
}

void s3l_host_dist2(const double* p, const float* q, long long n, double* out)
{
    for (long long i = 0; i < n; i++) out[i] = s3l::dist2(p + 3 * i, q[3 * i], q[3 * i + 1], q[3 * i + 2]);
}

int s3l_host_closer(double d, uint32_t ord, double best_d, uint32_t best_ord) { return s3l::closer(d, ord, best_d, best_ord); }

void s3l_host_rows(const double* p, const float* q, const float* nrm, long long n, double* J, double* r)
{
    for (long long i = 0; i < n; i++)
        s3l::row(p + 3 * i, q[3 * i], q[3 * i + 1], q[3 * i + 2], nrm[3 * i], nrm[3 * i + 1], nrm[3 * i + 2], J + 6 * i,
                 r + i);
}

// the sums of n rows, sequentially
void s3l_host_sums(const double* J, const double* r, long long n, double* s)
{
    for (int k = 0; k < s3l::NSUM; k++) s[k] = 0.0;
    for (long long i = 0; i < n; i++) s3l::accumulate(J + 6 * i, r[i], s);
}

int s3l_host_solve(const double* s, double* x) { return s3l::solve6(s, x); }

int s3l_host_rodrigues(const double* w, double* R, double* th) { return s3l::rodrigues(w, R, th); }

void s3l_host_sincos(double h, double* sn, double* cs) { s3l::sincos_halving(h, sn, cs); }

void s3l_host_compose(const double* dR, const double* v, double* T) { s3l::compose(dR, v, T); }

// The whole alignment, sequentially: model = m points with normals (those with a zero normal are skipped), source n
// points, sample j = point j * stride.  T (12 doubles) holds T_init on entry and the result on return.
// info: [iterations, status, pairs_first, pairs_last]; rms: [first, last].
void s3l_host_icp(const float* mxyz, const float* mnrm, long long m, const float* src, long long n, double* T,
                  float max_distance, int max_iterations, int stride, double stop_rotation, double stop_translation,
                  long long* info, double* rms)
{
    const double S = s3l::cell_edge(max_distance);
    const double md = (double)max_distance;
    const double r2 = S3A_MUL(md, md);
    std::unordered_map<unsigned long long, std::vector<uint32_t>> cells;
    for (long long o = 0; o < m; o++) {
        const float* q = mxyz + 3 * o;
        const float* nq = mnrm + 3 * o;
        if (nq[0] == 0.0f && nq[1] == 0.0f && nq[2] == 0.0f) continue;
        const double p[3] = {q[0], q[1], q[2]};
        long long c[3];
        if (!s3l::cell_of(p, S, c)) continue;
        cells[s3v::pack_key(c[0], c[1], c[2])].push_back((uint32_t)o);
    }
    int iterations = 0, status = 1;
    long long pairs_first = 0, pairs_last = 0;
    double rms_first = 0.0, rms_last = 0.0;
    for (int it = 0; it < max_iterations; it++) {
        double s[s3l::NSUM];
        for (int k = 0; k < s3l::NSUM; k++) s[k] = 0.0;
        long long pairs = 0;
        for (long long j = 0; j * stride < n; j++) {
            const float* x = src + 3 * (j * stride);
            double p[3];
            s3l::transform(T, x[0], x[1], x[2], p);
            long long c[3];
            if (!s3l::cell_of(p, S, c)) continue;
            double best = 0.0;
            uint32_t best_o = 0xffffffffu;
            for (int dz = -1; dz <= 1; dz++)
                for (int dy = -1; dy <= 1; dy++)
                    for (int dx = -1; dx <= 1; dx++) {
                        const long long a = c[0] + dx, b = c[1] + dy, e = c[2] + dz;
                        if (a < s3v::I_MIN || a >= s3v::I_MAX || b < s3v::I_MIN || b >= s3v::I_MAX || e < s3v::I_MIN ||
                            e >= s3v::I_MAX)
                            continue;
                        auto f = cells.find(s3v::pack_key(a, b, e));
                        if (f == cells.end()) continue;
                        for (uint32_t o : f->second) {
                            const double d = s3l::dist2(p, mxyz[3 * o], mxyz[3 * o + 1], mxyz[3 * o + 2]);
                            if (d <= r2 && (best_o == 0xffffffffu || s3l::closer(d, o, best, best_o))) {
                                best = d;
                                best_o = o;
                            }
                        }
                    }
            if (best_o == 0xffffffffu) continue;
            double J[6], r;
            s3l::row(p, mxyz[3 * best_o], mxyz[3 * best_o + 1], mxyz[3 * best_o + 2], mnrm[3 * best_o],
                     mnrm[3 * best_o + 1], mnrm[3 * best_o + 2], J, &r);
            s3l::accumulate(J, r, s);
            pairs++;
        }
        if (it == 0) {
            pairs_first = pairs;
            rms_first = s3l::rms(s[27], pairs);
        }
        pairs_last = pairs;
        rms_last = s3l::rms(s[27], pairs);
        double x[6], dR[9], th;
        if (pairs < 6 || !s3l::solve6(s, x) || !s3l::rodrigues(x, dR, &th)) {
            status = 2;
            break;
        }
        s3l::compose(dR, x + 3, T);
        iterations++;
        if (s3l::converged(th, x + 3, stop_rotation, stop_translation)) {
            status = 0;
            break;
        }
    }
    info[0] = iterations;
    info[1] = status;
    info[2] = pairs_first;
    info[3] = pairs_last;
    rms[0] = rms_first;
    rms[1] = rms_last;
}
}

// the field layout of the public structs, for the ctypes mirror
extern "C" void s3l_host_layout(long long* out)
{
    out[0] = sizeof(scan3d_align_params);
    out[1] = offsetof(scan3d_align_params, max_distance);
    out[2] = offsetof(scan3d_align_params, max_iterations);
    out[3] = offsetof(scan3d_align_params, stride);
    out[4] = offsetof(scan3d_align_params, stop_rotation);
    out[5] = offsetof(scan3d_align_params, stop_translation);
    out[6] = offsetof(scan3d_align_params, apply);
    out[7] = sizeof(scan3d_align_result);
    out[8] = offsetof(scan3d_align_result, iterations);
    out[9] = offsetof(scan3d_align_result, status);
    out[10] = offsetof(scan3d_align_result, pairs_first);
    out[11] = offsetof(scan3d_align_result, pairs_last);
    out[12] = offsetof(scan3d_align_result, rms_first);
    out[13] = offsetof(scan3d_align_result, rms_last);
}
