// scan3d_fused_kernel7.cu -- second-generation fused kernel ("v7").  Same work, same results and
// same warp-specialised idea as the first-generation kernel of round 1 (gone), re-cut so that more consumer warps fit on
// an SM (throughput of this path follows the number of consumer warps: it is latency/issue bound,
// see DESIGN.md section 7):
//
//   * plane outputs (phases, fringe orders, valid, c_p_map) leave straight from registers as
//     vector stores -- each thread owns 4 consecutive pixels -- so nothing but the points is
//     staged in shared memory;
//   * the input slot is therefore dead right after the integer phase: consumers hand it back at
//     once and ONE slot per CTA keeps the loads a full FP64 phase ahead; a tile is loaded by one
//     2-D tensor-map TMA copy ([frames] x [tile bytes]);
//   * a block scan of the valid bits gives every pixel its raster rank BEFORE the triangulation,
//     which then writes each point straight to its rank in one of two small point buffers (a
//     rolled loop: the unrolled version did not fit the instruction cache);
//   * the tile's count is published before its triangulation, by the consumers, so the grid-wide
//     prefix chain (decoupled look-back) runs ahead of the FP64 work;
//   * work-list positions are drawn from a global counter: the CTAs of an SM run at different
//     speeds, and equal static shares made the fast ones wait for the slow one's counts;
//   * producer and epilogue are one "IO warp" running an event loop: issue the next tile's load
//     when the slot frees, note a counted tile, advance a resumable look-back (walking back window
//     after window while the words are there), stream staged tiles out.
//
//   CTA = CW consumer warps + 1 IO warp; shared memory per CTA = NF*T + ROI window + 2*12*T bytes
//   (76.7 KB for the 12 MP config at CW = 7) -> 3 CTAs = 21 consumer warps per SM at 80 registers
//   (the 16 K registers of an SM sub-partition bound the shape, see regs7).  History and
//   measurements: DESIGN.md section 5.1, profiles/r1_optimisation_log.md.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include "scan3d_fused_common.cuh"

// the IO warp's back-off when an event-loop pass found nothing to do (100 / 250 / 600 / 1500 ns measured: no difference)
constexpr unsigned S3D_IO_IDLE_NS = 250;

namespace s3d {

struct Geom7 {
    int T, roi_row, roi_bytes;
};
__host__ __device__ constexpr Geom7 geom7(int T) { return Geom7{T, T + 2 * ROI_HALO, 4 * (T + 2 * ROI_HALO)}; }

constexpr int FIXED7 = 64 /*8 mbarriers*/ + ATAN_TAB_DOUBLES * 8 + 16 /*cur_pos*/ + 128 /*cnt[2][16]*/ + 32 /*pos ring[8]*/;

static int num_frames7(const scan3d_config& c)
{
    return c.dirs == 2 ? 2 * c.N + 2 * (c.M_v + c.M_h) : c.N + 2 * c.M_v;
}
static bool mod7(const scan3d_config& c) { return (c.flags & SCAN3D_FLAG_MODULATION_MASK) != 0; }
static size_t smem7(const scan3d_config& c, int cw)
{
    const int T = 128 * cw;
    // (with the modulation criterion the two directions have their own validity planes: a second ROI window)
    return (size_t)num_frames7(c) * T + geom7(T).roi_bytes * (mod7(c) && c.dirs == 2 ? 2 : 1) +
           (c.dirs == 2 ? 2 * 12 * T + 2 * (T / 4) : 0) + FIXED7;
}

struct Plan7 {
    int cw, minb;
    size_t smem;
};

static bool plan7(const scan3d_config& c, Plan7* out)
{
    if (c.W % 16 != 0) return false;
    if (!(c.N == 3 || c.N == 4 || c.N == 5 || c.N == 8)) return false;
    if (mod7(c) && c.N != 3) return false;
    // Shapes are bounded by the register file of an SM sub-partition (16 K registers): warps are
    // dealt round-robin to the 4 sub-partitions, so ceil(warps per SM / 4) * 32 * regs <= 16384:
    // 24 warps at 80 registers (7, 3), 20 at 96 (9, 2), 16 at 128 (7, 2).  The first shape that fits
    // the shared memory wins; (7, 2) fits every configuration accepted above (at most 76 frames).
    auto fits = [&](int w, int b) {
        const size_t sm = smem7(c, w);
        if ((sm + 1024) * b > (size_t)SMEM_MAX + 1024) return false;
        out->cw = w; out->minb = b; out->smem = sm;
        return true;
    };
    return fits(7, 3) || (!mod7(c) && fits(9, 2)) || fits(7, 2);
}

bool fused7_supported(const scan3d_config& c)
{
    Plan7 p;
    return plan7(c, &p);
}

// does the single-pass kernel for this configuration apply scan3d_set_registration's transform itself?
bool fused7_folds_registration(const scan3d_config& c)
{
    Plan7 p;
    return plan7(c, &p) && c.dirs == 2 && !mod7(c) && p.cw == 7;
}

constexpr int regs7(int cw, int minb)
{
    // per sub-partition: ceil(resident warps / 4) warps share 16384 registers
    const int warps = minb * (cw + 1);
    const int r = 16384 / (((warps + 3) / 4) * 32);
    return r > 255 ? 255 : (r / 8) * 8;
}



// MOD: check_I_mod_criteria's modulation criterion (3/wrapped_phase.cpp:84-104, SCAN3D_FLAG_MODULATION_MASK): a pre-pass
// has written one effective ROI plane per direction (a.roi = vertical, a.roi2 = horizontal); the mask recurrence runs
// on each, so the two directions have their own masks (the reference's valid_map_vertical / _horizontal).
// REG: register_point_clouds' turntable transform applied to every point where it is staged (scan3d_set_registration).
template <int N, int DIRS, int CW, int MINB, bool EXACT, bool MOD = false, bool REG = false, int MV = 0, int MH = 0, int LUTS = -1>
__global__ void __launch_bounds__((CW + 1) * 32) __maxnreg__(regs7(CW, MINB))
k_fused7(const __grid_constant__ FusedArgs a, const __grid_constant__ DeviceCalib cal, const __grid_constant__ CUtensorMap stack_map)
{
    constexpr int T = 128 * CW;
    constexpr int NCONS = 32 * CW;
    constexpr int WPF = T / 4;
    constexpr Geom7 G = geom7(T);

    extern __shared__ __align__(128) uint8_t smem[];
    // MV / MH != 0: the Gray depths as compile-time constants (the named configurations): plane loops without guards,
    // frame offsets as immediates -- 4 % of the kernel time at 10 + 10 bits
    const int M_v = MV ? MV : a.M_v, M_h = MH ? MH : a.M_h;
    // LUTS >= 0: which undistortion tables exist is a compile-time fact (bit 0 camera, bit 1 projector; -1: look at the
    // pointers).  LUTS = 1 is the reference's calibration class: distorted camera, distortion-free projector.
    const bool has_cam_lut = LUTS < 0 ? a.cam_lut != nullptr : (LUTS & 1) != 0;
    const bool has_proj_lut = LUTS < 0 ? a.proj_lut != nullptr : (LUTS & 2) != 0;
    const int NF = DIRS == 2 ? 2 * N + 2 * (M_v + M_h) : N + 2 * M_v;
    uint8_t* slot = smem;
    uint8_t* sroi = smem + (size_t)NF * T;
    constexpr int NROI = (MOD && DIRS == 2) ? 2 : 1;                           // ROI windows: one per direction with MOD
    uint8_t* sroi2 = sroi + (NROI - 1) * G.roi_bytes;
    float* cxb = reinterpret_cast<float*>(sroi + NROI * G.roi_bytes);          // [2][3*T]
    uint8_t* vfl = reinterpret_cast<uint8_t*>(cxb + (DIRS == 2 ? 2 * 3 * T : 0));   // [2][T/4] 4 valid bits per thread
    uint64_t* bars = reinterpret_cast<uint64_t*>(vfl + (DIRS == 2 ? 2 * (T / 4) : 0));
    double* tab = reinterpret_cast<double*>(bars + 8);
    volatile int* ctl = reinterpret_cast<volatile int*>(tab + ATAN_TAB_DOUBLES);   // [0] cur_pos, [1..2] staged_pos
    volatile uint32_t* cnts = reinterpret_cast<volatile uint32_t*>(const_cast<int*>(ctl) + 4);   // [2][16]
    volatile int* posr = reinterpret_cast<volatile int*>(const_cast<uint32_t*>(cnts) + 32);       // [8] list positions of the tiles in flight
    const uint32_t bar_full = smem_u32(bars), bar_free = smem_u32(bars + 1), bar_staged = smem_u32(bars + 2),
                   bar_cxfree = smem_u32(bars + 4), bar_counted = smem_u32(bars + 6);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int W = a.W;
    const int plane = W * a.H;

    if (tid == 0) {
        mbar_init(bar_full, 1);
        mbar_init(bar_free, CW);
        mbar_init(bar_staged, CW);
        mbar_init(bar_staged + 8, CW);
        mbar_init(bar_cxfree, 1);
        mbar_init(bar_cxfree + 8, 1);
        mbar_init(bar_counted, 1);
        mbar_init(bar_counted + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_async_smem();
    }
    for (int i = tid; i < ATAN_TAB_DOUBLES; i += (CW + 1) * 32) tab[i] = a.atan_tab[i];
    __syncthreads();

    // Work-list positions are handed out in order: the IO warp draws the next position from a global
    // counter whenever its slot frees.  The CTAs of an SM do not run at the same speed (the warp
    // schedulers favour the lower warp slots: measured 14k / 15k / 19k cycles per tile for the 1st /
    // 2nd / 3rd CTA of an SM), so equal static shares leave the fast CTAs waiting for the slow one's counts.
    const int n_work = *a.n_list;
    int* const next_pos = a.n_list + a.n_tiles + 8;      // zeroed by k_tile_list

    if (warp == CW) {
        // ================================ IO WARP (producer + epilogue) ================================
        const unsigned long long tag = (unsigned long long)(a.epoch & 0x3fffffffu) << 34;
        const long long roi_total = (long long)W * a.H_total;
        int load_it = 0;                         // next tile to load
        int agg_it = 0;                          // next counted tile whose count gets published
        int epi_it = 0;                          // next tile whose points get streamed out
        bool ended = false;
        bool resolving = false, published = false;
        int look = 0;
        uint32_t excl = 0;
        // per staging buffer (0 / 1): count, list position, "empty tile" -- as scalars selected by the buffer index
        // (arrays indexed by a run-time value live in local memory: ~2 M local accesses and 110 MB of L2 writes per scan)
        uint32_t tot0 = 0, tot1 = 0;
        int epos0 = 0, epos1 = 0;
        bool skip0 = false, skip1 = false;
        while (!ended || (DIRS == 2 && epi_it < load_it)) {
            bool progressed = false;
            // ---- (1) the slot is free again: issue the next tile's loads (or the end marker) ----
            if (!ended && __any_sync(0xffffffffu, mbar_try(bar_free, (load_it & 1) ^ 1))) {
                progressed = true;
                int pos = 0;
                if (lane == 0) pos = atomicAdd(next_pos, 1);
                pos = __shfl_sync(0xffffffffu, pos, 0);
                if (pos < n_work) {
                    const int tile = a.tile_list[pos];
                    const int p0 = tile * T, wt = min(T, plane - p0);
                    const long long gbase = (long long)a.row0 * W + p0 - ROI_HALO;
                    long long seg0 = 0, seg1 = 0;
                    uint32_t roi_tx = 0;
                    if (lane < 4) {
                        seg0 = max(gbase + (long long)(lane - 2) * W, 0LL);
                        seg1 = min(gbase + (long long)(lane - 2) * W + wt + 2 * ROI_HALO, roi_total);
                        if (seg1 > seg0) roi_tx = (uint32_t)(seg1 - seg0);
                    }
                    uint32_t roi_sum = roi_tx;
                    roi_sum += __shfl_xor_sync(0xffffffffu, roi_sum, 1);
                    roi_sum += __shfl_xor_sync(0xffffffffu, roi_sum, 2);
                    roi_sum = __shfl_sync(0xffffffffu, roi_sum, 0);
                    if (lane == 0) {
                        trace(a.trace, load_it, 0);
                        ctl[0] = pos;
                        posr[load_it & 7] = pos;
                        mbar_expect_tx(bar_full, (uint32_t)NF * T + NROI * roi_sum);
                    }
                    __syncwarp();
                    // the whole [NF frames] x [T bytes] tile is ONE 2-D tensor copy (64-bit elements;
                    // bytes past the end of a frame are zero-filled).  56 per-frame bulk copies took the
                    // warp ~5k cycles to issue, squarely on the slot-free -> data-ready path.
                    if (lane == 0) tensor_g2s_2d(smem_u32(slot), &stack_map, p0 >> 3, 0, bar_full);
                    if (roi_tx) {
                        bulk_g2s(smem_u32(sroi) + lane * G.roi_row + (uint32_t)(seg0 - (gbase + (long long)(lane - 2) * W)),
                                 a.roi + seg0, roi_tx, bar_full);
                        if (NROI == 2)
                            bulk_g2s(smem_u32(sroi2) + lane * G.roi_row + (uint32_t)(seg0 - (gbase + (long long)(lane - 2) * W)),
                                     a.roi2 + seg0, roi_tx, bar_full);
                    }
                    if (lane == 0) trace(a.trace, load_it, 1);
                    load_it++;
                } else {
                    if (lane == 0) {
                        ctl[0] = -1;
                        mbar_arrive(bar_full);
                    }
                    ended = true;
                }
            }
            if (DIRS == 2) {
                // ---- (2) a tile's valid pixels are counted (its triangulation is still running; the
                //      consumers have published the count themselves): note it for the look-back ----
                if (agg_it < load_it && agg_it < epi_it + 2 &&
                    __any_sync(0xffffffffu, mbar_try(bar_counted + 8 * (agg_it & 1), (agg_it >> 1) & 1))) {
                    progressed = true;
                    const int b = agg_it & 1;
                    const int pos = posr[agg_it & 7];
                    uint32_t total = lane < CW ? cnts[b * 16 + lane] : 0u;
#pragma unroll
                    for (int o = 16; o; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
                    if (lane == 0) trace(a.trace, agg_it, 5);
                    const bool skip_b = total == 0 && pos != n_work - 1 && pos > 0;
                    if (b) { tot1 = total; epos1 = pos; skip1 = skip_b; }
                    else { tot0 = total; epos0 = pos; skip0 = skip_b; }
                    if (skip_b) {
                        // empty tile: nothing to write, never waits; its count (0) is already out --
                        // upgrade it to a prefix if the predecessor's happens to be known
                        if (lane == 0) {
                            const unsigned long long w = ld_state(a.tile_state + pos - 1);
                            if ((w >> 34) == (tag >> 34) && ((w >> 32) & 3ull) == 2) st_state(a.tile_state + pos, w);
                        }
                    }
                    agg_it++;
                }
                // ---- (3) resumable decoupled look-back, then (once the points are staged) streaming
                //      of the oldest pending tile ----
                if (epi_it < agg_it) {
                    const int b = epi_it & 1;
                    const uint32_t tot_b = b ? tot1 : tot0;
                    const int epos_b = b ? epos1 : epos0;
                    const bool skip_b = b ? skip1 : skip0;
                    if (skip_b) {
                        if (__any_sync(0xffffffffu, mbar_try(bar_staged + 8 * b, (epi_it >> 1) & 1))) {
                            if (lane == 0) mbar_arrive(bar_cxfree + 8 * b);
                            epi_it++;
                            progressed = true;
                        }
                    } else {
                        if (!resolving) { resolving = true; published = false; excl = 0; look = epos_b - 1; }
                        bool resolved = published || epos_b == 0;
                        if (!resolved) {
                            // Walk back window after window while the words are there.  The distance
                            // to the nearest known prefix is (count->prefix latency) x (tile rate of
                            // the grid), so a slow walk feeds itself: one window per event-loop pass
                            // settled at ~30k cycles and ~600 tiles; a back-to-back walk at ~2k.
#pragma unroll 1
                            for (int hop = 0; hop < 24; hop++) {
                                const int idx = look - lane;
                                unsigned long long w = tag | (2ull << 32);   // virtual tile < 0: prefix 0
                                if (idx >= 0) w = ld_state(a.tile_state + idx);
                                const bool ready = (w >> 34) == (tag >> 34) && ((w >> 32) & 3ull) != 0;
                                const bool is_prefix = ready && ((w >> 32) & 3ull) == 2;
                                const unsigned rm = __ballot_sync(0xffffffffu, ready);
                                const unsigned pm = __ballot_sync(0xffffffffu, is_prefix);
                                // needed lanes: from the nearest tile up to the first known prefix
                                const int stop = pm ? __ffs(pm) - 1 : 31;
                                const unsigned need = stop == 31 ? 0xffffffffu : ((2u << stop) - 1u);
                                if ((rm & need) != need) break;            // a needed count is not out yet
                                progressed = true;
                                uint32_t v = lane <= stop ? (uint32_t)w : 0;
#pragma unroll
                                for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                                excl += v;
                                if (pm) { resolved = true; break; }
                                look -= 32;
                            }
                        }
                        if (resolved && !published) {
                            // the inclusive prefix goes out now, before this tile's points exist
                            published = true;
                            progressed = true;
                            if (lane == 0) {
                                st_state(a.tile_state + epos_b, tag | (2ull << 32) | (excl + tot_b));
                                if (epos_b == n_work - 1) *a.d_count = excl + tot_b;
                                trace(a.trace, epi_it, 6);
                            }
                        }
                        resolved = published && __any_sync(0xffffffffu, mbar_try(bar_staged + 8 * b, (epi_it >> 1) & 1));
                        if (resolved) {
                            progressed = true;
                            const uint32_t total = tot_b;
                            const int pos = epos_b;
                            if (total) {
                                // stream the tile's compacted points as one contiguous block
                                const float* cx = cxb + b * 3 * T;
                                float* dstp = a.pts + 3 * (size_t)excl;
                                const int n = 3 * (int)total;
                                const int head = min(n, (int)((4 - (((uintptr_t)dstp >> 2) & 3)) & 3));
                                if (lane < head) dstp[lane] = cx[lane];
                                const int nvec = (n - head) >> 2;
                                for (int v = lane; v < nvec; v += 32) {
                                    const int i = head + 4 * v;
                                    *reinterpret_cast<float4*>(dstp + i) = make_float4(cx[i], cx[i + 1], cx[i + 2], cx[i + 3]);
                                }
                                const int tail0 = head + 4 * nvec;
                                if (lane < n - tail0) dstp[tail0 + lane] = cx[tail0 + lane];
                                if (a.pix || a.rgb) {   // optional extras from the per-thread valid bits
                                    const int p0 = a.tile_list[pos] * T;
                                    uint32_t run = excl;
                                    for (int k = 0; k < CW; k++) {
                                        const int th = k * 32 + lane;
                                        const uint32_t f = vfl[b * (T / 4) + th];
                                        const uint32_t c = __popc(f);
                                        uint32_t incl = c;
#pragma unroll
                                        for (int o = 1; o < 32; o <<= 1) {
                                            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                                            if (lane >= o) incl += t;
                                        }
                                        uint32_t dp = run + incl - c;
                                        run += __shfl_sync(0xffffffffu, incl, 31);
                                        for (int j = 0; j < 4; j++)
                                            if ((f >> j) & 1u) {
                                                const size_t gp = (size_t)p0 + 4 * th + j;
                                                if (a.pix) a.pix[dp] = (uint32_t)((size_t)a.row0 * W + gp);
                                                if (a.rgb) {
                                                    a.rgb[3 * (size_t)dp + 0] = a.texture[3 * gp + 2];
                                                    a.rgb[3 * (size_t)dp + 1] = a.texture[3 * gp + 1];
                                                    a.rgb[3 * (size_t)dp + 2] = a.texture[3 * gp + 0];
                                                }
                                                dp++;
                                            }
                                    }
                                }
                            }
                            __syncwarp();
                            if (lane == 0) {
                                trace(a.trace, epi_it, 7);
                                mbar_arrive(bar_cxfree + 8 * b);
                            }
                            epi_it++;
                            resolving = false;
                        }
                    }
                }
            }
            if (!progressed) __nanosleep(S3D_IO_IDLE_NS);
        }
        return;
    }

    // ================================ CONSUMERS ================================
    for (int it = 0;; it++) {
        if (!mbar_try(bar_full, it & 1))
            while (!mbar_try(bar_full, it & 1)) __nanosleep(64);
        if (tid == 0) trace(a.trace, it, 2);
        const int pos = ctl[0];
        if (pos < 0) break;
        const int p0 = a.tile_list[pos] * T, wt = min(T, plane - p0);
        const int lp0 = 4 * tid;
        const bool active = lp0 < wt;
        const int row = (p0 + lp0) / W;
        const int xt = (p0 + lp0) - row * W;
        const int y = a.row0 + row;
        const uint32_t* sw = reinterpret_cast<const uint32_t*>(slot);

        // ---------------- integer phase: mask, fringe terms, Gray bits ----------------
        uint32_t mbits = 0, mbits_h = 0;      // mask of the vertical direction (of both without MOD) / of the horizontal one
        Terms Tv, Th;
        uint32_t gvA = 0, gvB = 0, ghA = 0, ghB = 0;
        if (active) {
            const bool window_ok = y >= 2 && y + 1 < a.H_total && xt >= 4 && xt + 7 < W;
            // the mask recurrence's closed form on one ROI window -> the thread's 4 mask bits
            auto mask_of = [&](const uint8_t* win) -> uint32_t {
                if (window_ok) {
                    uint32_t any_zero = 0;
#pragma unroll
                    for (int r = 0; r < 4; r++)
#pragma unroll
                        for (int c = 0; c < 3; c++) {
                            const uint32_t v = *reinterpret_cast<const uint32_t*>(win + r * G.roi_row + (lp0 + ROI_HALO - 4) + 4 * c);
                            any_zero |= (v - 0x01010101u) & ~v & 0x80808080u;
                        }
                    if (any_zero == 0) return 0xfu;
                }
                uint32_t mb = 0;
                const uint32_t centre = *reinterpret_cast<const uint32_t*>(win + 2 * G.roi_row + lp0 + ROI_HALO);
                if (centre != 0) {
#pragma unroll 1
                    for (int j = 0; j < 4; j++) {
                        const int x = xt + j;
                        auto inv = [&](int gx, int gy) {
                            return win[(gy - y + 2) * G.roi_row + (lp0 + j + (gx - x) + ROI_HALO)] == 0;
                        };
                        bool v = !inv(x, y);
                        const bool border = x == 0 || y == 0 || x == W - 1 || y == a.H_total - 1;
                        if (v && !border) v = !mask_trigger(x, y, W, a.H_total, inv);
                        mb |= (v ? 1u : 0u) << j;
                    }
                }
                return mb;
            };
            mbits = mask_of(sroi);
            mbits_h = NROI == 2 ? mask_of(sroi2) : mbits;
            if (mbits | mbits_h) {
                fringe_terms<N>(sw, 0, WPF, tid, Tv);
                gray_bits(sw, N, N + M_v, M_v, WPF, tid, gvA, gvB);
                if (DIRS == 2) {
                    const int fh = N + 2 * M_v;
                    fringe_terms<N>(sw, fh, WPF, tid, Th);
                    gray_bits(sw, fh + N, fh + N + M_h, M_h, WPF, tid, ghA, ghB);
                }
            }
        }
        // this warp is done with the slot: the IO warp may refill it once every warp has arrived
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_free);
        if (tid == 0) trace(a.trace, it, 3);

        // ---------------- FP64 phase (registers only) ----------------
        uint32_t vbits = 0;
        int4 cp01 = make_int4(0, 0, 0, 0), cp23 = cp01;   // the 4 pixels' correspondences, for the triangulation below
        // a warp whose 128 pixels hold no pixel of the mask writes the constant outputs and leaves its issue slots
        // to the other warps of the SM (about one warp in ten inside a tile that does hold ROI pixels)
        const bool warp_has_px = __any_sync(0xffffffffu, (mbits | mbits_h) != 0);
        if (active && !warp_has_px) {
            const size_t g = (size_t)p0 + lp0;
            *reinterpret_cast<float4*>(a.unw_v + g) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<uint2*>(a.code_v + g) = make_uint2(~0u, ~0u);
            *reinterpret_cast<uint32_t*>(a.valid + g) = 0u;
            if (DIRS == 2) {
                *reinterpret_cast<float4*>(a.unw_h + g) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<uint2*>(a.code_h + g) = make_uint2(~0u, ~0u);
                reinterpret_cast<int4*>(a.cpmap + g)[0] = make_int4(0, 0, 0, 0);
                reinterpret_cast<int4*>(a.cpmap + g)[1] = make_int4(0, 0, 0, 0);
            }
        }
        if (active && warp_has_px) {
            // Two passes of 2 pixels: inside a pass everything is straight-line (2 pixels x 2
            // directions interleave in the FP64 pipe); the pass loop is rolled to keep the
            // consumer loop inside the instruction cache.
            const size_t g = (size_t)p0 + lp0;
#pragma unroll 1
            for (int h = 0; h < 2; h++) {
                float r_unwv[2], r_unwh[2];
                int r_cv[2], r_ch[2];
                int2 r_cp[2];
                uint32_t vb = 0;
                // the pair's term registers, Gray accumulators and mask bits, selected once by h
                const TermsPair Pv = terms_pair(Tv, h), Ph = terms_pair(Th, h);
                const uint32_t gvA_h = gvA >> (16 * h), gvB_h = gvB >> (16 * h), ghA_h = ghA >> (16 * h), ghB_h = ghB >> (16 * h);
                const uint32_t mb_v = mbits >> (2 * h), mb_h = mbits_h >> (2 * h);
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int x = xt + 2 * h + u;
                    const bool mv = (mb_v >> u) & 1u, mh = (mb_h >> u) & 1u;
                    const bool m = mv && mh;                                             // merge_valid_maps, 5/compute_correspondance.cpp:60-77
                    const int cv = code_of_pair(gvA_h, gvB_h, u, M_v);
                    const float wv = add_pi(phase_of_pair<N>(Pv, u, tab));               // 4/phase_unwrap.cpp:290
                    // two directions: the unwrap term comes from the per-order table (one cached load instead of 4 FP64
                    // instructions); one direction has too few independent chains per pass to cover the load (1080p
                    // 3-step measured 4 % slower with it) and divides
                    float unwv = (x == 0 || x == W - 1) ? 0.0f
                                 : DIRS == 2 ? unwrap_abs_k(wv, __ldg(a.code_term + cv)) : unwrap_abs(wv, cv, true);  // :285, :291
                    unwv = mv ? unwv : 0.0f;
                    bool v = mv;
                    r_cv[u] = mv ? cv : -1;
                    if (DIRS == 2) {
                        const int ch = code_of_pair(ghA_h, ghB_h, u, M_h);
                        const float wh = add_pi(phase_of_pair<N>(Ph, u, tab));
                        float unwh = (y == 0 || y == a.H_total - 1) ? 0.0f : unwrap_abs_k(wh, __ldg(a.code_term + ch));  // :304, :309
                        unwh = mh ? unwh : 0.0f;
                        // 5/compute_correspondance.cpp:648-675.  Both phases are finite here (see
                        // correspond32_finite), so lrint's FE_INVALID rejection never fires.
                        const int px = correspond32_finite(unwv, a.fw_v_d);
                        const int py = correspond32_finite(unwh, a.fw_h_d);
                        r_cp[u].x = m ? px : 0;
                        r_cp[u].y = m ? py : 0;
                        // 0 <= p <= P-1 as one unsigned compare (saturated values fall outside as well)
                        v = m && (unsigned)px <= (unsigned)(a.PW - 1) && (unsigned)py <= (unsigned)(a.PH - 1);
                        r_unwh[u] = unwh;
                        r_ch[u] = mh ? ch : -1;
                    }
                    r_unwv[u] = unwv;
                    vb |= (v ? 1u : 0u) << u;
                }
                // plane outputs of the 2 pixels: one (vector) store per plane
                const size_t gh = g + 2 * h;
                *reinterpret_cast<float2*>(a.unw_v + gh) = make_float2(r_unwv[0], r_unwv[1]);
                *reinterpret_cast<uint32_t*>(a.code_v + gh) = (uint32_t)(r_cv[0] & 0xffff) | ((uint32_t)r_cv[1] << 16);
                *reinterpret_cast<uint16_t*>(a.valid + gh) = (uint16_t)((vb & 1u) | ((vb & 2u) << 7));
                if (DIRS == 2) {
                    *reinterpret_cast<float2*>(a.unw_h + gh) = make_float2(r_unwh[0], r_unwh[1]);
                    *reinterpret_cast<uint32_t*>(a.code_h + gh) = (uint32_t)(r_ch[0] & 0xffff) | ((uint32_t)r_ch[1] << 16);
                    const int4 c4 = make_int4(r_cp[0].x, r_cp[0].y, r_cp[1].x, r_cp[1].y);
                    *reinterpret_cast<int4*>(a.cpmap + gh) = c4;
                    if (h == 0) cp01 = c4; else cp23 = c4;
                    // the undistortion tables are gathered once per surviving pixel a few thousand
                    // cycles from now: pull the lines into L2 meanwhile (DRAM latency -> L2 latency)
                    if (vb) {
                        if (has_cam_lut) prefetch_l2(a.cam_lut + gh);
                        if (has_proj_lut) {
                            if (vb & 1u) prefetch_l2(a.proj_lut + (size_t)c4.y * a.PW + c4.x);
                            if (vb & 2u) prefetch_l2(a.proj_lut + (size_t)c4.w * a.PW + c4.z);
                        }
                    }
                }
                vbits |= vb << (2 * h);
            }
        }
        if (DIRS == 2) {
            // ---- block scan of the valid counts first: every pixel then knows its raster rank in
            //      the tile, and the triangulation writes its point straight to that rank ----
            const int b = it & 1;
            const uint32_t cnt = __popc(vbits);
            uint32_t incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            // buffer b (points, counts, valid bits) must have been drained by the IO warp (tile it-2)
            if (!mbar_try(bar_cxfree + 8 * b, ((it >> 1) & 1) ^ 1))
                while (!mbar_try(bar_cxfree + 8 * b, ((it >> 1) & 1) ^ 1)) __nanosleep(64);
            if (lane == 31) cnts[b * 16 + warp] = incl;
            // the camera-table entries of the thread's surviving pixels (64 contiguous bytes): into L1 while the warp
            // waits at the barrier -- the triangulation's first use of them was 5 % of all stall samples (-1 % time)
            if (has_cam_lut && vbits) prefetch_l1(a.cam_lut + (size_t)p0 + lp0);
            cons_sync<NCONS>();
            uint32_t rank = incl - cnt, total = 0;
#pragma unroll
            for (int w2 = 0; w2 < CW; w2++) {
                const uint32_t c = cnts[b * 16 + w2];
                rank += w2 < warp ? c : 0u;
                total += c;
            }
            if (tid == 0) {
                // The tile's count goes out NOW, from here, before the triangulation: every later
                // tile's look-back needs it, and the IO warp may be busy issuing loads or streaming.
                const unsigned long long tag = (unsigned long long)(a.epoch & 0x3fffffffu) << 34;
                st_state(a.tile_state + pos, tag | ((pos ? 1ull : 2ull) << 32) | total);
                mbar_arrive(bar_counted + 8 * b);
            }
            float* cx = cxb + b * 3 * T;
            vfl[b * (T / 4) + tid] = (uint8_t)vbits;
            // triangulation of the surviving pixels (7/triangulation.cpp:1230-1247)
#pragma unroll 1
            for (int j = 0; j < 4; j++) {
                if (!((vbits >> j) & 1u)) continue;
                const int x = xt + j;
                const int cpx = j == 0 ? cp01.x : j == 1 ? cp01.z : j == 2 ? cp23.x : cp23.z;
                const int cpy = j == 0 ? cp01.y : j == 1 ? cp01.w : j == 2 ? cp23.y : cp23.w;
                double uc, vc, up, vp, Xd[3];
                if (has_cam_lut) {
                    const double2 t = a.cam_lut[(size_t)p0 + lp0 + j];
                    uc = t.x; vc = t.y;
                } else if (EXACT) {
                    undistorted_pixel_std(cal.Kc, cal.ifx_c, cal.ify_c, (double)x, (double)y, &uc, &vc);
                } else {
                    // fast mode: without distortion the normalise / re-project round trip f * ((u - c) / f) + c is the
                    // identity up to two roundings (~1e-16 relative, against the mode's 1e-6 bound on the points)
                    uc = (double)x; vc = (double)y;
                }
                if (has_proj_lut) {
                    const double2 t = a.proj_lut[(size_t)cpy * a.PW + cpx];
                    up = t.x; vp = t.y;
                } else if (EXACT) {
                    undistorted_pixel_std(cal.Kp, cal.ifx_p, cal.ify_p, (double)cpx, (double)cpy, &up, &vp);
                } else {
                    up = (double)cpx; vp = (double)cpy;
                }
                if (EXACT) triangulate_point(cal.Ac, cal.Ap, uc, vc, up, vp, Xd);
                else triangulate_point_camframe(cal, uc, vc, up, vp, Xd);   // cam_std (launch_fused7)
                float px = __double2float_rn(Xd[0]), py = __double2float_rn(Xd[1]), pz = __double2float_rn(Xd[2]);   // 8/save_point_cloud.cpp:94-96
                // optional: register_point_clouds' turntable transform on the float point (9/register_point_clouds.cpp:117-137)
                if (REG) s3a::register_point(a.reg_R, a.reg_t[0], a.reg_t[1], a.reg_t[2], px, py, pz);
                cx[3 * rank + 0] = px;
                cx[3 * rank + 1] = py;
                cx[3 * rank + 2] = pz;
                rank++;
            }
            if (tid == 0) trace(a.trace, it, 4);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_staged + 8 * b);
        }
    }
}

// 2-D view of the capture stack for the tile loads: inner dimension = one frame as 64-bit words,
// outer = the frames; box = [T/8 words] x [NF frames], landing in shared memory as [NF][T] bytes.
static cudaError_t stack_tensor_map(CUtensorMap* map, const uint8_t* stack, size_t plane, int NF, int T)
{
    typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    // looked up once per process (a function-local static is initialised once even when several host threads launch)
    static const encode_fn encode = []() -> encode_fn {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        return (encode_fn)fn;
    }();
    if (!encode) return cudaErrorNotSupported;
    const cuuint64_t gdim[2] = {(cuuint64_t)(plane / 8), (cuuint64_t)NF};
    const cuuint64_t gstride[1] = {(cuuint64_t)plane};
    const cuuint32_t box[2] = {(cuuint32_t)(T / 8), (cuuint32_t)NF};
    const cuuint32_t estr[2] = {1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<uint8_t*>(stack), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS
               ? cudaSuccess
               : cudaErrorInvalidValue;
}

template <int N, int DIRS, int CW, int MINB, bool EXACT, bool MOD = false, bool REG = false, int MV = 0, int MH = 0, int LUTS = -1>
static cudaError_t launch7_t(const FusedArgs& a, const DeviceCalib& cal, int sm_count, const Plan7& p, cudaStream_t st)
{
    auto kern = k_fused7<N, DIRS, CW, MINB, EXACT, MOD, REG, MV, MH, LUTS>;
    // per instantiation, once per process and shared-memory size: attributes and occupancy (a scan of a small frame
    // is a few tens of microseconds: the host side of a launch must not cost as much)
    static size_t smem_cached = 0;
    static int per_sm_cached = 0;
    cudaError_t e;
    if (smem_cached != p.smem) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
        if (e != cudaSuccess) return e;
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        int per_sm = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, (CW + 1) * 32, p.smem);
        if (e != cudaSuccess) return e;
        if (per_sm < 1) return cudaErrorLaunchOutOfResources;
        if (getenv("SCAN3D_DEBUG")) {
            cudaFuncAttributes fa;
            cudaFuncGetAttributes(&fa, kern);
            fprintf(stderr, "k_fused7<%d,%d,%d,%d,%d,%d>: occupancy %d CTAs/SM, %d regs, %zu B dyn smem, %zu B static, local %zu B\n", N, DIRS, CW, MINB,
                    (int)EXACT, (int)MOD, per_sm, fa.numRegs, p.smem, fa.sharedSizeBytes, fa.localSizeBytes);
        }
        per_sm_cached = per_sm > MINB ? MINB : per_sm;
        smem_cached = p.smem;
    }
    // a.ctas_per_sm > 0 (scan3d_set_cta_limit): this context's launches take only that many of the SM's CTA slots, so
    // that the persistent kernels of several contexts (streams) are resident side by side and one scan's pipeline
    // fill and drain overlap the other scans' steady state
    const int per_sm = a.ctas_per_sm > 0 && a.ctas_per_sm < per_sm_cached ? a.ctas_per_sm : per_sm_cached;
    const int grid = a.n_tiles < sm_count * per_sm ? a.n_tiles : sm_count * per_sm;   // all CTAs resident
    // the tensor map depends on the stack's address and the tile size only: the context keeps the last few
    TensorMapCache& cache = *a.tmap_cache;
    const CUtensorMap* map = nullptr;
    for (int i = 0; i < TensorMapCache::SLOTS; i++)
        if (cache.stack[i] == a.stack && cache.box[i] == 128 * CW) map = &cache.map[i];
    if (!map) {
        const int slot = cache.next++ % TensorMapCache::SLOTS;
        cache.stack[slot] = nullptr;
        const int NF = DIRS == 2 ? 2 * N + 2 * (a.M_v + a.M_h) : N + 2 * a.M_v;
        e = stack_tensor_map(&cache.map[slot], a.stack, (size_t)a.W * a.H, NF, 128 * CW);
        if (e != cudaSuccess) return e;
        cache.stack[slot] = a.stack;
        cache.box[slot] = 128 * CW;
        map = &cache.map[slot];
    }
    e = launch_worklist(a, 128 * CW, DIRS, st);
    if (e != cudaSuccess) return e;
    kern<<<grid, (CW + 1) * 32, p.smem, st>>>(a, cal, *map);
    return cudaGetLastError();
}

// One instantiation per (shape, N, DIRS, variant) that plan7 and fused7_folds_registration can select: one direction
// runs at (7, 3) only (at most 38 frames); (9, 2) serves two directions without the folded transform; (7, 2) without
// the modulation mask is reached by 8-step scans only (72-76 frames; every other N stays below 72).
template <int N, int DIRS>
static cudaError_t launch7_nd(const FusedArgs& a, const DeviceCalib& cal, int sm_count, const Plan7& p, bool exact,
                              cudaStream_t st)
{
    if (p.cw == 7 && p.minb == 3) {
        // The named configurations in the default shape get their Gray depths as compile-time constants:
        // C3 / C4 / C5 (8-step, 10 + 10 bits), C1 (3-step, 6 + 5 bits), C2 (3-step, 8 bits, one direction).
        // ... and with them the reference's calibration class (distorted camera, distortion-free projector: LUTS = 1)
        const bool ref_class = a.cam_lut != nullptr && a.proj_lut == nullptr;
        if (N == 8 && DIRS == 2 && a.M_v == 10 && a.M_h == 10) {
#define S3D_M10(EX, RG)                                                                                               \
    (ref_class ? launch7_t<8, 2, 7, 3, EX, false, RG, 10, 10, 1>(a, cal, sm_count, p, st)                              \
               : launch7_t<8, 2, 7, 3, EX, false, RG, 10, 10>(a, cal, sm_count, p, st))
            if (a.reg_on) return exact ? S3D_M10(true, true) : S3D_M10(false, true);
            return exact ? S3D_M10(true, false) : S3D_M10(false, false);
#undef S3D_M10
        }
        if (N == 3 && DIRS == 2 && a.M_v == 6 && a.M_h == 5 && !a.reg_on) {
            if (ref_class) return exact ? launch7_t<3, 2, 7, 3, true, false, false, 6, 5, 1>(a, cal, sm_count, p, st)
                                        : launch7_t<3, 2, 7, 3, false, false, false, 6, 5, 1>(a, cal, sm_count, p, st);
            return exact ? launch7_t<3, 2, 7, 3, true, false, false, 6, 5>(a, cal, sm_count, p, st)
                         : launch7_t<3, 2, 7, 3, false, false, false, 6, 5>(a, cal, sm_count, p, st);
        }
        if (N == 3 && DIRS == 1 && a.M_v == 8) return launch7_t<3, 1, 7, 3, true, false, false, 8, 0>(a, cal, sm_count, p, st);
        if (DIRS == 2 && a.reg_on) return exact ? launch7_t<N, 2, 7, 3, true, false, true>(a, cal, sm_count, p, st)
                                                : launch7_t<N, 2, 7, 3, false, false, true>(a, cal, sm_count, p, st);
        if (exact || DIRS == 1) return launch7_t<N, DIRS, 7, 3, true>(a, cal, sm_count, p, st);
        return launch7_t<N, DIRS, 7, 3, (DIRS == 1)>(a, cal, sm_count, p, st);
    }
    if constexpr (DIRS == 2) {
        if (p.cw == 9 && p.minb == 2)
            return exact ? launch7_t<N, 2, 9, 2, true>(a, cal, sm_count, p, st) : launch7_t<N, 2, 9, 2, false>(a, cal, sm_count, p, st);
        if constexpr (N == 8) {
            if (p.cw == 7 && p.minb == 2) {
                if (a.reg_on) return exact ? launch7_t<8, 2, 7, 2, true, false, true>(a, cal, sm_count, p, st)
                                           : launch7_t<8, 2, 7, 2, false, false, true>(a, cal, sm_count, p, st);
                return exact ? launch7_t<8, 2, 7, 2, true>(a, cal, sm_count, p, st) : launch7_t<8, 2, 7, 2, false>(a, cal, sm_count, p, st);
            }
        }
    }
    return cudaErrorInvalidValue;
}

// the modulation-criterion variant (3-step only): (7, 3), and (7, 2) for two directions from 54 frames on
template <int DIRS>
static cudaError_t launch7_mod(const FusedArgs& a, const DeviceCalib& cal, int sm_count, const Plan7& p, bool exact, cudaStream_t st)
{
    if (p.cw == 7 && p.minb == 3) {
        if (exact || DIRS == 1) return launch7_t<3, DIRS, 7, 3, true, true>(a, cal, sm_count, p, st);
        return launch7_t<3, DIRS, 7, 3, (DIRS == 1), true>(a, cal, sm_count, p, st);
    }
    if constexpr (DIRS == 2) {
        if (p.cw == 7 && p.minb == 2)
            return exact ? launch7_t<3, 2, 7, 2, true, true>(a, cal, sm_count, p, st) : launch7_t<3, 2, 7, 2, false, true>(a, cal, sm_count, p, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_fused7(const scan3d_config& c, const FusedArgs& a_in, const DeviceCalib& cal, int sm_count,
                          cudaStream_t st)
{
    Plan7 p;
    if (!plan7(c, &p)) return cudaErrorInvalidValue;
    if (((uintptr_t)a_in.stack & 15) || ((uintptr_t)a_in.roi & 15)) return cudaErrorMisalignedAddress;
    FusedArgs a = a_in;
    const int T = 128 * p.cw;
    a.n_tiles = (int)(((size_t)c.W * c.H + T - 1) / T);
    // the fast solve runs in the camera's frame and needs the standard camera matrix; otherwise the exact one runs
    const bool exact = !(c.flags & SCAN3D_FLAG_FAST_TRIANGULATION) || !cal.cam_std;
    if (mod7(c)) {
        if (!a.roi2 || !a.roi_list) return cudaErrorInvalidValue;
        return c.dirs == 2 ? launch7_mod<2>(a, cal, sm_count, p, exact, st) : launch7_mod<1>(a, cal, sm_count, p, exact, st);
    }
#define S3D_F7(NN) (c.dirs == 2 ? launch7_nd<NN, 2>(a, cal, sm_count, p, exact, st) : launch7_nd<NN, 1>(a, cal, sm_count, p, exact, st))
    switch (c.N) {
        case 3: return S3D_F7(3);
        case 4: return S3D_F7(4);
        case 5: return S3D_F7(5);
        case 8: return S3D_F7(8);
    }
#undef S3D_F7
    return cudaErrorInvalidValue;
}

}  // namespace s3d
