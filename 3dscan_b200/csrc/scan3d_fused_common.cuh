// scan3d_fused_common.cuh -- device helpers shared by the fused kernels: PTX wrappers (mbarrier,
// TMA bulk copies, look-back words) and the pipeline timeline hooks.  The SWAR integer decode of 4
// pixels per 32-bit word lives in scan3d_fused_math.cuh.
#pragma once
#include "scan3d_internal.h"
#include "scan3d_fused_math.cuh"
#include "../common/scan3d_aux_math.h"

namespace s3d {

constexpr int ROI_HALO = 16;               // bytes of halo each side (16 B aligned bulk copies)
constexpr int SMEM_MAX = 227 * 1024;

// ---- PTX helpers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity)
{
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done != 0;
}
// (A non-blocking mbarrier.test_wait probe in the IO warp's event loop measured 4-10 % SLOWER than
// try_wait, whose hardware suspend keeps the polling warp out of the issue slots.)
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// one 2-D tiled tensor copy global -> shared through a CUtensorMap (coordinates in elements)
__device__ __forceinline__ void tensor_g2s_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(tmap), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
template <int NT>
__device__ __forceinline__ void cons_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory"); }

__device__ __forceinline__ unsigned long long ld_state(const unsigned long long* p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_state(unsigned long long* p, unsigned long long v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// optional per-CTA timeline (library built with SCAN3D_BUILD_TRACE=1, run with SCAN3D_TRACE=1):
// clock64 stamps of the pipeline events of the first TRACE_TILES tiles of every CTA;
// slot = (cta * TRACE_TILES + it) * 8 + event
#ifndef S3D_TRACE
#define S3D_TRACE 0
#endif
constexpr int TRACE_TILES = 64;
__device__ __forceinline__ void trace(unsigned long long* t, int it, int ev)
{
    if (S3D_TRACE && t && it < TRACE_TILES) t[((size_t)blockIdx.x * TRACE_TILES + it) * 8 + ev] = clock64();
}


// work-list kernels (scan3d_worklist.cu)
cudaError_t launch_worklist(const FusedArgs& a, int T, int dirs, cudaStream_t st);

}  // namespace s3d
