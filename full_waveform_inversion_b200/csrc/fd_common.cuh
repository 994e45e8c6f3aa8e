// Track B shared device helpers: stencil coefficients, TMA / mbarrier PTX wrappers (sm_100a).
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace fwi {

// 8th-order central second-derivative coefficients (oracle/fd_oracle.py COEF)
__device__ constexpr float kC0 = -205.0f / 72.0f;
__device__ constexpr float kC1 = 8.0f / 5.0f;
__device__ constexpr float kC2 = -1.0f / 5.0f;
__device__ constexpr float kC3 = 8.0f / 315.0f;
__device__ constexpr float kC4 = -1.0f / 560.0f;
constexpr int kHalo = 4;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
// TMA tiled loads (cp.async.bulk.tensor): out-of-bounds elements are zero-filled by the hardware, which is
// exactly the Dirichlet halo of the oracle (values outside the grid are 0).
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(x), "r"(y)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, int x, int y, int z, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}

// programmatic dependent launch: wait for the grid this launch was chained to
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
// streaming (evict-first) accesses for the wavefield snapshots: written once / read once, must not evict the
// L2-resident wavefields
__device__ __forceinline__ void st4_stream(float* p, const float4& v) { __stcs(reinterpret_cast<float4*>(p), v); }
__device__ __forceinline__ float4 ld4_stream(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }

// Free surface at z = 0 (spec B6): the 4 shared-memory rows above the surface become the odd mirror of the rows below it,
// u[-k] = -u[k] for k = 1..4, over `width` floats of rows `stride` apart; row `row0` holds z = 0.  The whole CTA takes part;
// the caller synchronises before the rows are read.
__device__ __forceinline__ void mirror_rows(float* s, int stride, int row0, int width) {
    for (int i = threadIdx.x; i < kHalo * width; i += blockDim.x) {
        const int k = 1 + i / width, c = i - (k - 1) * width;
        s[(row0 - k) * stride + c] = -s[(row0 + k) * stride + c];
    }
}

// sparse point lists (sources / receivers) binned by the CTA tile that owns the point
struct PointListDev {
    const int* tile_ptr;   // [ntiles + 1]
    const int* off;        // linear offset into the pitched field
    const int* id;         // column in the per-step value row
};

}  // namespace fwi
