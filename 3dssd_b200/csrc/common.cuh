// common.cuh -- shared helpers for the sm_100a kernels of libssd3d.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ssd3d.h"

namespace ssd3d {

// ---- status / error string (thread-local, read back through ssd3d_last_error) -----------------
void set_error(const char *fmt, ...);
int cuda_status(cudaError_t e, const char *what);

#define SSD3D_REQUIRE(cond, ...)                                   \
    do {                                                           \
        if (!(cond)) {                                             \
            ::ssd3d::set_error(__VA_ARGS__);                       \
            return SSD3D_ERR_INVALID_ARGUMENT;                     \
        }                                                          \
    } while (0)

// cudaGetLastError (capture-safe) reports a failed launch once AND clears it, so later calls do not inherit it
#define SSD3D_LAUNCH_CHECK(what) return ::ssd3d::cuda_status(cudaGetLastError(), what)

constexpr int kNumSMs = 148;  // B200

static inline int ceil_div(long a, long b) { return (int)((a + b - 1) / b); }

// ---- PTX wrappers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_id_x()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same variable in CTA `rank`
__device__ __forceinline__ uint32_t mapa(uint32_t cta_addr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init_cluster()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        ::"r"(bar), "r"(parity) : "memory");
}
// named barrier `id` (1..15) over `nthreads` threads (a multiple of 32)
__device__ __forceinline__ void bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
// One lane of a converged warp (for single-thread instructions such as tcgen05.mma / commit issued from code the
// whole warp runs, so that their operands stay in uniform registers).
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// CTA-scope acquire: enough for data that lands in THIS CTA's shared memory (TMA, st.async from peers); a
// cluster-scope acquire makes ptxas emit CCTL.IVALL (an L1 invalidate) on every wait -- 32% of the FPS round.
__device__ __forceinline__ void mbar_wait_cta(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        ::"r"(bar), "r"(parity) : "memory");
}
// 16-byte store into a peer CTA's shared memory that also completes 16 tx-bytes on the peer's mbarrier
__device__ __forceinline__ void st_async_v4(uint32_t remote_addr, uint32_t remote_bar, uint4 v)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(remote_addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(remote_bar) : "memory");
}
__device__ __forceinline__ void st_async_b64(uint32_t remote_addr, uint32_t remote_bar, uint64_t v)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                 ::"r"(remote_addr), "l"(v), "r"(remote_bar) : "memory");
}
__device__ __forceinline__ float ld_dsmem_f32(uint32_t cluster_addr)
{
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr) : "memory");
    return v;
}
// 1-D bulk copy global -> shared::cta, completion on an mbarrier of this CTA
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}


// Order-preserving float <-> uint map: unsigned comparisons (redux.min/max, sort keys) of ord(x) order the floats x,
// negative values included.
__device__ __forceinline__ uint32_t f2ord(float x)
{
    const uint32_t b = __float_as_uint(x);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

}  // namespace ssd3d
