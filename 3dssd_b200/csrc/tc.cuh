// tc.cuh -- the tcgen05 / TMEM / TMA wrappers and the split-bf16 precision scheme of the tensor-core kernels
// (linear_tc_kernel in mlp_tc.cu, sa_fused_kernel in sa_fused.cu).
//
// Precision (DESIGN.md "Grouped MLP"): every fp32 operand travels as two bf16 terms, x = hi + lo with hi = bf16(x) and
// lo = bf16(x - hi) (16 mantissa bits), and a product is evaluated as three bf16 MMAs accumulating in fp32 in TMEM:
//     x.W ~= x_hi.W_hi + x_lo.W_hi + x_hi.W_lo          (error ~2^-16)
// split_pair / split8_store make the terms, umma_bf16x3 issues the product.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"

namespace ssd3d {

// ---- fences ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy stores to shared memory -> visible to the tensor core and TMA (async proxy)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- UMMA descriptors and issue ---------------------------------------------------------------------------------------
// K-major operand tile in shared memory; row_bytes = bytes per row = swizzle span (128 -> SWIZZLE_128B, 64 -> _64B,
// 32 -> _32B), 8-row groups are 8 * row_bytes apart (SBO), descriptor version 1.  Advancing the address field by 2
// moves 16 bf16 (one k-step) along K.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, int row_bytes)
{
    const uint64_t layout = row_bytes == 128 ? 2ull : (row_bytes == 64 ? 4ull : 6ull);
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)((8 * row_bytes) >> 4) << 32) |
           (1ull << 46) | (layout << 61);
}
// instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t umma_idesc_bf16(int n)
{
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}
// One k-step of the split product (see the top of this file): d = [d +] a.b, acc == 0 overwrites d.  One thread issues.
__device__ __forceinline__ void umma_bf16x3(uint32_t d_tmem, uint64_t a_hi, uint64_t a_lo, uint64_t b_hi, uint64_t b_lo,
                                            uint32_t idesc, uint32_t acc)
{
    umma_bf16(d_tmem, a_hi, b_hi, idesc, acc);
    umma_bf16(d_tmem, a_lo, b_hi, idesc, 1u);
    umma_bf16(d_tmem, a_hi, b_lo, idesc, 1u);
}
// arrives on the mbarrier once every MMA this thread issued before has completed
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- TMEM ---------------------------------------------------------------------------------------------------------------
// Whole warp: allocates ncols (a power of two >= 32) columns, writes their base address to *base (shared memory), and
// gives up the right to allocate more so that other CTAs on the SM can.
__device__ __forceinline__ void tmem_alloc(uint32_t *base, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(base)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}
// 32 consecutive fp32 columns of this warp's 32 TMEM lanes (one row per thread)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- TMA ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int x, int y, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, uint32_t src, int x, int y)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- operand construction -------------------------------------------------------------------------------------------------
// x = hi + lo for two values, packed {x1 : x0} like two adjacent bf16
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t &hw, uint32_t &lw)
{
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hw) : "f"(x1), "f"(x0));
    const float h0 = __uint_as_float(hw << 16), h1 = __uint_as_float(hw & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lw) : "f"(x1 - h1), "f"(x0 - h0));
}
// 8 consecutive columns f[0..7] -> one 16-byte chunk of hi terms at `hi`, one of lo terms at `lo`
__device__ __forceinline__ void split8_store(const float *f, void *hi, void *lo)
{
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int t = 0; t < 4; t++) split_pair(f[2 * t], f[2 * t + 1], hw[t], lw[t]);
    *reinterpret_cast<uint4 *>(hi) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    *reinterpret_cast<uint4 *>(lo) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
}
// The operand of the conv that follows a HOISTED first conv, 8 columns at a time: f = relu(z + dx*Wx'[0] + dy*Wx'[1] +
// dz*Wx'[2]), f holding the z row on entry, wx pointing at the chunk's columns of row 0 of Wx' = [3][ld] (16-byte aligned,
// zero beyond the conv's width, so padded columns come out +0).  Every route that builds this operand (the gather of
// sa_fused_kernel, the producer warps of linear_tc_kernel, hoist_expand_split_kernel) calls this function: the FMA order
// is part of the result, and the routes agree bit for bit.
__device__ __forceinline__ void hoist_relu8(float *f, float dx, float dy, float dz, const float *wx, int ld)
{
#pragma unroll
    for (int e4 = 0; e4 < 8; e4 += 4) {
        const float4 w0 = *reinterpret_cast<const float4 *>(wx + e4);
        const float4 w1 = *reinterpret_cast<const float4 *>(wx + ld + e4);
        const float4 w2 = *reinterpret_cast<const float4 *>(wx + 2 * ld + e4);
        f[e4 + 0] = fmaxf(fmaf(dz, w2.x, fmaf(dy, w1.x, fmaf(dx, w0.x, f[e4 + 0]))), 0.0f);
        f[e4 + 1] = fmaxf(fmaf(dz, w2.y, fmaf(dy, w1.y, fmaf(dx, w0.y, f[e4 + 1]))), 0.0f);
        f[e4 + 2] = fmaxf(fmaf(dz, w2.z, fmaf(dy, w1.z, fmaf(dx, w0.z, f[e4 + 2]))), 0.0f);
        f[e4 + 3] = fmaxf(fmaf(dz, w2.w, fmaf(dy, w1.w, fmaf(dx, w0.w, f[e4 + 3]))), 0.0f);
    }
}

}  // namespace ssd3d
