// pool.cuh -- the max-pool epilogue of the tensor-core kernels: "reduce and transpose" butterfly, then the stores.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace ssd3d {

// Each lane holds one ROW of a [32 rows x 32 columns] block in v[0..31].  Computes, for every run of GP consecutive
// lanes (rows), the column-wise maximum; on return lane L owns columns (L % GP) * (32/GP) + k, k < 32/GP, of its
// group's result in v[k].  31 shuffles for GP = 32 (instead of 32 full-warp reductions): every step halves the
// number of live values per lane while exchanging the other half with the xor-partner.
template <int GP>
__device__ __forceinline__ void warp_colmax_transpose(float (&v)[32], int lane)
{
#pragma unroll
    for (int o = GP / 2, cnt = 32; o >= 1; o >>= 1, cnt >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < cnt / 2; i++) {
            const float send = up ? v[i] : v[i + cnt / 2];
            const float keep = up ? v[i + cnt / 2] : v[i];
            v[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, o));
        }
    }
}

// The pooled outputs below are written through the output fields of the kernel's parameter block P: out_f32 / ld_f32
// and, when out_hi is set, the split copy out_hi / out_lo / ld_split.  The pointers arrive in a by-value struct, which
// carries no address space, so the stores are spelled st.global (a generic store would resolve it at run time).
__device__ __forceinline__ void st_global(float *p, float x) { asm volatile("st.global.f32 [%0], %1;" ::"l"(p), "f"(x) : "memory"); }
__device__ __forceinline__ void st_global(__nv_bfloat16 *p, __nv_bfloat16 x)
{
    asm volatile("st.global.b16 [%0], %1;" ::"l"(p), "h"(__bfloat16_as_ushort(x)) : "memory");
}

// Max-pool of one 32-column chunk of a 128-row tile over runs of POOL rows (tf.reduce_max(axis=2), layers_util.py:178),
// mask (:180) and store.  Warp q of the tile's four holds rows 32q..32q+31, one per lane, in v; groups of POOL <= 32 rows
// are lanes of one warp, groups of 64 / 128 rows span 2 / 4 warps and meet through xs[4][32] under the named barrier
// `bar` of those 128 threads.  Pooled row g = tile * 128 / POOL + ...; rows g * POOL >= p.rows are not stored.
// mask (may be null): mask[g] == 0 stores zeros.  col0: output column of v[0]; columns >= ncols are not stored.
// AFTER: v holds RAW accumulators and the folded affine + ReLU (sc / sh, indexed by output column) is applied to the
// pooled values only -- valid when the scale is >= 0: fma(x, s, t) is then monotone non-decreasing in x, so
// max_i relu(fma(x_i, s, t)) == relu(fma(max_i x_i, s, t)) exactly -- 1/POOL of the epilogue math.
template <int POOL, bool AFTER, class P>
__device__ __forceinline__ void pool_rows(const P &p, const int *mask, float (&v)[32], int lane, int q, int tile, int col0,
                                          int ncols, const float *sc, const float *sh, float *xs, int bar)
{
    constexpr int GP = POOL >= 32 ? 32 : POOL;           // lanes per group inside a warp
    constexpr int KEEP = 32 / GP;                        // columns a lane ends up owning
    constexpr int WPG = POOL > 32 ? POOL / 32 : 1;       // warps per group
    warp_colmax_transpose<GP>(v, lane);                  // lane owns columns (lane % GP) * KEEP + k in v[k]
    if (POOL > 32) {
        xs[q * 32 + lane] = v[0];
        bar_sync(bar, 128);
        if ((q % WPG) == 0) {
#pragma unroll
            for (int w = 1; w < WPG; w++) v[0] = fmaxf(v[0], xs[(q + w) * 32 + lane]);
        }
        bar_sync(bar, 128);                              // xs reusable by the next chunk
        if ((q % WPG) != 0) return;
    }
    const int gg = tile * (128 / POOL) + (q * 32 + lane) / POOL;
    if ((long)gg * POOL >= p.rows) return;
    const bool masked = mask && mask[gg] == 0;
#pragma unroll
    for (int k = 0; k < KEEP; k++) {
        const int col = col0 + (lane % GP) * KEEP + k;
        if (col >= ncols) continue;
        float mx = v[k];
        if (AFTER) mx = fmaxf(fmaf(mx, sc[col], sh[col]), 0.0f);
        mx = masked ? 0.0f : mx;
        if (p.out_f32) st_global(p.out_f32 + (size_t)gg * p.ld_f32 + col, mx);
        if (p.out_hi) {
            const __nv_bfloat16 hb = __float2bfloat16_rn(mx);
            st_global(p.out_hi + (size_t)gg * p.ld_split + col, hb);
            st_global(p.out_lo + (size_t)gg * p.ld_split + col, __float2bfloat16_rn(mx - __bfloat162float(hb)));
        }
    }
}
// pool_rows for a run-time POOL (8, 16, 32, 64 or 128)
template <bool AFTER, class P>
__device__ __forceinline__ void pool_rows(int pool, const P &p, const int *mask, float (&v)[32], int lane, int q, int tile,
                                          int col0, int ncols, const float *sc, const float *sh, float *xs, int bar)
{
    switch (pool) {
        case 8: pool_rows<8, AFTER>(p, mask, v, lane, q, tile, col0, ncols, sc, sh, xs, bar); break;
        case 16: pool_rows<16, AFTER>(p, mask, v, lane, q, tile, col0, ncols, sc, sh, xs, bar); break;
        case 32: pool_rows<32, AFTER>(p, mask, v, lane, q, tile, col0, ncols, sc, sh, xs, bar); break;
        case 64: pool_rows<64, AFTER>(p, mask, v, lane, q, tile, col0, ncols, sc, sh, xs, bar); break;
        default: pool_rows<128, AFTER>(p, mask, v, lane, q, tile, col0, ncols, sc, sh, xs, bar); break;
    }
}

// Unit-list mode: a unit is 8 listed rows of a group = 8 consecutive lanes.  Max over the unit, then atomicMax into
// p.out_f32[group] (ok == false: this lane's unit does not exist).  Post-ReLU values are >= 0, where the unsigned order
// of the bit patterns is the float order (a -0.0 is folded to +0.0), and the caller zero-fills the output, which is also
// the result of a group without hits (the mask of layers_util.py:180).  col0 / ncols / AFTER / sc / sh as in pool_rows.
template <bool AFTER, class P>
__device__ __forceinline__ void pool_units(const P &p, float (&v)[32], int lane, int col0, int ncols, const float *sc,
                                           const float *sh, int group, bool ok)
{
    warp_colmax_transpose<8>(v, lane);                   // lane owns columns (lane % 8) * 4 + k of its unit in v[k]
    if (!ok) return;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int cc = (lane & 7) * 4 + k;
        const int col = col0 + cc;
        if (col >= ncols) continue;
        float mx = v[k];
        if (AFTER) mx = fmaxf(fmaf(mx, sc[col0 + cc], sh[col0 + cc]), 0.0f);
        atomicMax(reinterpret_cast<unsigned int *>(p.out_f32 + (size_t)group * p.ld_f32 + col), __float_as_uint(mx) & 0x7fffffffu);
    }
}

}  // namespace ssd3d
