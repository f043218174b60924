// mlp_tc.cu -- the grouped-MLP layers on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// One layer of the SA point MLP, y = act((x . W) * scale + shift) [+ max-pool over the neighbour axis], i.e. the
// conv2d/bias/BN/ReLU/reduce_max chain of /root/reference/lib/utils/tf_util.py:127-201, :424-444 and
// /root/reference/lib/utils/layers_util.py:167-180, as ONE persistent warp-specialised GEMM kernel.
//
// Precision (DESIGN.md "Grouped MLP"): the reference computes in fp32 and the parity budget is 1e-3 relative.
// A single TF32/BF16 pass does not hold that through three chained layers, so every fp32 operand is split into
// two bf16 terms, x = x_hi + x_lo (16 mantissa bits), and the product is evaluated as three bf16 MMAs
//     x.W ~= x_hi.W_hi + x_lo.W_hi + x_hi.W_lo          (error ~2^-16, fp32 accumulation in TMEM; tc.cuh)
// at 3x the bf16 tensor rate instead of the 2x-slower TF32 pipe.  Activations travel between layers already
// split (two bf16 matrices, row-major == K-major), so every operand tile is a plain TMA box in the 128B-swizzled
// canonical UMMA layout and no conversion happens on the load path.
//
// Kernel shape: 576 threads; warp 0 = TMA producer, warp 1 = MMA issuer (whole warp runs the loop, one elect.sync lane
// issues), warps 2-9 = operand producers of the gather modes (warp 2 also allocates TMEM), warps 10-17 = epilogue
// (TMEM -> registers -> scale/shift/ReLU -> fp32 / split-bf16 through TMA tensor stores, or max-pool as a shuffle
// reduce-and-transpose butterfly; two warps per TMEM lane quarter share the 32-column chunks).
// Tile 128 rows x BN<=256 columns, K streamed in 64-element blocks through a multi-stage mbarrier ring;
// two TMEM accumulator buffers let the epilogue of tile i overlap the MMAs of tile i+1.
// Gather modes (TcParams::gather): the operand tile is not read from memory but built in shared memory by the
// producer warps from neighbour indices (1: concat(features, xyz - centre); 2: the hoisted first conv) and kept
// resident across the n-tiles of its m-tile (TcParams::astat).
// Unit-list mode (TcParams::units, round 2): the grouped matrix holds only the 8-row units the ball query listed (rows
// that repeat a group's first neighbour cannot change the max-pool); the row count comes from the list at run time, the
// gather producers look their source up through it, and the last conv of a scale pools each unit and combines the units
// of a group with atomicMax (pool_units, pool.cuh).  Same bits as the dense schedule.
#include <cstdio>
#include <cstring>

#include "common.cuh"
#include "pool.cuh"
#include "tc.cuh"

namespace ssd3d {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;                 // bf16 elements per k-block = one 128-byte swizzle row
constexpr int TC_PROD_WARP0 = 2;          // warps 2..9: A-operand producers of the gather modes: two threads per tile row, each
constexpr int TC_PROD_WARPS = 8;          // builds 4 of the 8 16-byte chunks of a k-block (round 2: with 4 warps the producers
                                          // were busy 50% of the kernel while the MMA warp waited for them 35% of it)
constexpr int TC_EPI_WARP0 = TC_PROD_WARP0 + TC_PROD_WARPS;   // warps 6..13: epilogue (warp%4 selects the TMEM lane quarter)
constexpr int TC_EPI_WARPS = 8;
constexpr int TC_THREADS = (TC_EPI_WARP0 + TC_EPI_WARPS) * 32;
constexpr int TC_MAX_STAGES = 4;
constexpr int TC_MAX_AKB = 4;            // A-stationary mode: k-blocks of the resident A tile (K <= 256)
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 2;   // one A tile (hi or lo): 16 KiB

struct TcParams {
    long rows;
    int kp;          // K padded to a multiple of 16
    int n;           // output channels
    int bn;          // tile width (multiple of 16, <= 256)
    int n_tiles, m_tiles, stages;
    const float *scale, *shift;
    int relu, pool;
    const int *rowmask;
    float *out_f32; int ld_f32;
    __nv_bfloat16 *out_hi, *out_lo; int ld_split;
    int tma_store;   // non-pooled outputs leave through per-warp shared-memory blocks + TMA tensor stores
    // gather mode (first layer of an SA scale): the A operand is not read from memory but BUILT by two producer warps:
    // x[row] = concat(points[scene, idx[row], :], xyz[scene, idx[row], :] - new_xyz[scene, row/ns, :])  (layers_util.py:160-165)
    // gather == 2 ("hoisted first layer"): the operand of THIS layer is the OUTPUT of the scale's first conv, rebuilt per
    // grouped row from a per-point table instead of being computed per row:  with W1 = [Wf ; Wx] split by input rows,
    //   relu((concat(f_j, x_j - c_i) . W1) * s + t) = relu(z[j] + (x_j - c_i) . (Wx * s)),   z = (f . Wf) * s + t  [per point]
    // g_points = z (row pitch g_ldz, this scale's columns), g_c = first-layer width (= K of this layer), g_wx = Wx*s [3][g_c]
    // astat ("A-stationary", gather modes): the produced A tile of an m-tile (all its k-blocks) stays in shared memory
    // while the CTA sweeps that m-tile's n-tiles, so the producers build it once instead of once per n-tile; only the
    // weights travel through the ring.  Tiles are then enumerated m-major per CTA.  (A second resident tile, built under
    // the MMAs of the first, was measured slower and removed: DESIGN.md section 8.)
    int astat;       // 0: A through the ring; 1: one resident A tile
    int gather, g_n, g_c, g_m, g_ns, g_ldz;
    const float *g_xyz, *g_points, *g_new_xyz, *g_wx;
    const int *g_idx;
    // UNIT-LIST mode (include/ssd3d.h, ssd3d_query_ball_point_multi_ws): units[0] = U, units[1 + u] = (group << 4) | j names
    // rows 8j .. 8j+7 of a group's neighbour list.  The matrix this launch works on then has U * 8 rows -- compact row
    // 8u + e is neighbour slot 8j + e of that group -- instead of `rows` (which stays the capacity of the buffers): the
    // gather producers look their source up through the list, and unit_pool max-pools each 8-row unit and combines the
    // units of a group with atomicMax on out_f32[group] (zero-filled by the caller; values are post-ReLU, >= 0).
    const int *units;
    int unit_pool;
};

// Developer instrumentation (nvcc -DTC_PROFILE): CTA 0 accumulates, per role, the cycles spent waiting on each barrier
// and the cycles spent working; printed by the launcher.  Slots: 0 total | 1 tma wait-empty | 2 mma wait-afull |
// 3 mma wait-full(B) | 4 mma wait-tempty | 5 mma issue | 6 prod wait-slot | 7 prod load+math | 8 epi wait-tfull | 9 epi work
#ifdef TC_PROFILE
__device__ long long tc_prof[16];
#define TCP_DECL long long tcp_t = clock64(); const bool tcp_on = blockIdx.x == 0 && lane == 0
#define TCP(i) do { if (tcp_on) { const long long t_ = clock64(); atomicAdd((unsigned long long *)&tc_prof[i], (unsigned long long)(t_ - tcp_t)); tcp_t = t_; } } while (0)
#else
#define TCP_DECL do { } while (0)
#define TCP(i) do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TC_THREADS, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap map_ahi, const __grid_constant__ CUtensorMap map_alo,
                 const __grid_constant__ CUtensorMap map_bhi, const __grid_constant__ CUtensorMap map_blo,
                 const __grid_constant__ CUtensorMap map_ohi, const __grid_constant__ CUtensorMap map_olo,
                 const __grid_constant__ CUtensorMap map_of32, const TcParams p)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve: [stages] x { A_hi | A_lo | B_hi | B_lo }, per-warp output blocks (4 KiB each), then scale/shift
    const uint32_t b_bytes = (uint32_t)p.bn * TC_BK * 2;
    const int nkb = (p.kp + TC_BK - 1) / TC_BK;
    const uint32_t a_tile = (uint32_t)nkb * 2u * TC_A_BYTES;                        // one resident A tile: [nkb] x { A_hi | A_lo }
    const uint32_t a_region = p.astat ? a_tile : 0u;
    const uint32_t stage_bytes = (p.astat ? 0u : 2 * TC_A_BYTES) + 2 * b_bytes;     // ring stage
    const uint32_t b_off = p.astat ? 0u : 2 * TC_A_BYTES;                           // B_hi inside a stage
    // 1 KiB alignment by pointer arithmetic on the __shared__ array (an integer round-trip would demote every access
    // through these pointers to generic LD/ST with 64-bit address math)
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int ncov = p.n_tiles * p.bn + 32;
    uint8_t *ring = smem + a_region;
    uint8_t *out_stage = ring + (size_t)p.stages * stage_bytes;          // [8 warps][4 KiB], 4 KiB aligned
    float *s_scale = reinterpret_cast<float *>(out_stage + (p.tma_store ? TC_EPI_WARPS * 4096 : 0));
    float *s_shift = s_scale + ncov;
    float *s_wx = s_shift + ncov;                                        // [3][kp] (hoisted mode only)

    __shared__ unsigned long long full_bar[TC_MAX_STAGES], empty_bar[TC_MAX_STAGES], tfull_bar[2], tempty_bar[2];
    __shared__ unsigned long long afull_bar[TC_MAX_AKB], aempty_bar[TC_MAX_AKB];   // per k-block of the resident A tile
    __shared__ uint32_t tmem_base_smem;
    __shared__ float pool_xs[2 * 4 * 32];

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // provably warp-uniform
    // unit-list mode: the row count comes from the list (written earlier on this stream), p.rows is the buffers' capacity
    const int nunits = p.units ? __ldg(p.units) : 0;
    const long rows = p.units ? (long)nunits * 8 : p.rows;
    const int m_tiles = p.units ? (nunits + TC_BM / 8 - 1) / (TC_BM / 8) : p.m_tiles;
    // local tile i of this CTA -> (mt, nt): n-major round robin over all tiles, or (astat) every n-tile of an m-tile
    auto tile_at = [&](int i, int &mt, int &nt) -> bool {
        if (p.astat) {
            mt = (int)blockIdx.x + (i / p.n_tiles) * (int)gridDim.x;
            nt = i % p.n_tiles;
            return mt < m_tiles;
        }
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        mt = tile / p.n_tiles;
        nt = tile - mt * p.n_tiles;
        return tile < m_tiles * p.n_tiles;
    };

    if (threadIdx.x == 0) {
        // full barrier: the TMA thread's expect_tx arrival (+ one arrival per producer warp in gather mode)
        for (int s = 0; s < p.stages; s++) { mbar_init(smem_u32(&full_bar[s]), (p.gather && !p.astat) ? 1 + TC_PROD_WARPS : 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
        for (int k = 0; k < TC_MAX_AKB; k++) { mbar_init(smem_u32(&afull_bar[k]), TC_PROD_WARPS); mbar_init(smem_u32(&aempty_bar[k]), 1); }
        for (int a = 0; a < 2; a++) { mbar_init(smem_u32(&tfull_bar[a]), 1); mbar_init(smem_u32(&tempty_bar[a]), TC_EPI_WARPS); }
        fence_mbar_init_cluster();
    }
    if (warp == 2) tmem_alloc(&tmem_base_smem, 512u);
    for (int i = threadIdx.x; i < ncov; i += TC_THREADS) {      // columns >= n: scale = shift = 0 -> exact zeros
        s_scale[i] = i < p.n ? __ldg(p.scale + i) : 0.0f;
        s_shift[i] = i < p.n ? __ldg(p.shift + i) : 0.0f;
    }
    if (p.gather == 2)
        for (int i = threadIdx.x; i < 3 * p.kp; i += TC_THREADS) {
            const int a = i / p.kp, k = i - a * p.kp;
            s_wx[i] = k < p.g_c ? __ldg(p.g_wx + a * p.g_c + k) : 0.0f;
        }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ahi) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_alo) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bhi) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_blo) : "memory");
            int it = 0, mt, nt;
            TCP_DECL;
            for (int i = 0; tile_at(i, mt, nt); i++) {
                for (int kb = 0; kb < nkb; kb++, it++) {
                    const int s = it % p.stages;
                    const uint32_t ph = (uint32_t)(it / p.stages) & 1u;
                    TCP(15);
                    mbar_wait_cta(smem_u32(&empty_bar[s]), ph ^ 1u);
                    TCP(1);
                    const uint32_t base = smem_u32(ring + (size_t)s * stage_bytes);
                    const uint32_t fb = smem_u32(&full_bar[s]);
                    mbar_arrive_expect_tx(fb, p.gather ? 2 * b_bytes : stage_bytes);
                    if (!p.gather) {
                        tma_load_2d(base, &map_ahi, kb * TC_BK, mt * TC_BM, fb);
                        tma_load_2d(base + TC_A_BYTES, &map_alo, kb * TC_BK, mt * TC_BM, fb);
                    }
                    tma_load_2d(base + b_off, &map_bhi, kb * TC_BK, nt * p.bn, fb);
                    tma_load_2d(base + b_off + b_bytes, &map_blo, kb * TC_BK, nt * p.bn, fb);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp runs the loop (uniform control flow keeps descriptors in uniform registers
        // and tcgen05.mma free of a per-instruction election loop), one elected lane issues =====
        {
            const uint32_t idesc = umma_idesc_bf16(p.bn);
            int it = 0, tcount = 0, mi = 0, mt, nt;
            TCP_DECL;
            for (int i = 0; tile_at(i, mt, nt); i++, tcount++) {
                const int acc = tcount & 1;
                TCP(5);
                mbar_wait_cta(smem_u32(&tempty_bar[acc]), (((uint32_t)(tcount >> 1)) & 1u) ^ 1u);
                TCP(4);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.bn);
                const bool last_nt = nt == p.n_tiles - 1;
                for (int kb = 0; kb < nkb; kb++, it++) {
                    const int s = it % p.stages;
                    TCP(5);
                    if (p.astat && nt == 0) mbar_wait_cta(smem_u32(&afull_bar[kb]), (uint32_t)mi & 1u);   // this m-tile's A k-block
                    TCP(2);
                    mbar_wait_cta(smem_u32(&full_bar[s]), (uint32_t)(it / p.stages) & 1u);
                    TCP(3);
                    tc_fence_after();
                    const uint32_t base = smem_u32(ring + (size_t)s * stage_bytes);
                    const uint32_t abase = p.astat ? smem_u32(smem) + (uint32_t)kb * 2u * TC_A_BYTES : base;
                    const int ksteps = min(TC_BK, p.kp - kb * TC_BK) / 16;
                    const uint64_t a_hi = umma_desc(abase, 128), a_lo = umma_desc(abase + TC_A_BYTES, 128);
                    const uint64_t b_hi = umma_desc(base + b_off, 128), b_lo = umma_desc(base + b_off + b_bytes, 128);
                    if (elect_one()) {
                        for (int ks = 0; ks < ksteps; ks++)           // +2 per k-step: 32 bytes in the address field
                            umma_bf16x3(d_tmem, a_hi + 2 * ks, a_lo + 2 * ks, b_hi + 2 * ks, b_lo + 2 * ks, idesc, (kb | ks) ? 1u : 0u);
                        umma_commit(smem_u32(&empty_bar[s]));   // ring stage free once these MMAs retire
                        if (p.astat && last_nt) umma_commit(smem_u32(&aempty_bar[kb]));   // A k-block free again
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(smem_u32(&tfull_bar[acc]));   // accumulator ready for the epilogue
                __syncwarp();
                if (last_nt) mi++;
            }
        }
    } else if (warp >= TC_PROD_WARP0 && warp < TC_EPI_WARP0) {
        // ===== A-operand producers (gather mode): 128 threads, one row of the tile each.  A row's source features are
        // one contiguous run (16-byte loads when c % 4 == 0); all loads of a 64-wide k-block are issued before the
        // values are split into bf16 hi/lo and stored as 16-byte chunks in the K-major SWIZZLE_128B layout the UMMA
        // descriptor expects.
        if (p.gather) {
            const int pt = threadIdx.x - TC_PROD_WARP0 * 32;
            const int r = pt & (TC_BM - 1);                      // tile row
            const int c16_0 = (pt >> 7) * 4;                     // this thread's 4 chunks of every k-block
            const uint32_t rps = (uint32_t)p.g_m * (uint32_t)p.g_ns;
            const bool hoisted = p.gather == 2;
            const int src_pitch = hoisted ? p.g_ldz : p.g_c;
            const bool vec4 = (p.g_c % 4 == 0) && (src_pitch % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.g_points) & 15u) == 0);
            const uint32_t row_off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u;
            int it = 0, mi = 0, mt, nt;
            TCP_DECL;
            for (int i = 0; tile_at(i, mt, nt); i++) {
                if (p.astat && nt != 0) continue;                 // A-stationary: the tile built for nt == 0 serves every n-tile
                const uint32_t row = (uint32_t)mt * TC_BM + (uint32_t)r;
                const bool ok = (long)row < rows;
                uint32_t rr = ok ? row : 0u;                      // position of this row's neighbour in idx[]
                if (p.units && ok) {
                    const uint32_t desc = (uint32_t)__ldg(p.units + 1 + (row >> 3));
                    rr = (desc >> 4) * (uint32_t)p.g_ns + ((desc & 15u) << 3) + (row & 7u);
                }
                const uint32_t scene = rr / rps, q = rr / (uint32_t)p.g_ns;
                const int a = __ldg(p.g_idx + rr);
                const float *src_f = p.g_points + ((size_t)scene * p.g_n + a) * src_pitch;
                const float *src_x = p.g_xyz + ((size_t)scene * p.g_n + a) * 3;
                const float *ctr = p.g_new_xyz + (size_t)q * 3;
                float dx = 0.0f, dy = 0.0f, dz = 0.0f;
                if (hoisted && ok) {
                    dx = __ldg(src_x) - __ldg(ctr); dy = __ldg(src_x + 1) - __ldg(ctr + 1); dz = __ldg(src_x + 2) - __ldg(ctr + 2);
                }
                for (int kb = 0; kb < nkb; kb++, it++) {
                    const int s = it % p.stages;
                    float f[4][8];
#pragma unroll
                    for (int cc = 0; cc < 4; cc++) {
                        const int k0 = kb * TC_BK + (c16_0 + cc) * 8;
                        if (vec4 && ok && k0 + 8 <= p.g_c) {
                            const float4 u0 = __ldg(reinterpret_cast<const float4 *>(src_f + k0));
                            const float4 u1 = __ldg(reinterpret_cast<const float4 *>(src_f + k0 + 4));
                            f[cc][0] = u0.x; f[cc][1] = u0.y; f[cc][2] = u0.z; f[cc][3] = u0.w;
                            f[cc][4] = u1.x; f[cc][5] = u1.y; f[cc][6] = u1.z; f[cc][7] = u1.w;
                        } else {
#pragma unroll
                            for (int e = 0; e < 8; e++) {
                                const int k = k0 + e;
                                float val = 0.0f;
                                if (ok && k < p.kp) {
                                    if (k < p.g_c) val = __ldg(src_f + k);
                                    else if (!hoisted && k < p.g_c + 3) val = __ldg(src_x + (k - p.g_c)) - __ldg(ctr + (k - p.g_c));
                                }
                                f[cc][e] = val;
                            }
                        }
                    }
                    // (loads already in flight) wait for the slot: ring stage, or this k-block of the resident A tile
                    if (warp == TC_PROD_WARP0) TCP(7);
                    if (p.astat) mbar_wait_cta(smem_u32(&aempty_bar[kb]), ((uint32_t)mi & 1u) ^ 1u);
                    else mbar_wait_cta(smem_u32(&empty_bar[s]), ((uint32_t)(it / p.stages) & 1u) ^ 1u);
                    if (warp == TC_PROD_WARP0) TCP(6);
                    uint8_t *rowp = (p.astat ? smem + (size_t)kb * 2 * TC_A_BYTES : ring + (size_t)s * stage_bytes) + row_off;
#pragma unroll
                    for (int cc = 0; cc < 4; cc++) {
                        const int c16 = c16_0 + cc;
                        const int k0 = kb * TC_BK + c16 * 8;
                        if (k0 >= p.kp) break;
                        if (hoisted) hoist_relu8(f[cc], dx, dy, dz, s_wx + k0, p.kp);   // rows beyond the tensor stay 0
                        const uint32_t off = (uint32_t)((c16 ^ (r & 7)) << 4);
                        split8_store(f[cc], rowp + off, rowp + TC_A_BYTES + off);
                    }
                    fence_async_smem();                                   // generic-proxy stores -> visible to the tensor core
                    __syncwarp();
                    if (lane == 0) mbar_arrive(smem_u32(p.astat ? &afull_bar[kb] : &full_bar[s]));
                }
                mi++;
            }
        }
    } else if (warp >= TC_EPI_WARP0) {
        // ===== epilogue: 8 warps; warp%4 = TMEM lane quarter (rows), (warp-4)/4 = which half of the 32-column chunks
        const int q = warp & 3;
        const int h = (warp - TC_EPI_WARP0) >> 2;
        const int nchunks = (p.bn + 31) / 32;
        int tcount = 0, mt, nt;
        TCP_DECL;
        for (int i = 0; tile_at(i, mt, nt); i++, tcount++) {
            const int acc = tcount & 1;
            if (warp == TC_EPI_WARP0) TCP(9);
            mbar_wait_cta(smem_u32(&tfull_bar[acc]), ((uint32_t)(tcount >> 1)) & 1u);
            if (warp == TC_EPI_WARP0) TCP(8);
            tc_fence_after();
            const long row = (long)mt * TC_BM + q * 32 + lane;
            const bool row_ok = row < rows;
            for (int ci = h; ci < nchunks; ci += 2) {
                const int c0 = ci * 32;
                uint32_t r[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * p.bn + c0), r);
                const int col0 = nt * p.bn + c0;
                float v[32];
#pragma unroll
                for (int j4 = 0; j4 < 32; j4 += 4) {
                    const float4 sc = *reinterpret_cast<const float4 *>(s_scale + col0 + j4);
                    const float4 sh = *reinterpret_cast<const float4 *>(s_shift + col0 + j4);
                    v[j4 + 0] = fmaf(__uint_as_float(r[j4 + 0]), sc.x, sh.x);
                    v[j4 + 1] = fmaf(__uint_as_float(r[j4 + 1]), sc.y, sh.y);
                    v[j4 + 2] = fmaf(__uint_as_float(r[j4 + 2]), sc.z, sh.z);
                    v[j4 + 3] = fmaf(__uint_as_float(r[j4 + 3]), sc.w, sh.w);
                }
                if (p.relu) {
#pragma unroll
                    for (int j = 0; j < 32; j++) v[j] = fmaxf(v[j], 0.0f);
                }
                if (p.pool <= 1 && p.tma_store) {
                    // Each warp owns a [32 rows x 32 columns] block: stage it in shared memory in the TMA swizzle and
                    // let one bulk tensor store write whole 64/128-byte row segments (rows / columns beyond the tensor
                    // are clipped by the hardware); the block is reused once the previous store has read it.
                    uint8_t *blk = out_stage + (warp - TC_EPI_WARP0) * 4096;
                    if (lane == 0) tma_store_wait_read();
                    __syncwarp();
                    const int row0 = mt * TC_BM + q * 32;
                    if (p.out_f32) {                                   // 128-byte rows, SWIZZLE_128B
#pragma unroll
                        for (int c = 0; c < 8; c++)
                            *reinterpret_cast<float4 *>(blk + lane * 128 + ((c ^ (lane & 7)) << 4)) =
                                make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) { tma_store_2d(&map_of32, smem_u32(blk), col0, row0); tma_store_commit(); }
                    } else {                                           // two 64-byte-row blocks (hi, lo), SWIZZLE_64B
#pragma unroll
                        for (int c = 0; c < 4; c++) {
                            const uint32_t off = (uint32_t)lane * 64u + (uint32_t)((c ^ ((lane >> 1) & 3)) << 4);
                            split8_store(v + 8 * c, blk + off, blk + 2048 + off);
                        }
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_2d(&map_ohi, smem_u32(blk), col0, row0);
                            tma_store_2d(&map_olo, smem_u32(blk + 2048), col0, row0);
                            tma_store_commit();
                        }
                    }
                } else if (p.pool <= 1) {
                    if (row_ok) {
                        if (p.out_f32) {
                            float *dst = p.out_f32 + (size_t)row * p.ld_f32 + col0;
                            if (col0 + 32 <= p.n && ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0)) {
#pragma unroll
                                for (int j4 = 0; j4 < 32; j4 += 4)
                                    *reinterpret_cast<float4 *>(dst + j4) = make_float4(v[j4], v[j4 + 1], v[j4 + 2], v[j4 + 3]);
                            } else {
#pragma unroll
                                for (int j = 0; j < 32; j++)
                                    if (col0 + j < p.n) dst[j] = v[j];
                            }
                        }
                        if (p.out_hi) {
                            // x = hi + lo (bf16 each); columns n..ld_split-1 come out as exact zeros (next layer's K padding)
                            __nv_bfloat16 *dh = p.out_hi + (size_t)row * p.ld_split + col0;
                            __nv_bfloat16 *dl = p.out_lo + (size_t)row * p.ld_split + col0;
#pragma unroll
                            for (int j8 = 0; j8 < 32; j8 += 8) {
                                if (col0 + j8 >= p.ld_split) break;
                                split8_store(v + j8, dh + j8, dl + j8);
                            }
                        }
                    }
                } else if (p.unit_pool) {                              // lanes 8u' .. 8u'+7 of a warp hold one unit
                    const int ui = mt * (TC_BM / 8) + ((q * 32 + lane) >> 3);
                    const bool ok = ui < nunits;
                    pool_units<false>(p, v, lane, col0, p.n, nullptr, nullptr, ok ? __ldg(p.units + 1 + ui) >> 4 : 0, ok);
                } else {                                               // the 4 quarter-warps of column half h: barrier 2 + h
                    pool_rows<false>(p.pool, p, p.rowmask, v, lane, q, mt, col0, p.n, nullptr, nullptr, pool_xs + h * 4 * 32, 2 + h);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&tempty_bar[acc]));   // 8 arrivals (one per epilogue warp) free the buffer
        }
        if (p.tma_store && lane == 0) tma_store_wait_all();           // global writes complete before the CTA retires
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512u);
    }
}

// ---- fp32 -> split bf16 producers -------------------------------------------------------------------------
__device__ __forceinline__ void split_store(float x, __nv_bfloat16 *hi, __nv_bfloat16 *lo)
{
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    *hi = h;
    *lo = __float2bfloat16_rn(x - __bfloat162float(h));
}

// hi/lo[row, 0:kp] = split(x[row, 0:c]) zero-padded
__global__ void split_rows_kernel(long rows, int c, const float *__restrict__ x, int ldx, __nv_bfloat16 *__restrict__ hi,
                                  __nv_bfloat16 *__restrict__ lo, int kp)
{
    const long total = rows * kp;
    for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const long row = e / kp;
        const int col = (int)(e - row * kp);
        split_store(col < c ? __ldg(x + (size_t)row * ldx + col) : 0.0f, hi + e, lo + e);
    }
}

// the same, one 8-column chunk per thread and step: two 16-byte loads (when the source rows allow), two 16-byte stores
__global__ void __launch_bounds__(256)
split_rows_v8_kernel(unsigned nchunks, int c, const float *__restrict__ x, int ldx, __nv_bfloat16 *__restrict__ hi,
                     __nv_bfloat16 *__restrict__ lo, int kp, int vec)
{
    const unsigned cpr = (unsigned)kp >> 3;                            // chunks per row
    for (unsigned ch = blockIdx.x * blockDim.x + threadIdx.x; ch < nchunks; ch += gridDim.x * blockDim.x) {
        const unsigned row = ch / cpr;
        const int k0 = (int)(ch - row * cpr) * 8;
        const float *src = x + (size_t)row * ldx + k0;
        float f[8];
        if (vec && k0 + 8 <= c) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(src)), b2 = __ldg(reinterpret_cast<const float4 *>(src + 4));
            f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b2.x; f[5] = b2.y; f[6] = b2.z; f[7] = b2.w;
        } else {
#pragma unroll
            for (int e = 0; e < 8; e++) f[e] = k0 + e < c ? __ldg(src + e) : 0.0f;
        }
        uint32_t hw[4], lw[4];
#pragma unroll
        for (int t = 0; t < 4; t++) split_pair(f[2 * t], f[2 * t + 1], hw[t], lw[t]);
        const size_t off = (size_t)row * kp + k0;
        *reinterpret_cast<uint4 *>(hi + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4 *>(lo + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
}

// fused gather + concat[features, rel-xyz] + split (layers_util.py:160-165), zero-padded to kp columns.
// One warp per output row: the source feature row is one contiguous run (coalesced 16-byte loads when c % 4 == 0),
// the two bf16 rows are written as contiguous 8-byte pieces.
__global__ void __launch_bounds__(256)
group_concat_split_kernel(long rows, int n, int c, int m, int ns, const float *__restrict__ xyz,
                          const float *__restrict__ points, const float *__restrict__ new_xyz,
                          const int *__restrict__ idx, __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo,
                          int kp, int vec4)
{
    constexpr int U = 4;                              // rows in flight per warp (independent load chains)
    extern __shared__ __align__(16) __nv_bfloat16 gcs_stage[];   // [8 warps][U rows][hi kp | lo kp]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    __nv_bfloat16 *st = gcs_stage + (size_t)wib * U * 2 * kp;
    const long warp0 = (blockIdx.x * (long)blockDim.x + threadIdx.x) >> 5;
    const long nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    const long rows_per_scene = (long)m * ns;
    const int nchunk = kp >> 3;                       // 16-byte chunks per (hi or lo) row
    for (long rbase = warp0 * U; rbase < rows; rbase += nwarps * U) {
        int a[U];
        long scene[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const long row = rbase + u;
            a[u] = row < rows ? __ldg(idx + row) : 0;
            scene[u] = row < rows ? row / rows_per_scene : 0;
        }
        int k4 = 0;
        if (vec4) {                                   // c % 4 == 0, 16-byte aligned feature rows
            for (k4 = lane * 4; k4 + 3 < c; k4 += 128) {
                float4 f[U];
#pragma unroll
                for (int u = 0; u < U; u++)
                    f[u] = __ldg(reinterpret_cast<const float4 *>(points + ((size_t)scene[u] * n + a[u]) * c + k4));
#pragma unroll
                for (int u = 0; u < U; u++) {
                    uint32_t h0, l0, h1, l1;
                    split_pair(f[u].x, f[u].y, h0, l0);
                    split_pair(f[u].z, f[u].w, h1, l1);
                    *reinterpret_cast<uint2 *>(st + (size_t)u * 2 * kp + k4) = make_uint2(h0, h1);
                    *reinterpret_cast<uint2 *>(st + (size_t)u * 2 * kp + kp + k4) = make_uint2(l0, l1);
                }
            }
            k4 = c & ~3;
        }
        // tail: remaining feature columns, the 3 relative coordinates, zero padding up to kp
#pragma unroll
        for (int u = 0; u < U; u++) {
            const long row = rbase + u;
            const float *src = points + ((size_t)scene[u] * n + a[u]) * c;
            for (int k = k4 + lane; k < kp; k += 32) {
                float val = 0.0f;
                if (row < rows) {
                    if (k < c) val = __ldg(src + k);
                    else if (k < c + 3) {
                        const long q = row / ns;
                        val = __ldg(xyz + ((size_t)scene[u] * n + a[u]) * 3 + (k - c)) - __ldg(new_xyz + q * 3 + (k - c));
                    }
                }
                split_store(val, st + (size_t)u * 2 * kp + k, st + (size_t)u * 2 * kp + kp + k);
            }
        }
        __syncwarp();
        // whole 16-byte chunks to global: the U rows are consecutive, so hi (and lo) of the warp is one contiguous run
#pragma unroll
        for (int u = 0; u < U; u++) {
            const long row = rbase + u;
            if (row >= rows) break;
            const uint4 *sv = reinterpret_cast<const uint4 *>(st + (size_t)u * 2 * kp);
            uint4 *dh = reinterpret_cast<uint4 *>(hi + (size_t)row * kp);
            uint4 *dl = reinterpret_cast<uint4 *>(lo + (size_t)row * kp);
            for (int ch = lane; ch < 2 * nchunk; ch += 32) {
                if (ch < nchunk) dh[ch] = sv[ch];
                else dl[ch - nchunk] = sv[ch];
            }
        }
        __syncwarp();
    }
}

// The operand of the conv that follows a HOISTED first conv (TcParams::gather == 2), materialised once in split bf16:
//   row (i, j):  relu(z[idx[i,j], :] + (xyz[idx[i,j]] - new_xyz[i]) . wx)        zero-padded to kp columns.
// For wide layers (K >= 256, 3DSSD layer 4) the A-stationary in-kernel producers starve the tensor pipe -- 128 KiB of
// resident operand leave room for two narrow weight stages -- while this elementwise pass runs at memory speed on the whole
// machine and the GEMM then takes the plain TMA-fed path.  One warp per row, one 8-column chunk per lane per step.
// 8 blocks per SM: a full SM of warps for this memory-bound pass (the compiler would otherwise take 43 registers).
__global__ void __launch_bounds__(256, 8)
hoist_expand_split_kernel(long rows, int n, int n1, int m, int ns, const float *__restrict__ xyz, const float *__restrict__ z,
                          int ldz, const float *__restrict__ wx, const float *__restrict__ new_xyz,
                          const int *__restrict__ idx, const int *__restrict__ units, __nv_bfloat16 *__restrict__ hi,
                          __nv_bfloat16 *__restrict__ lo, int kp)
{
    extern __shared__ __align__(16) float hx_wx[];                      // [3][kp] zero padded
    if (units) rows = (long)__ldg(units) * 8;                           // unit-list mode (TcParams::units): compact rows
    for (int i = threadIdx.x; i < 3 * kp; i += blockDim.x) {
        const int a = i / kp, k = i - a * kp;
        hx_wx[i] = k < n1 ? __ldg(wx + a * n1 + k) : 0.0f;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long warp0 = (blockIdx.x * (long)blockDim.x + threadIdx.x) >> 5, nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    const long rps = (long)m * ns;
    const int nchunk = kp >> 3;
    for (long row = warp0; row < rows; row += nwarps) {
        long src = row;                                                  // position of this row's neighbour in idx[]
        if (units) {
            const unsigned desc = (unsigned)__ldg(units + 1 + (row >> 3));
            src = (long)(desc >> 4) * ns + ((desc & 15u) << 3) + (row & 7);
        }
        const long scene = src / rps, q = src / ns;
        const int a = __ldg(idx + src);
        const float *px = xyz + ((size_t)scene * n + a) * 3, *pc = new_xyz + (size_t)q * 3;
        const float dx = __ldg(px) - __ldg(pc), dy = __ldg(px + 1) - __ldg(pc + 1), dz = __ldg(px + 2) - __ldg(pc + 2);
        const float *zr = z + ((size_t)scene * n + a) * ldz;
        for (int ch = lane; ch < nchunk; ch += 32) {
            const int k0 = ch * 8;
            float f[8];
            if (k0 + 8 <= n1) {
                const float4 u0 = __ldg(reinterpret_cast<const float4 *>(zr + k0)), u1 = __ldg(reinterpret_cast<const float4 *>(zr + k0 + 4));
                f[0] = u0.x; f[1] = u0.y; f[2] = u0.z; f[3] = u0.w; f[4] = u1.x; f[5] = u1.y; f[6] = u1.z; f[7] = u1.w;
            } else {
#pragma unroll
                for (int e = 0; e < 8; e++) f[e] = k0 + e < n1 ? __ldg(zr + k0 + e) : 0.0f;
            }
            hoist_relu8(f, dx, dy, dz, hx_wx + k0, kp);
            split8_store(f, hi + (size_t)row * kp + k0, lo + (size_t)row * kp + k0);
        }
    }
}

// ---- host side ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// bf16 matrix [nrows x kp] row-major -> 2D tensor map, box = 64 columns x box_rows, 128B swizzle, zero OOB fill
static int make_map(CUtensorMap *map, const void *ptr, long nrows, int kp, int box_rows)
{
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return SSD3D_ERR_UNSUPPORTED; }
    cuuint64_t dims[2] = {(cuuint64_t)kp, (cuuint64_t)nrows};
    cuuint64_t strides[1] = {(cuuint64_t)kp * 2};
    cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (CUresult %d) for [%ld x %d]", (int)r, nrows, kp); return SSD3D_ERR_INVALID_ARGUMENT; }
    return 0;
}

// output matrix [nrows x ncols] (row pitch ld elements) -> 2D map with a [32 x 32] box for the per-warp stores
static int make_out_map(CUtensorMap *map, const void *ptr, long nrows, int ncols, int ld, bool f32)
{
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return SSD3D_ERR_UNSUPPORTED; }
    const int esz = f32 ? 4 : 2;
    cuuint64_t dims[2] = {(cuuint64_t)ncols, (cuuint64_t)nrows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(ptr),
                     dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (output) failed (CUresult %d)", (int)r); return SSD3D_ERR_INVALID_ARGUMENT; }
    return 0;
}

}  // namespace ssd3d

using namespace ssd3d;


struct TcGather { int b, n, c, m, ns; const float *xyz, *points, *new_xyz; const int *idx; int ldz; const float *wx; };

static int linear_tc_launch(long rows, int kp, int n, const void *a_hi, const void *a_lo, const TcGather *g,
                            const void *b_hi, const void *b_lo, const float *scale, const float *shift, int relu, int pool,
                            const int *rowmask, float *out_f32, int ld_f32, void *out_hi, void *out_lo, int ld_split,
                            cudaStream_t stream, const int *units = nullptr, int unit_pool = 0)
{
    SSD3D_REQUIRE(rows >= 0 && kp > 0 && n > 0, "linear_tc: bad shape rows=%ld kp=%d n=%d", rows, kp, n);
    if (units) {
        SSD3D_REQUIRE(rows % 8 == 0 && pool == 1 && rowmask == nullptr, "linear_tc (unit list): rows=%ld must be a multiple of 8, no pool / rowmask", rows);
        if (unit_pool) {
            SSD3D_REQUIRE(relu && out_f32 && !out_hi, "linear_tc (unit list): pooling combines post-ReLU values by atomicMax into out_f32 only");
            pool = 8;
        }
    } else {
        SSD3D_REQUIRE(!unit_pool, "linear_tc: unit_pool needs a unit list");
    }
    SSD3D_REQUIRE(kp % 16 == 0, "linear_tc: kp=%d must be a multiple of 16", kp);
    SSD3D_REQUIRE((g || (a_hi && a_lo)) && b_hi && b_lo && scale && shift, "linear_tc: null operand pointer");
    SSD3D_REQUIRE(out_f32 || (out_hi && out_lo), "linear_tc: no output requested");
    SSD3D_REQUIRE(!out_f32 || ld_f32 >= n, "linear_tc: ld_f32=%d < n=%d", ld_f32, n);
    SSD3D_REQUIRE(!out_hi || (out_lo && ld_split >= n && ld_split % 8 == 0), "linear_tc: bad split output (ld_split=%d)", ld_split);
    SSD3D_REQUIRE(pool == 1 || pool == 8 || pool == 16 || pool == 32 || pool == 64 || pool == 128,
                  "linear_tc: pool=%d must be one of 1, 8, 16, 32, 64, 128", pool);
    SSD3D_REQUIRE(rows % pool == 0, "linear_tc: rows=%ld not a multiple of pool=%d", rows, pool);
    SSD3D_REQUIRE(rows < (1L << 31) - 256, "linear_tc: too many rows (%ld)", rows);
    for (const void *ptr : {a_hi, a_lo, b_hi, b_lo, (const void *)out_hi, (const void *)out_lo})
        SSD3D_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15u) == 0, "linear_tc: operand pointers must be 16-byte aligned");
    if (rows == 0) return 0;

    TcParams p = {};
    p.rows = rows; p.kp = kp; p.n = n;
    if (g) {
        p.gather = g->wx ? 2 : 1; p.g_n = g->n; p.g_c = g->c; p.g_m = g->m; p.g_ns = g->ns;
        p.g_xyz = g->xyz; p.g_points = g->points; p.g_new_xyz = g->new_xyz; p.g_idx = g->idx;
        p.g_ldz = g->ldz; p.g_wx = g->wx;
    }
    const int n16 = (n + 15) / 16 * 16;
    // when split outputs are requested the tile must also cover (and zero) the padding columns n..ld_split-1
    const int ncover = out_hi && pool <= 1 ? (ld_split > n16 ? ld_split : n16) : n16;
    // Non-pooled outputs go through TMA tensor stores when exactly one kind is requested and it is 16-byte
    // addressable; their tiles are capped at 128 columns to leave shared memory for the per-warp store blocks.
    const bool want_f32 = out_f32 != nullptr, want_split = out_hi != nullptr;
    bool tma_store = pool <= 1 && (want_f32 != want_split);
    if (tma_store && want_f32) tma_store = (ld_f32 % 4 == 0) && ((reinterpret_cast<uintptr_t>(out_f32) & 15u) == 0);
    p.tma_store = tma_store ? 1 : 0;
    const size_t budget = 224 * 1024 - 1024;   // 227 KiB per CTA minus static barriers and the 1 KiB alignment slack
    const int nkb = (kp + TC_BK - 1) / TC_BK;
    auto misc_bytes = [&](int bn) {            // scale/shift (+ hoisted Wx) + per-warp store blocks
        const int nt = (ncover + bn - 1) / bn;
        return 2 * ((size_t)nt * bn + 32) * sizeof(float) + (tma_store ? TC_EPI_WARPS * 4096 : 0) +
               (g && g->wx ? (size_t)3 * kp * sizeof(float) : 0);
    };
    // gather modes keep the produced A tile resident (A-stationary) when all its k-blocks fit next to a >= 2-stage
    // weight ring: the producers then build it once per m-tile, not once per (m, n) tile.  A second resident tile (the
    // producers building m-tile i+1 under the MMAs of m-tile i) had to be paid for with the TMA store blocks and lost on
    // the layer-3 shapes; it was removed (DESIGN.md section 8 keeps the measurement).
    int bn = 0, stages = 0;
    p.astat = 0;
    if (g && nkb <= TC_MAX_AKB) {
        const size_t a_tile = (size_t)nkb * 2 * TC_A_BYTES;
        const int cands[4] = {256, 128, 96, 64};            // widest tile first: a tcgen05.mma has a fixed cost per instruction
        for (int ci = tma_store ? 1 : 0; ci < 4 && !bn; ci++) {
            const int cand = cands[ci];
            const int b = ncover < cand ? ncover : cand;
            const size_t need = a_tile + misc_bytes(b);
            if (need + 2 * (size_t)(2 * b * TC_BK * 2) <= budget) {
                bn = b;
                stages = (int)((budget - need) / (size_t)(2 * b * TC_BK * 2));
                p.astat = 1;
            }
        }
    }
    if (!bn) {
        const int bn_cap = tma_store ? 128 : 256;
        bn = ncover < bn_cap ? ncover : bn_cap;
        stages = (int)((budget - misc_bytes(bn)) / (2 * (size_t)TC_A_BYTES + 2 * (size_t)bn * TC_BK * 2));
    }
    p.bn = bn;
    p.n_tiles = (ncover + p.bn - 1) / p.bn;
    p.m_tiles = (int)((rows + TC_BM - 1) / TC_BM);
    const size_t stage_bytes = (p.astat ? 0 : 2 * (size_t)TC_A_BYTES) + 2 * (size_t)p.bn * TC_BK * 2;
    const size_t pool_bytes = misc_bytes(p.bn) + (p.astat ? (size_t)nkb * 2 * TC_A_BYTES : 0);
    SSD3D_REQUIRE((size_t)p.n_tiles * p.bn <= 4096, "linear_tc: n=%d too wide for the staged scale/shift", n);
    if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
    SSD3D_REQUIRE(stages >= 2, "linear_tc: tile does not fit shared memory");
    p.stages = stages;
    p.scale = scale; p.shift = shift; p.relu = relu; p.pool = pool; p.rowmask = rowmask;
    p.units = units; p.unit_pool = unit_pool;
    p.out_f32 = out_f32; p.ld_f32 = ld_f32;
    p.out_hi = (__nv_bfloat16 *)out_hi; p.out_lo = (__nv_bfloat16 *)out_lo; p.ld_split = ld_split;

    CUtensorMap mah, mal, mbh, mbl;
    int rc;
    if ((rc = make_map(&mbh, b_hi, n, kp, p.bn)) != 0) return rc;
    if ((rc = make_map(&mbl, b_lo, n, kp, p.bn)) != 0) return rc;
    mah = mbh; mal = mbh;                          // placeholders in gather mode (never dereferenced)
    if (!g) {
        if ((rc = make_map(&mah, a_hi, rows, kp, TC_BM)) != 0) return rc;
        if ((rc = make_map(&mal, a_lo, rows, kp, TC_BM)) != 0) return rc;
    }
    CUtensorMap moh = mbh, mol = mbh, mof = mbh;   // placeholders when unused
    if (tma_store && want_split) {
        if ((rc = make_out_map(&moh, out_hi, rows, ld_split, ld_split, false)) != 0) return rc;
        if ((rc = make_out_map(&mol, out_lo, rows, ld_split, ld_split, false)) != 0) return rc;
    }
    if (tma_store && want_f32 && (rc = make_out_map(&mof, out_f32, rows, n, ld_f32, true)) != 0) return rc;

    const size_t smem = stages * stage_bytes + pool_bytes + 1024;
    cudaError_t e = cudaFuncSetAttribute((const void *)linear_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "linear_tc attr");
    const int total = p.astat ? p.m_tiles : p.m_tiles * p.n_tiles;    // A-stationary CTAs own whole m-tiles
    const int grid = total < kNumSMs ? total : kNumSMs;
#ifdef TC_PROFILE
    const long long t_host0 = 0;
    (void)t_host0;
    cudaEvent_t pe0, pe1;
    cudaEventCreate(&pe0); cudaEventCreate(&pe1);
    cudaEventRecord(pe0, stream);
#endif
    linear_tc_kernel<<<grid, TC_THREADS, smem, stream>>>(mah, mal, mbh, mbl, moh, mol, mof, p);
#ifdef TC_PROFILE
    {
        cudaEventRecord(pe1, stream);
        cudaDeviceSynchronize();
        float ms = 0.f;
        cudaEventElapsedTime(&ms, pe0, pe1);
        long long h[16];
        cudaMemcpyFromSymbol(h, tc_prof, sizeof(h));
        fprintf(stderr, "tc_prof rows=%ld kp=%d n=%d bn=%d astat=%d stages=%d gather=%d pool=%d tiles/cta=%.1f  %.1f us |"
                " tma_wait %lld | mma: afull %lld bfull %lld tempty %lld issue %lld | prod: wait %lld work %lld | epi: wait %lld work %lld\n",
                rows, kp, n, p.bn, p.astat, p.stages, p.gather, pool, (double)total / grid, ms * 1e3, h[1], h[2], h[3], h[4], h[5], h[6], h[7],
                h[8], h[9]);
        memset(h, 0, sizeof(h));
        cudaMemcpyToSymbol(tc_prof, h, sizeof(h));
        cudaEventDestroy(pe0); cudaEventDestroy(pe1);
    }
#endif
    SSD3D_LAUNCH_CHECK("linear_tc_kernel");
}

static int hoist_expand_split_launch(int b, int n, int n1, int m, int nsample, const float *xyz, const float *z, int ldz,
                                     const float *wx, const float *new_xyz, const int *idx, const int *units, void *hi,
                                     void *lo, int kp, ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(b >= 0 && n > 0 && m >= 0 && n1 > 0 && nsample > 0 && ldz >= n1, "hoist_expand_split: bad shape");
    SSD3D_REQUIRE(kp % 16 == 0 && kp >= n1 && kp <= 4096, "hoist_expand_split: kp=%d must be a multiple of 16 in [n1, 4096]", kp);
    SSD3D_REQUIRE(ldz % 4 == 0 && (reinterpret_cast<uintptr_t>(z) & 15u) == 0, "hoist_expand_split: z rows must be 16-byte aligned");
    SSD3D_REQUIRE(xyz && z && wx && new_xyz && idx && hi && lo, "hoist_expand_split: null pointer");
    SSD3D_REQUIRE(((reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15u) == 0, "hoist_expand_split: outputs must be 16-byte aligned");
    const long rows = (long)b * m * nsample;
    if (rows == 0) return 0;
    const long blocks_want = (rows + 7) / 8;
    const int blocks = (int)(blocks_want < (long)kNumSMs * 32 ? blocks_want : (long)kNumSMs * 32);
    hoist_expand_split_kernel<<<blocks, 256, (size_t)3 * kp * sizeof(float), (cudaStream_t)stream>>>(
        rows, n, n1, m, nsample, xyz, z, ldz, wx, new_xyz, idx, units, (__nv_bfloat16 *)hi, (__nv_bfloat16 *)lo, kp);
    SSD3D_LAUNCH_CHECK("hoist_expand_split_kernel");
}

extern "C" int ssd3d_hoist_expand_split(int b, int n, int n1, int m, int nsample, const float *xyz, const float *z, int ldz,
                                        const float *wx, const float *new_xyz, const int *idx, void *hi, void *lo, int kp,
                                        ssd3d_stream_t stream)
{
    return hoist_expand_split_launch(b, n, n1, m, nsample, xyz, z, ldz, wx, new_xyz, idx, nullptr, hi, lo, kp, stream);
}

extern "C" int ssd3d_hoist_expand_split_units(int b, int n, int n1, int m, int nsample, const float *xyz, const float *z,
                                              int ldz, const float *wx, const float *new_xyz, const int *idx,
                                              const int *units, void *hi, void *lo, int kp, ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(units && nsample % 8 == 0 && nsample <= 128, "hoist_expand_split_units: needs a unit list and nsample a multiple of 8, <= 128");
    return hoist_expand_split_launch(b, n, n1, m, nsample, xyz, z, ldz, wx, new_xyz, idx, units, hi, lo, kp, stream);
}

// Unit-list forms of ssd3d_linear_tc / ssd3d_linear_tc_hoisted (TcParams::units): the matrix has units[0] * 8 rows (`rows` /
// b*m*nsample is the capacity of the buffers).  unit_pool != 0: each 8-row unit is max-pooled and combined into
// out_f32[group] by atomicMax (ReLU required, out_f32 zero-filled by the caller, no split output).
extern "C" int ssd3d_linear_tc_units(long rows, int kp, int n, const void *a_hi, const void *a_lo, const void *b_hi,
                                     const void *b_lo, const float *scale, const float *shift, int relu, const int *units,
                                     int unit_pool, float *out_f32, int ld_f32, void *out_hi, void *out_lo, int ld_split,
                                     ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(units, "linear_tc_units: null unit list");
    return linear_tc_launch(rows, kp, n, a_hi, a_lo, nullptr, b_hi, b_lo, scale, shift, relu, 1, nullptr, out_f32, ld_f32,
                            out_hi, out_lo, ld_split, (cudaStream_t)stream, units, unit_pool);
}

extern "C" int ssd3d_linear_tc_hoisted_units(int b, int n, int n1, int m, int nsample, const float *xyz, const float *z,
                                             int ldz, const float *wx, const float *new_xyz, const int *idx,
                                             const int *units, int nout, const void *b_hi, const void *b_lo,
                                             const float *scale, const float *shift, int relu, int unit_pool, float *out_f32,
                                             int ld_f32, void *out_hi, void *out_lo, int ld_split, ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(b >= 0 && n > 0 && m >= 0 && n1 > 0 && nsample > 0 && ldz >= n1, "linear_tc_hoisted_units: bad shape");
    SSD3D_REQUIRE(xyz && new_xyz && idx && z && wx && units, "linear_tc_hoisted_units: null pointer");
    SSD3D_REQUIRE(nsample % 8 == 0 && nsample <= 128, "linear_tc_hoisted_units: nsample=%d must be a multiple of 8, <= 128", nsample);
    TcGather g = {b, n, n1, m, nsample, xyz, z, new_xyz, idx, ldz, wx};
    const int kp = (n1 + 15) / 16 * 16;
    return linear_tc_launch((long)b * m * nsample, kp, nout, nullptr, nullptr, &g, b_hi, b_lo, scale, shift, relu, 1, nullptr,
                            out_f32, ld_f32, out_hi, out_lo, ld_split, (cudaStream_t)stream, units, unit_pool);
}

extern "C" int ssd3d_linear_tc(long rows, int kp, int n, const void *a_hi, const void *a_lo, const void *b_hi,
                               const void *b_lo, const float *scale, const float *shift, int relu, int pool,
                               const int *rowmask, float *out_f32, int ld_f32, void *out_hi, void *out_lo, int ld_split,
                               ssd3d_stream_t stream)
{
    return linear_tc_launch(rows, kp, n, a_hi, a_lo, nullptr, b_hi, b_lo, scale, shift, relu, pool, rowmask, out_f32, ld_f32,
                            out_hi, out_lo, ld_split, (cudaStream_t)stream);
}

// First layer of an SA scale with the gather fused into the operand load: rows = b*m*nsample, K = c+3 (kp = round16).
extern "C" int ssd3d_linear_tc_gather(int b, int n, int c, int m, int nsample, const float *xyz, const float *points,
                                      const float *new_xyz, const int *idx, int nout, const void *b_hi, const void *b_lo,
                                      const float *scale, const float *shift, int relu, int pool, const int *rowmask,
                                      float *out_f32, int ld_f32, void *out_hi, void *out_lo, int ld_split,
                                      ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(b >= 0 && n > 0 && m >= 0 && c >= 0 && nsample > 0, "linear_tc_gather: bad shape");
    SSD3D_REQUIRE(xyz && new_xyz && idx && (points || c == 0), "linear_tc_gather: null pointer");
    TcGather g = {b, n, c, m, nsample, xyz, points, new_xyz, idx, 0, nullptr};
    const int kp = (c + 3 + 15) / 16 * 16;
    return linear_tc_launch((long)b * m * nsample, kp, nout, nullptr, nullptr, &g, b_hi, b_lo, scale, shift, relu, pool,
                            rowmask, out_f32, ld_f32, out_hi, out_lo, ld_split, (cudaStream_t)stream);
}

// Second layer of an SA scale fed by the HOISTED first layer (see TcParams): z[b,n,ldz] holds (f . Wf) * s1 + t1 per
// point (this scale's n1 columns start at z), wx = Wx * s1 as [3][n1]; the operand row of grouped element (i,j) is
// relu(z[idx] + (xyz[idx] - new_xyz[i]) . wx), built by the producer warps.  K of this layer = n1 (kp = round16).
extern "C" int ssd3d_linear_tc_hoisted(int b, int n, int n1, int m, int nsample, const float *xyz, const float *z, int ldz,
                                       const float *wx, const float *new_xyz, const int *idx, int nout, const void *b_hi,
                                       const void *b_lo, const float *scale, const float *shift, int relu, int pool,
                                       const int *rowmask, float *out_f32, int ld_f32, void *out_hi, void *out_lo,
                                       int ld_split, ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(b >= 0 && n > 0 && m >= 0 && n1 > 0 && nsample > 0 && ldz >= n1, "linear_tc_hoisted: bad shape");
    SSD3D_REQUIRE(xyz && new_xyz && idx && z && wx, "linear_tc_hoisted: null pointer");
    TcGather g = {b, n, n1, m, nsample, xyz, z, new_xyz, idx, ldz, wx};
    const int kp = (n1 + 15) / 16 * 16;
    return linear_tc_launch((long)b * m * nsample, kp, nout, nullptr, nullptr, &g, b_hi, b_lo, scale, shift, relu, pool,
                            rowmask, out_f32, ld_f32, out_hi, out_lo, ld_split, (cudaStream_t)stream);
}

extern "C" int ssd3d_split_rows(long rows, int c, const float *x, int ldx, void *hi, void *lo, int kp, ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(rows >= 0 && c > 0 && ldx >= c && kp >= c && kp % 8 == 0, "split_rows: bad shape rows=%ld c=%d ldx=%d kp=%d", rows, c, ldx, kp);
    SSD3D_REQUIRE(x && hi && lo, "split_rows: null pointer");
    const long total = rows * kp;
    if (total == 0) return 0;
    const long nchunks = total / 8;
    if (nchunks < (1L << 31) && ((reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15u) == 0) {
        const int vec = (ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15u) == 0) ? 1 : 0;
        const long want = (nchunks + 255) / 256;
        const int blocks = (int)(want < (long)kNumSMs * 16 ? want : (long)kNumSMs * 16);
        split_rows_v8_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((unsigned)nchunks, c, x, ldx, (__nv_bfloat16 *)hi,
                                                                       (__nv_bfloat16 *)lo, kp, vec);
        SSD3D_LAUNCH_CHECK("split_rows_v8_kernel");
    }
    const long want = (total + 255) / 256;
    const int blocks = (int)(want < (long)kNumSMs * 16 ? want : (long)kNumSMs * 16);
    split_rows_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rows, c, x, ldx, (__nv_bfloat16 *)hi, (__nv_bfloat16 *)lo, kp);
    SSD3D_LAUNCH_CHECK("split_rows_kernel");
}

extern "C" int ssd3d_group_concat_split(int b, int n, int c, int m, int nsample, const float *xyz, const float *points,
                                        const float *new_xyz, const int *idx, void *hi, void *lo, int kp,
                                        ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(b >= 0 && n > 0 && m >= 0 && c >= 0 && nsample > 0, "group_concat_split: bad shape");
    SSD3D_REQUIRE(kp >= c + 3 && kp % 8 == 0, "group_concat_split: kp=%d must be >= c+3=%d and a multiple of 8", kp, c + 3);
    SSD3D_REQUIRE(xyz && new_xyz && idx && hi && lo && (points || c == 0), "group_concat_split: null pointer");
    const long rows = (long)b * m * nsample;
    if (rows == 0) return 0;
    const long want = (rows + 31) / 32;                             // 8 warps x 4 rows per block
    const int blocks = (int)(want < (long)kNumSMs * 32 ? want : (long)kNumSMs * 32);
    const int vec4 = (c >= 4 && c % 4 == 0 && (reinterpret_cast<uintptr_t>(points) & 15u) == 0) ? 1 : 0;
    const size_t gsm = (size_t)8 * 4 * 2 * kp * sizeof(__nv_bfloat16);
    SSD3D_REQUIRE(gsm <= 96 * 1024, "group_concat_split: kp=%d too wide", kp);
    const cudaError_t ea = cudaFuncSetAttribute((const void *)group_concat_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm);
    if (ea != cudaSuccess) return cuda_status(ea, "group_concat_split shared-memory opt-in");
    group_concat_split_kernel<<<blocks, 256, gsm, (cudaStream_t)stream>>>(rows, n, c, m, nsample, xyz, points, new_xyz, idx,
                                                                          (__nv_bfloat16 *)hi, (__nv_bfloat16 *)lo, kp, vec4);
    SSD3D_LAUNCH_CHECK("group_concat_split_kernel");
}
