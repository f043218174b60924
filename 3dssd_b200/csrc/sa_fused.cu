// sa_fused.cu -- one SA scale in ONE kernel: gather + concat + (conv+BN+ReLU) x L + max-pool + mask, tcgen05.
//
// Fuses lib/utils/layers_util.py:157-180 of the reference (idx masking, 2x group_point, centre subtraction, concat,
// the conv2d/bias/BN/ReLU stack, reduce_max, mask multiply -- ~25 TF kernels per scale, each streaming [B,M,K,C]
// through HBM) for the layers whose weights fit in shared memory (3DSSD layer1/layer2: 93% of the grouped rows).
// Nothing but the neighbour indices, the gathered source rows (L2-resident) and the pooled [B,M,C3] result touches
// global memory; activations go TMEM -> registers -> shared memory (already split in bf16 hi/lo and already in the
// 128B-swizzled K-major layout the next layer's UMMA descriptor expects).
//
// Per CTA: S "slots" of 128*WG threads (a slot works on one 128-row tile = 128/K neighbour groups; its WG warpgroups
// split the 16-byte chunks of the gather and the 32-column chunks of every epilogue):
//   weights of all layers (hi+lo images, pre-swizzled on the host) are bulk-copied to shared memory once and shared
//   by the slots; each slot owns ONE operand buffer, one TMEM accumulator and one mbarrier and loops over tiles:
//   gather+split -> [fence.proxy.async] -> layer-0 MMAs (one thread) -> epilogue (tcgen05.ld, scale/shift/ReLU,
//   split) written IN PLACE over the operand the finished MMAs no longer need -> ... -> last layer: max-pool.
// Small stacks (layer1: ~30 KiB) run S=1 with up to 6 CTAs per SM; stacks whose weights fill most of shared memory
// (layer2: 68-92 KiB) run one CTA per SM with S=2..3 slots, so gather / MMA / epilogue phases still overlap.
// Hoisted mode (SfParams::hoist): the scale's first conv has been moved to a per-point table z (include/ssd3d.h,
// ssd3d_sa_mlp_fused_hoisted); the gather then builds relu(z[idx] + (xyz[idx] - centre) . Wx') and the stack starts at
// the second conv.
// Unit-list mode (SfParams::units, round 2): a neighbour list repeats its first hit beyond pts_cnt
// (grouping/tf_grouping_g.cu:245-248) and the copies cannot change the max-pool, so a tile is made of 16 listed 8-row units
// (the ball query lists ceil(cnt / 8) units per non-empty group) instead of 128 consecutive rows; each unit is pooled by the
// shuffle butterfly and the units of a group meet through atomicMax on the non-negative fp32 result, which the caller
// zero-fills (= the cnt == 0 mask of layers_util.py:180).  Same bits as the dense schedule, 4-8x fewer rows on KITTI-like
// clouds (DESIGN.md section 3.4).
//
// Precision: the bf16 hi/lo split and 3-MMA scheme of tc.cuh, as in mlp_tc.cu.
#include <cstdio>
#include <cstring>

#include "common.cuh"
#include "pool.cuh"
#include "tc.cuh"

namespace ssd3d {

constexpr int SF_THREADS = 128;
constexpr int SF_MAX_LAYERS = 3;

struct SfParams {
    int n, c, m, ns;                 // points per scene, feature channels, queries per scene, neighbours per query
    long rows;                       // b*m*ns
    int tiles;
    const float *xyz, *points, *new_xyz;
    const int *idx, *cnt;
    // unit list (ssd3d_query_ball_point_multi_ws): when set, a tile is 16 UNITS of 8 rows -- units[1 + u] = (group << 4) | j
    // names rows 8j..8j+7 of neighbour list `group` -- instead of 128 consecutive rows, units[0] is their number, and the
    // pooled result is combined across the units of a group with atomicMax on the (non-negative) fp32 output
    const int *units;
    // hoisted first conv (see ssd3d_linear_tc_hoisted in include/ssd3d.h): `points` is the per-point table z (row pitch
    // ldz, c = its width n1), the operand row is relu(z[idx] + (xyz[idx] - new_xyz) . wx) with wx = [3][c], and the
    // stack starts at the scale's SECOND conv (K = c, no xyz columns appended)
    int hoist, ldz;
    const float *wx;
    int nl;
    int kp[SF_MAX_LAYERS];           // K of layer l padded to 16
    int npad[SF_MAX_LAYERS];         // N of layer l padded to 16
    int nout[SF_MAX_LAYERS];         // true N
    uint32_t w_off[SF_MAX_LAYERS];   // byte offset of the layer's weight image in the packed blob / shared memory
    uint32_t w_half[SF_MAX_LAYERS];  // bytes of the hi half (lo follows)
    uint32_t ss_off[SF_MAX_LAYERS];  // float offset of the layer's scale (shift follows at +npad) in the ss blob
    uint32_t w_total, ss_total;      // bytes / floats
    const uint8_t *w_blob;
    const float *ss_blob;
    int sspad[SF_MAX_LAYERS];        // npad rounded up to 32 (scale/shift arrays are zero padded to this)
    int nfull[SF_MAX_LAYERS];        // layer l's K = nfull 64-wide k-blocks (128-byte rows) + one tail block
    int rbt[SF_MAX_LAYERS];          // bytes per row of the tail block: 0 (none), 32 (16 wide), 64 (32), 128 (48)
    uint32_t abuf_bytes;             // operand buffer of one slot
    uint32_t tmem_cols;              // accumulator columns of one slot
    uint32_t tmem_alloc;             // power of two >= slots * tmem_cols
    float *out_f32; int ld_f32;
    __nv_bfloat16 *out_hi, *out_lo; int ld_split;
    int pool_first;                  // caller guarantees scale >= 0 in the LAST layer: pool raw accumulators, affine after
};

// Where row r of a 128-row operand tile lives.  An A buffer is laid out as k-blocks of { hi tile | lo tile }
// (128 rows x rb bytes each), each tile in the canonical K-major swizzled layout of span rb: 16-byte chunk j of
// row r sits at chunk j ^ ((r >> log2(128/rb)) & (rb/16 - 1)).  The first nfull blocks are 64 wide (rb = 128),
// the tail block is rbt bytes wide.  Built once per (thread, layer); chunk() is then a handful of integer ops.
struct SfRowMap {
    uint32_t row_f, xor_f;            // full blocks: byte offset of the row inside a tile, swizzle mask
    uint32_t base_t, row_t, xor_t;    // tail block: byte offset of the block, of the row, swizzle mask
    uint32_t lo_t;                    // hi -> lo tile distance in the tail block (full blocks: 16 KiB)
    int full8;                        // nfull * 8: first 16-byte chunk index of the tail block
    __device__ __forceinline__ SfRowMap(int r, int nfull, int rbt)
    {
        row_f = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u;
        xor_f = (uint32_t)(r & 7);
        const int sh = rbt == 128 ? 0 : (rbt == 64 ? 1 : 2);
        base_t = (uint32_t)nfull * (2u * 128u * 128u);
        row_t = (uint32_t)(r >> 3) * (uint32_t)(8 * rbt) + (uint32_t)(r & 7) * (uint32_t)rbt;
        xor_t = (uint32_t)((r >> sh) & ((rbt >> 4) - 1));
        lo_t = 128u * (uint32_t)rbt;
        full8 = nfull * 8;
    }
    // byte offset of the 16-byte chunk holding columns [8*c16g, 8*c16g+8); *lo_off = distance to the lo tile
    __device__ __forceinline__ uint32_t chunk(int c16g, uint32_t *lo_off) const
    {
        if (c16g < full8) {
            *lo_off = 128u * 128u;
            return (uint32_t)(c16g >> 3) * (2u * 128u * 128u) + row_f + ((((uint32_t)c16g & 7u) ^ xor_f) << 4);
        }
        *lo_off = lo_t;
        return base_t + row_t + (((uint32_t)(c16g - full8) ^ xor_t) << 4);
    }
};

// ---- shape policies -------------------------------------------------------------------------------------------------
// The kernel body is written once against a policy C that answers every shape question (layer count, padded K / N of a
// layer, block layout, blob offsets, neighbours per group).  SfDyn reads the answers from the parameter block at run
// time (any stack the planner accepts); SfStat<...> answers at COMPILE time for the stacks of the shipped 3DSSD
// configuration, so that after unrolling the layer loop every address computation, chunk bound and pooling width is a
// literal: profiling the dynamic kernel showed ~50% of its issued instructions to be integer / branch / uniform-register
// bookkeeping of exactly these questions (profiles/r02_fused_instruction_mix.txt).
__host__ __device__ constexpr int sf_r16(int x) { return (x + 15) / 16 * 16; }
// Operand layout of a layer with padded K = kp: kp / 64 full 64-wide k-blocks of 128-byte rows + a tail block whose rows
// are sf_rbt_of(kp) = 32 / 64 / 128 bytes for a remainder of 16 / 32 / 48 columns (must match params._k_blocks).
// An operand buffer holds { hi | lo } tiles of 128 rows per block, 1 KiB granular.
__host__ __device__ constexpr int sf_rbt_of(int kp) { return kp % 64 == 0 ? 0 : (kp % 64 <= 16 ? 32 : (kp % 64 <= 32 ? 64 : 128)); }
__host__ __device__ constexpr uint32_t sf_abuf_of(int kp)
{
    return (uint32_t)(((kp / 64) * 2 * 128 * 128 + 2 * 128 * sf_rbt_of(kp) + 1023) / 1024 * 1024);
}

struct SfDyn {
    static constexpr bool kStatic = false;
    const SfParams &p;
    __device__ __forceinline__ explicit SfDyn(const SfParams &p_) : p(p_) {}
    __device__ __forceinline__ int nl() const { return p.nl; }
    __device__ __forceinline__ int ns() const { return p.ns; }
    __device__ __forceinline__ int c() const { return p.c; }
    __device__ __forceinline__ bool hoist() const { return p.hoist != 0; }
    __device__ __forceinline__ int kp(int l) const { return p.kp[l]; }
    __device__ __forceinline__ int npad(int l) const { return p.npad[l]; }
    __device__ __forceinline__ int nout(int l) const { return p.nout[l]; }
    __device__ __forceinline__ int nfull(int l) const { return p.nfull[l]; }
    __device__ __forceinline__ int rbt(int l) const { return p.rbt[l]; }
    __device__ __forceinline__ uint32_t w_off(int l) const { return p.w_off[l]; }
    __device__ __forceinline__ uint32_t w_half(int l) const { return p.w_half[l]; }
    __device__ __forceinline__ uint32_t ss_off(int l) const { return p.ss_off[l]; }
    __device__ __forceinline__ int sspad(int l) const { return p.sspad[l]; }
    __device__ __forceinline__ uint32_t w_total() const { return p.w_total; }
    __device__ __forceinline__ uint32_t ss_total() const { return p.ss_total; }
    __device__ __forceinline__ uint32_t abuf_bytes() const { return p.abuf_bytes; }
    __device__ __forceinline__ uint32_t tmem_cols() const { return p.tmem_cols; }
};

// Hoisted stacks of two convs (the shipped configuration): operand width K0 = n1 of the hoisted first conv, then
// K0 -> N0 -> N1, NS neighbours per group.
template <int K0, int N0, int N1, int NS>
struct SfStat {
    static constexpr bool kStatic = true;
    __device__ __forceinline__ explicit SfStat(const SfParams &) {}
    static constexpr int KP0 = sf_r16(K0), NP0 = sf_r16(N0), NP1 = sf_r16(N1);
    __device__ __forceinline__ constexpr int nl() const { return 2; }
    __device__ __forceinline__ constexpr int ns() const { return NS; }
    __device__ __forceinline__ constexpr int c() const { return K0; }
    __device__ __forceinline__ constexpr bool hoist() const { return true; }
    __device__ __forceinline__ constexpr int kp(int l) const { return l == 0 ? KP0 : NP0; }
    __device__ __forceinline__ constexpr int npad(int l) const { return l == 0 ? NP0 : NP1; }
    __device__ __forceinline__ constexpr int nout(int l) const { return l == 0 ? N0 : N1; }
    __device__ __forceinline__ constexpr int nfull(int l) const { return kp(l) / 64; }
    __device__ __forceinline__ constexpr int rbt(int l) const { return sf_rbt_of(kp(l)); }
    __device__ __forceinline__ constexpr uint32_t w_half(int l) const { return (uint32_t)(npad(l) * (nfull(l) * 128 + rbt(l))); }
    __device__ __forceinline__ constexpr uint32_t w_off(int l) const { return l == 0 ? 0u : 2u * w_half(0); }
    __device__ __forceinline__ constexpr int sspad(int l) const { return (npad(l) + 31) / 32 * 32; }
    __device__ __forceinline__ constexpr uint32_t ss_off(int l) const { return l == 0 ? 0u : 2u * (uint32_t)sspad(0); }
    __device__ __forceinline__ constexpr uint32_t w_total() const { return 2u * w_half(0) + 2u * w_half(1); }
    __device__ __forceinline__ constexpr uint32_t ss_total() const { return 2u * (uint32_t)sspad(0) + 2u * (uint32_t)sspad(1); }
    __device__ __forceinline__ constexpr uint32_t abuf_bytes() const { return sf_abuf_of(KP0) > sf_abuf_of(NP0) ? sf_abuf_of(KP0) : sf_abuf_of(NP0); }
    __device__ __forceinline__ constexpr uint32_t tmem_cols() const
    {
        return (NP0 > NP1 ? NP0 : NP1) <= 32 ? 32u : ((NP0 > NP1 ? NP0 : NP1) <= 64 ? 64u : ((NP0 > NP1 ? NP0 : NP1) <= 128 ? 128u : 256u));
    }
};

#ifdef SF_PROFILE
__device__ long long sf_prof[16];
#define SF_T(i) do { if (prof_on) { const long long t_ = clock64(); sf_prof[i] += t_ - t_prev; t_prev = t_; } } while (0)
#else
#define SF_T(i) do { } while (0)
#endif

// SLOTS tiles in flight per CTA, WG warpgroups (128 threads) working on each: the warpgroups of a slot split the
// 16-byte chunks of the gather and the 32-column chunks of every epilogue between them.  C: shape policy (above).
template <class C, int SLOTS, int WG>
__global__ void __launch_bounds__(SF_THREADS * SLOTS * WG, SLOTS * WG == 1 ? 6 : 1)
sa_fused_kernel(const SfParams p)
{
    const C cfg(p);
    // pointers inside the by-value parameter struct carry no address space: tell the compiler they are global
    __builtin_assume(__isGlobal(p.xyz)); __builtin_assume(__isGlobal(p.new_xyz)); __builtin_assume(__isGlobal(p.idx));
    __builtin_assume(p.points == nullptr || __isGlobal(p.points)); __builtin_assume(p.cnt == nullptr || __isGlobal(p.cnt));
    __builtin_assume(__isGlobal(p.w_blob)); __builtin_assume(__isGlobal(p.ss_blob));
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1 KiB alignment by pointer arithmetic on the __shared__ array (an integer round-trip would demote every access
    // through these pointers to generic LD/ST with 64-bit address math)
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *wsm = smem + (size_t)SLOTS * cfg.abuf_bytes();  // weight images (1024-aligned: buffers are multiples of 1 KiB)
    float *ss = reinterpret_cast<float *>(wsm + cfg.w_total());
    float *wxs = ss + cfg.ss_total();                    // [3][kp0] hoisted mode: Wx * s1, zero beyond c

    __shared__ unsigned long long w_bar, mma_bar[SLOTS];
    __shared__ uint32_t tmem_base_smem;
    __shared__ float xs_all[SLOTS * WG][4 * 32];

    constexpr int NT = SF_THREADS * SLOTS * WG, ST = SF_THREADS * WG;     // threads per CTA / per slot
    constexpr int U = WG == 1 ? 4 : 3;                   // gather chunks in flight per thread
    const int tid = threadIdx.x, lane = tid & 31, q = (tid >> 5) & 3;
    const int slot = tid / ST, wg = (tid >> 7) % WG;
    const int r = tid & 127;                             // row of the slot's tile this thread works on
    // the slot's first warp issues the MMAs; its index is made provably warp-uniform (shfl) so that descriptors are
    // computed on the uniform datapath and tcgen05.mma takes them without a per-operand R2UR "waterfall" loop
    const int slot_u = __shfl_sync(0xffffffffu, slot, 0);
    const bool issuer_warp = __shfl_sync(0xffffffffu, (tid % ST) >> 5, 0) == 0;
    const int slot_bar = 1 + slot, wg_bar = 1 + SLOTS + slot * WG + wg;
    uint8_t *buf = smem + (size_t)slot * cfg.abuf_bytes();   // the slot's operand buffer (every layer, in place)
    float *xs = xs_all[slot * WG + wg];
    const int kp0 = cfg.kp(0);

    if (tid == 0) {
        mbar_init(smem_u32(&w_bar), 1);
#pragma unroll
        for (int i = 0; i < SLOTS; i++) mbar_init(smem_u32(&mma_bar[i]), 1);
        fence_mbar_init_cluster();
        mbar_arrive_expect_tx(smem_u32(&w_bar), cfg.w_total());
        bulk_g2s(smem_u32(wsm), p.w_blob, cfg.w_total(), smem_u32(&w_bar));
    }
    if (tid < 32) tmem_alloc(&tmem_base_smem, p.tmem_alloc);
    for (uint32_t i = tid; i < cfg.ss_total(); i += NT) ss[i] = __ldg(p.ss_blob + i);
    if (cfg.hoist())
        for (int i = tid; i < 3 * kp0; i += NT) {
            const int a3 = i / kp0, k = i - a3 * kp0;
            wxs[i] = k < cfg.c() ? __ldg(p.wx + a3 * cfg.c() + k) : 0.0f;
        }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_smem + (uint32_t)slot * cfg.tmem_cols();
    const uint32_t bar = smem_u32(&mma_bar[slot]);
    mbar_wait_cta(smem_u32(&w_bar), 0);                  // weights landed (async proxy writes, read by UMMA only)

#ifdef SF_PROFILE
    const bool prof_on = blockIdx.x == 0 && (tid % ST) == 0 && slot == 0;
    long long t_prev = clock64();
#endif
    uint32_t mma_phase = 0;
    const int k0 = cfg.hoist() ? cfg.c() : cfg.c() + 3;  // valid operand columns
    const int pitch = cfg.hoist() ? p.ldz : cfg.c();
    const bool vec = (cfg.c() & 3) == 0 && (pitch & 3) == 0; // source rows are 16-byte aligned: float4 gathers

    const int tile0 = blockIdx.x * SLOTS + slot, tstep = gridDim.x * SLOTS;
    const int *units = p.units;
    __builtin_assume(units == nullptr || __isGlobal(units));
    const bool compact = units != nullptr;
    const int nunits = compact ? __ldg(units) : 0;
    const int tiles = compact ? (nunits + 15) >> 4 : p.tiles;
    // neighbour index (and, in unit-list mode, unit descriptor) of this thread's row, fetched one tile ahead
    // (rows < 2^31: checked by the launcher)
    auto fetch = [&](int t, int &desc, int &a) {
        desc = -1; a = 0;
        if (t >= tiles) return;
        if (compact) {
            const int ui = t * 16 + (r >> 3);
            if (ui < nunits) {
                desc = __ldg(units + 1 + ui);
                a = __ldg(p.idx + (size_t)(desc >> 4) * (uint32_t)cfg.ns() + (uint32_t)(((desc & 15) << 3) + (r & 7)));
            }
        } else if ((long)t * 128 + r < p.rows) {
            desc = 0;
            a = __ldg(p.idx + (size_t)t * 128u + r);
        }
    };
    int d_next, a_next;
    fetch(tile0, d_next, a_next);
    int my_group = 0;                                                  // unit-list mode: the group this thread's row belongs to
    bool my_ok = false;
    for (int tile = tile0; tile < tiles; tile += tstep) {
        // ---- gather + centre-subtract + concat + split -> buf (layers_util.py:157-165)
        {
            const uint32_t row = (uint32_t)tile * 128u + (uint32_t)r;
            const bool ok = d_next >= 0;
            const uint32_t qi = !ok ? 0u : (compact ? (uint32_t)(d_next >> 4) : row / (uint32_t)cfg.ns());    // == scene*m + query
            const uint32_t scene = qi / (uint32_t)p.m;
            const int a = a_next;
            my_group = (int)qi; my_ok = ok;
            fetch(tile + tstep, d_next, a_next);
            const float *src_f = p.points + ((size_t)scene * p.n + a) * pitch;
            const float *src_x = p.xyz + ((size_t)scene * p.n + a) * 3;
            const float *ctr = p.new_xyz + (size_t)qi * 3;
            const int nchunk = kp0 >> 3;
            const SfRowMap map0(r, cfg.nfull(0), cfg.rbt(0));
            float dx = 0.0f, dy = 0.0f, dz = 0.0f;
            if (cfg.hoist() && ok) {
                dx = __ldg(src_x) - __ldg(ctr); dy = __ldg(src_x + 1) - __ldg(ctr + 1); dz = __ldg(src_x + 2) - __ldg(ctr + 2);
            }
#pragma unroll (C::kStatic ? 4 : 1)
            for (int cg0 = wg * U; cg0 < nchunk; cg0 += WG * U) {     // U chunks of 8 columns in flight per thread
                float f[U][8];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int kb = (cg0 + u) * 8;
                    if (vec && ok && kb + 8 <= cfg.c()) {
                        const float4 lo4 = __ldg(reinterpret_cast<const float4 *>(src_f + kb));
                        const float4 hi4 = __ldg(reinterpret_cast<const float4 *>(src_f + kb + 4));
                        f[u][0] = lo4.x; f[u][1] = lo4.y; f[u][2] = lo4.z; f[u][3] = lo4.w;
                        f[u][4] = hi4.x; f[u][5] = hi4.y; f[u][6] = hi4.z; f[u][7] = hi4.w;
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; e++) {
                            const int k = kb + e;
                            float val = 0.0f;
                            if (ok) {
                                if (k < cfg.c()) val = __ldg(src_f + k);
                                else if (k < k0) val = __ldg(src_x + (k - cfg.c())) - __ldg(ctr + (k - cfg.c()));   // never in hoisted mode
                            }
                            f[u][e] = val;
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    if (cg0 + u >= nchunk) break;
                    if (cfg.hoist()) hoist_relu8(f[u], dx, dy, dz, wxs + (cg0 + u) * 8, kp0);   // padded columns and rows stay 0
                    // spelled out rather than split8_store(): with the chunk offset computed first, the single-slot
                    // run-time-shape kernel spills 20 more bytes
                    uint32_t hw[4], lw[4], lo_off;
#pragma unroll
                    for (int t = 0; t < 4; t++) split_pair(f[u][2 * t], f[u][2 * t + 1], hw[t], lw[t]);
                    const uint32_t off = map0.chunk(cg0 + u, &lo_off);
                    *reinterpret_cast<uint4 *>(buf + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                    *reinterpret_cast<uint4 *>(buf + off + lo_off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
                }
            }
        }
        SF_T(0);                                                       // gather
#pragma unroll (C::kStatic ? SF_MAX_LAYERS : 1)
        for (int l = 0; l < cfg.nl(); l++) {
            // operand written with ordinary stores -> make it visible to the tensor-core (async) proxy
            fence_async_smem();
            tc_fence_before();
            bar_sync(slot_bar, ST);
            SF_T(1 + 4 * l);                                           // barrier
            if (issuer_warp) {
                tc_fence_after();
                // one MMA per k-step covers the whole layer width: a tcgen05.mma costs ~N/2 cycles plus a fixed
                // per-instruction part, so narrower MMAs only add overhead (measured in round 1)
                const uint32_t idesc = umma_idesc_bf16(cfg.npad(l));
                const uint32_t tmem_u = tmem_base_smem + (uint32_t)slot_u * cfg.tmem_cols();
                const uint32_t abase = smem_u32(smem) + (uint32_t)slot_u * cfg.abuf_bytes();
                const uint32_t wbase = smem_u32(wsm) + cfg.w_off(l);
                const int nfull = cfg.nfull(l), rbt = cfg.rbt(l);
                uint32_t acc = 0u;
                // descriptors advance by (bytes >> 4) in their address field; shared memory < 256 KiB: no carry out of it
#pragma unroll (C::kStatic ? 4 : 1)
                for (int kb = 0; kb < nfull; kb++) {
                    const uint64_t a_hi = umma_desc(abase + (uint32_t)kb * (2u * 128u * 128u), 128);
                    const uint64_t b_hi = umma_desc(wbase + (uint32_t)kb * ((uint32_t)cfg.npad(l) * 128u), 128);
                    const uint64_t a_lo = a_hi + ((128u * 128u) >> 4), b_lo = b_hi + (cfg.w_half(l) >> 4);
#pragma unroll
                    for (int kin = 0; kin < 4; kin++) {
                        if (elect_one()) umma_bf16x3(tmem_u, a_hi + 2 * kin, a_lo + 2 * kin, b_hi + 2 * kin, b_lo + 2 * kin, idesc, acc);
                        acc = 1u;
                    }
                }
                if (rbt) {
                    const uint64_t a_hi = umma_desc(abase + (uint32_t)nfull * (2u * 128u * 128u), rbt);
                    const uint64_t b_hi = umma_desc(wbase + (uint32_t)nfull * ((uint32_t)cfg.npad(l) * 128u), rbt);
                    const uint64_t a_lo = a_hi + ((128u * (uint32_t)rbt) >> 4), b_lo = b_hi + (cfg.w_half(l) >> 4);
                    const int nt = rbt == 128 ? 3 : (rbt >> 5);              // 16-wide k-steps of the tail block
#pragma unroll (C::kStatic ? 3 : 1)
                    for (int kin = 0; kin < nt; kin++) {
                        if (elect_one()) umma_bf16x3(tmem_u, a_hi + 2 * kin, a_lo + 2 * kin, b_hi + 2 * kin, b_lo + 2 * kin, idesc, acc);
                        acc = 1u;
                    }
                }
                if (elect_one()) umma_commit(smem_u32(&mma_bar[slot_u]));
                __syncwarp();
                SF_T(2 + 4 * l);                                       // MMA issue
                // ONE warp of the slot polls the mbarrier; the others sleep at the slot's named barrier (a hardware
                // barrier costs no issue slots -- the all-warps poll loop was a quarter of the kernel's instructions)
                mbar_wait_cta(bar, mma_phase);                       // MMAs done: accumulator ready, operand buffer free
                tc_fence_before();
            }
            bar_sync(slot_bar, ST);
            mma_phase ^= 1u;
            SF_T(3 + 4 * l);                                           // MMA wait
            tc_fence_after();
            // ---- epilogue of layer l
            const float *sc = ss + cfg.ss_off(l);
            const float *sh = sc + cfg.sspad(l);
            const bool last = l == cfg.nl() - 1;
            const bool pool_first = last && p.pool_first;              // last layer with scale >= 0: pool raw accumulators
            const SfRowMap mapn(r, last ? 0 : cfg.nfull(l + 1), last ? 32 : cfg.rbt(l + 1));
            const int nchunks = (cfg.npad(l) + 31) / 32;
#pragma unroll (C::kStatic ? 4 : 1)
            for (int ci = wg; ci < nchunks; ci += WG) {
                const int c0 = ci * 32;
                uint32_t rr[32];
                tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, rr);
                float v[32];
                if (pool_first) {
#pragma unroll
                    for (int j = 0; j < 32; j++) v[j] = __uint_as_float(rr[j]);
                } else {
#pragma unroll
                    for (int j4 = 0; j4 < 32; j4 += 4) {              // scale/shift are zero-padded to 32-column chunks
                        const float4 s4 = *reinterpret_cast<const float4 *>(sc + c0 + j4);
                        const float4 h4 = *reinterpret_cast<const float4 *>(sh + c0 + j4);
                        v[j4 + 0] = fmaxf(fmaf(__uint_as_float(rr[j4 + 0]), s4.x, h4.x), 0.0f);   // every conv has a ReLU
                        v[j4 + 1] = fmaxf(fmaf(__uint_as_float(rr[j4 + 1]), s4.y, h4.y), 0.0f);
                        v[j4 + 2] = fmaxf(fmaf(__uint_as_float(rr[j4 + 2]), s4.z, h4.z), 0.0f);
                        v[j4 + 3] = fmaxf(fmaf(__uint_as_float(rr[j4 + 3]), s4.w, h4.w), 0.0f);
                    }
                }
                if (!last) {
#pragma unroll
                    for (int j8 = 0; j8 < 32; j8 += 8) {
                        if (c0 + j8 >= cfg.kp(l + 1)) break;
                        uint32_t lo_off;
                        const uint32_t off = mapn.chunk((c0 + j8) >> 3, &lo_off);
                        split8_store(v + j8, buf + off, buf + off + lo_off);
                    }
                } else if (compact) {
                    if (pool_first) pool_units<true>(p, v, lane, c0, cfg.nout(l), sc, sh, my_group, my_ok);
                    else pool_units<false>(p, v, lane, c0, cfg.nout(l), sc, sh, my_group, my_ok);
                } else if (pool_first) {
                    pool_rows<true>(cfg.ns(), p, p.cnt, v, lane, q, tile, c0, cfg.nout(l), sc, sh, xs, wg_bar);
                } else {
                    pool_rows<false>(cfg.ns(), p, p.cnt, v, lane, q, tile, c0, cfg.nout(l), sc, sh, xs, wg_bar);
                }
            }
            tc_fence_before();                                         // TMEM reads done before the next MMAs overwrite it
            SF_T(4 + 4 * l);                                           // epilogue
        }
    }

    tc_fence_before();
    __syncthreads();
    if (tid < 32) {
        tc_fence_after();
        tmem_dealloc(tmem_base_smem, p.tmem_alloc);
    }
}

}  // namespace ssd3d

using namespace ssd3d;

static size_t sf_wimg_bytes(int kp, int npad)              // one half (hi or lo) of a layer's weight image
{
    return (size_t)npad * ((kp / 64) * 128 + sf_rbt_of(kp));
}

struct SfPlan { size_t abuf, w, ssf; int maxn; };
static bool sf_plan(int k_in, int nl, const int *nout, SfPlan *pl)      // k_in: columns of the first operand
{
    if (nl < 1 || nl > SF_MAX_LAYERS) return false;
    pl->abuf = 0; pl->w = 0; pl->ssf = 0; pl->maxn = 32;
    int kp = (k_in + 15) / 16 * 16;
    pl->ssf = 3 * (size_t)kp;                               // room for the hoisted mode's Wx table
    for (int l = 0; l < nl; l++) {
        const int npad = (nout[l] + 15) / 16 * 16;
        if (npad > 256) return false;
        const size_t a = sf_abuf_of(kp);
        if (a > pl->abuf) pl->abuf = a;
        pl->w += 2 * sf_wimg_bytes(kp, npad);
        pl->ssf += (size_t)2 * ((npad + 31) / 32 * 32);
        if (npad > pl->maxn) pl->maxn = npad;
        kp = npad;
    }
    return true;
}
static size_t sf_total(const SfPlan &pl, int slots) { return slots * pl.abuf + pl.w + pl.ssf * sizeof(float) + 1024; }
constexpr size_t SF_SMEM_MAX = 226 * 1024;
constexpr size_t SF_SMALL = 36 * 1024;                     // <= this: single-slot CTAs, up to 6 per SM

// Developer build only (-DSSD3D_DEV_HOOKS, `python 3dssd_b200/build.py dev`, called by tools/fused_probe.py dyn=1):
// launch the run-time-shape kernel even where a compile-time-shape twin exists, for A/B timing of the two.  The shipped
// library has no such state.
#ifdef SSD3D_DEV_HOOKS
static int g_sf_dynamic = 0;
extern "C" void ssd3d_dev_set_fused_dynamic(int on) { g_sf_dynamic = on; }
#else
constexpr int g_sf_dynamic = 0;
#endif

// Slots per CTA for a stack: 1 for small stacks (several CTAs per SM), else as many as fit one SM (<= 3).  A slot of a
// multi-slot CTA has two warpgroups: on the layer-2 stacks 3 x 2 beat the slot x warpgroup shapes 4 x 1, 3 x 1, 2 x 2
// and 2 x 4.
static int sf_slots(const SfPlan &pl)
{
    if (sf_total(pl, 1) <= SF_SMALL) return 1;
    int cols = 32;
    while (cols < pl.maxn) cols *= 2;
    int s = 3;
    while (s > 1 && (sf_total(pl, s) > SF_SMEM_MAX || s * cols > 512)) s--;
    return s;
}

// Shared-memory bytes of the fused kernel for a layer stack, or 0 when it cannot hold it.
extern "C" size_t ssd3d_sa_fused_smem(int c, int nl, const int *nout)
{
    SfPlan pl;
    if (!sf_plan(c + 3, nl, nout, &pl)) return 0;
    const size_t total = sf_total(pl, sf_slots(pl));
    return total <= SF_SMEM_MAX ? total : 0;
}

template <class C, int SLOTS, int WG>
static cudaError_t sf_launch(const SfParams &p, size_t smem, int per_sm, cudaStream_t stream)
{
    cudaError_t e = cudaFuncSetAttribute((const void *)sa_fused_kernel<C, SLOTS, WG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int ctas = (p.tiles + SLOTS - 1) / SLOTS;
    int grid = kNumSMs * per_sm;
    if (grid > ctas) grid = ctas;
    sa_fused_kernel<C, SLOTS, WG><<<grid, SF_THREADS * SLOTS * WG, smem, stream>>>(p);
    return cudaSuccess;
}

// The hoisted two-conv stacks of the shipped 3DSSD configuration (configs/kitti/3dssd/3dssd.yaml:47-52) have compile-time
// twins of the kernel: layer 1 [16 -> 16 -> 32] x32 and [32 -> 32 -> 64] x64 neighbours, layer 2 [64 -> 64 -> 128] x32 and
// [64 -> 96 -> 128] x64.  Returns false when (shape, slots) has no twin: the caller takes the dynamic kernel.
static bool sf_launch_static(const SfParams &p, int slots, size_t smem, int per_sm, cudaStream_t st, cudaError_t *e)
{
    if (!p.hoist || p.nl != 2) return false;
    const int k0 = p.c, n0 = p.nout[0], n1 = p.nout[1], ns = p.ns;
    if (slots == 1) {
        if (k0 == 16 && n0 == 16 && n1 == 32 && ns == 32) { *e = sf_launch<SfStat<16, 16, 32, 32>, 1, 1>(p, smem, per_sm, st); return true; }
        if (k0 == 32 && n0 == 32 && n1 == 64 && ns == 64) { *e = sf_launch<SfStat<32, 32, 64, 64>, 1, 1>(p, smem, per_sm, st); return true; }
    }
    if (slots == 3) {
        if (k0 == 64 && n0 == 64 && n1 == 128 && ns == 32) { *e = sf_launch<SfStat<64, 64, 128, 32>, 3, 2>(p, smem, per_sm, st); return true; }
        if (k0 == 64 && n0 == 96 && n1 == 128 && ns == 64) { *e = sf_launch<SfStat<64, 96, 128, 64>, 3, 2>(p, smem, per_sm, st); return true; }
    }
    return false;
}

// w_blob: per layer { hi image | lo image }, each image = k-blocks of [npad x (64 | tail)] bf16 in the canonical
// K-major swizzled layout (built by params.FusedStack); ss_blob: per layer { scale[sspad] | shift[sspad] }.
// wx != NULL selects the hoisted mode: `points` is the per-point table z (pitch ldz), c its width.
static int sa_mlp_fused_impl(int b, int n, int c, int m, int nsample, const float *xyz, const float *points, int ldz,
                             const float *wx, const float *new_xyz, const int *idx, const int *pts_cnt, const int *units, int nl,
                             const int *nout, const void *w_blob, const float *ss_blob, int last_scale_nonneg,
                             float *out_f32, int ld_f32, void *out_hi, void *out_lo, int ld_split, ssd3d_stream_t stream)
{
    const bool hoist = wx != nullptr;
    SSD3D_REQUIRE(b >= 0 && n > 0 && m >= 0 && c >= 0, "sa_mlp_fused: bad shape");
    SSD3D_REQUIRE(nsample == 8 || nsample == 16 || nsample == 32 || nsample == 64 || nsample == 128,
                  "sa_mlp_fused: nsample=%d must be one of 8, 16, 32, 64, 128", nsample);
    SSD3D_REQUIRE(xyz && new_xyz && idx && w_blob && ss_blob && (points || c == 0), "sa_mlp_fused: null pointer");
    SSD3D_REQUIRE(!hoist || (c > 0 && ldz >= c), "sa_mlp_fused_hoisted: bad table shape n1=%d ldz=%d", c, ldz);
    SSD3D_REQUIRE(out_f32 || (out_hi && out_lo), "sa_mlp_fused: no output requested");
    SSD3D_REQUIRE(!units || (out_f32 && !out_hi && !out_lo), "sa_mlp_fused: a unit list combines through atomicMax on the (zero-filled) fp32 output only");
    SSD3D_REQUIRE((reinterpret_cast<uintptr_t>(w_blob) & 15u) == 0, "sa_mlp_fused: weight blob must be 16-byte aligned");
    SSD3D_REQUIRE(!points || (c & 3) || (hoist && (ldz & 3)) || (reinterpret_cast<uintptr_t>(points) & 15u) == 0,
                  "sa_mlp_fused: points must be 16-byte aligned when c is a multiple of 4");
    const int k_in = hoist ? c : c + 3;
    SfPlan pl;
    const bool planned = sf_plan(k_in, nl, nout, &pl);
    const int slots = planned ? sf_slots(pl) : 0;
    const size_t smem = planned ? sf_total(pl, slots) : 0;
    if (!planned || smem > SF_SMEM_MAX) { set_error("sa_mlp_fused: layer stack does not fit shared memory"); return SSD3D_ERR_UNSUPPORTED; }
    SfParams p = {};
    p.n = n; p.c = c; p.m = m; p.ns = nsample;
    p.rows = (long)b * m * nsample;
    if (p.rows == 0) return 0;
    SSD3D_REQUIRE(p.rows < (1L << 31) - 128, "sa_mlp_fused: too many grouped rows (%ld)", p.rows);
    p.tiles = (int)((p.rows + 127) / 128);
    p.xyz = xyz; p.points = points; p.new_xyz = new_xyz; p.idx = idx; p.cnt = pts_cnt; p.units = units;
    p.hoist = hoist ? 1 : 0; p.ldz = ldz; p.wx = wx;
    p.pool_first = last_scale_nonneg ? 1 : 0;
    p.nl = nl;
    int kprev = (k_in + 15) / 16 * 16;
    uint32_t woff = 0, ssoff = 0;
    for (int l = 0; l < nl; l++) {
        p.kp[l] = kprev;
        p.nout[l] = nout[l];
        p.npad[l] = (nout[l] + 15) / 16 * 16;
        p.nfull[l] = p.kp[l] / 64;
        p.rbt[l] = sf_rbt_of(p.kp[l]);
        p.w_off[l] = woff;
        p.w_half[l] = (uint32_t)sf_wimg_bytes(p.kp[l], p.npad[l]);
        woff += 2 * p.w_half[l];
        p.ss_off[l] = ssoff;
        p.sspad[l] = (p.npad[l] + 31) / 32 * 32;
        ssoff += 2 * p.sspad[l];
        kprev = p.npad[l];
    }
    p.w_total = woff; p.ss_total = ssoff;
    p.w_blob = (const uint8_t *)w_blob; p.ss_blob = ss_blob;
    p.abuf_bytes = (uint32_t)pl.abuf;
    uint32_t cols = 32;
    while ((int)cols < pl.maxn) cols *= 2;
    p.tmem_cols = cols;
    uint32_t alloc = 32;
    while (alloc < cols * (uint32_t)slots) alloc *= 2;
    p.tmem_alloc = alloc;
    p.out_f32 = out_f32; p.ld_f32 = ld_f32;
    p.out_hi = (__nv_bfloat16 *)out_hi; p.out_lo = (__nv_bfloat16 *)out_lo; p.ld_split = ld_split;

    // resident CTAs per SM: bounded by shared memory, TMEM columns (512 per SM) and, for single-slot CTAs, registers
    int per_sm = 1;
    if (slots == 1) {
        per_sm = (int)((227 * 1024) / (smem + 1024));
        if (per_sm > (int)(512 / alloc)) per_sm = 512 / alloc;
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 6) per_sm = 6;                                   // 6 x 128 threads x 80 registers
    }
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    if (g_sf_dynamic || !sf_launch_static(p, slots, smem, per_sm, st, &e))
        e = slots == 1 ? sf_launch<SfDyn, 1, 1>(p, smem, per_sm, st)
          : slots == 2 ? sf_launch<SfDyn, 2, 2>(p, smem, per_sm, st)
                       : sf_launch<SfDyn, 3, 2>(p, smem, per_sm, st);
    if (e != cudaSuccess) return cuda_status(e, "sa_mlp_fused attr");
#ifdef SF_PROFILE
    {
        long long h[16];
        cudaDeviceSynchronize();
        cudaMemcpyFromSymbol(h, sf_prof, sizeof(h));
        fprintf(stderr, "sf_prof slots=%d tiles=%d:", slots, p.tiles);
        for (int i = 0; i < 13; i++) fprintf(stderr, " %lld", h[i]);
        fprintf(stderr, "\n");
        memset(h, 0, sizeof(h));
        cudaMemcpyToSymbol(sf_prof, h, sizeof(h));
    }
#endif
    SSD3D_LAUNCH_CHECK("sa_fused_kernel");
}

extern "C" int ssd3d_sa_mlp_fused(int b, int n, int c, int m, int nsample, const float *xyz, const float *points,
                                  const float *new_xyz, const int *idx, const int *pts_cnt, const int *units, int nl,
                                  const int *nout, const void *w_blob, const float *ss_blob, int last_scale_nonneg,
                                  float *out_f32, int ld_f32, void *out_hi, void *out_lo, int ld_split, ssd3d_stream_t stream)
{
    return sa_mlp_fused_impl(b, n, c, m, nsample, xyz, points, c, nullptr, new_xyz, idx, pts_cnt, units, nl, nout, w_blob, ss_blob,
                             last_scale_nonneg, out_f32, ld_f32, out_hi, out_lo, ld_split, stream);
}

// The fused SA scale with its first conv hoisted (see ssd3d_linear_tc_hoisted): z[b,n,ldz] per-point table (this scale's
// n1 columns start at z), wx = Wx*s1 as [3][n1]; the stack (w_blob / ss_blob / nout) starts at the scale's SECOND conv.
extern "C" int ssd3d_sa_mlp_fused_hoisted(int b, int n, int n1, int m, int nsample, const float *xyz, const float *z, int ldz,
                                          const float *wx, const float *new_xyz, const int *idx, const int *pts_cnt,
                                          const int *units, int nl, const int *nout, const void *w_blob, const float *ss_blob,
                                          int last_scale_nonneg, float *out_f32, int ld_f32, void *out_hi, void *out_lo,
                                          int ld_split, ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(z && wx, "sa_mlp_fused_hoisted: null table pointer");
    return sa_mlp_fused_impl(b, n, n1, m, nsample, xyz, z, ldz, wx, new_xyz, idx, pts_cnt, units, nl, nout, w_blob, ss_blob,
                             last_scale_nonneg, out_f32, ld_f32, out_hi, out_lo, ld_split, stream);
}
