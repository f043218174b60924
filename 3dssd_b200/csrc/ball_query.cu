// ball_query.cu -- radius neighbour search for sm_100a.
//
// Replaces query_ball_point_gpu / query_ball_point_dilated_gpu
// (/root/reference/lib/utils/tf_ops/grouping/tf_grouping_g.cu:215-255, :308-357).
//
// Semantics kept bit-exact: per query, candidates are visited in ascending index order and the FIRST
// `nsample` hits are kept; the first hit back-fills every slot; pts_cnt = number of hits (<= nsample).
//
// Design (DESIGN.md "Ball query"):
//   * the reference runs one thread per query with a serial n-loop and one launch per radius; here a
//     warp owns QW=4 queries and tests 32 candidates per step for all of them (candidate coordinates
//     are read once from shared memory and reused from registers by the 4 queries), hits are appended
//     in index order with ballot + popc prefix, and up to 4 radius shells are answered in ONE pass;
//   * candidate blocks (1024 points, 12 KiB, raw [n,3] layout -- stride-3 reads are bank-conflict free)
//     are staged by 1-D bulk TMA copies (cp.async.bulk + mbarrier), double buffered;
//   * the compare is done on the SQUARED distance against thresholds precomputed on the host such that
//     sqrt_rn(t) < r  <=>  t < T(r): no sqrt in the inner loop, same decisions as the reference;
//   * neighbour lists are assembled in shared memory and written as full coalesced rows; the block
//     stops streaming as soon as every one of its queries is full.
#include <math.h>

#include "common.cuh"

namespace ssd3d {

constexpr int BQ_THREADS = 256;
constexpr int BQ_WARPS = BQ_THREADS / 32;
constexpr int BQ_QW = 4;                      // queries per warp
constexpr int BQ_QPB = BQ_WARPS * BQ_QW;      // queries per block
constexpr int BQ_TILE = 1024;                 // candidate points per stage
constexpr int BQ_MAX_SHELLS = 4;

struct BqParams {
    int n, m, nshell;
    int nsample[BQ_MAX_SHELLS];
    int koff[BQ_MAX_SHELLS];   // offset of the shell's slots inside a query's staging row
    int ktot;                  // staging ints per query
    float t_lo[BQ_MAX_SHELLS];
    float t_hi[BQ_MAX_SHELLS];
    float t_max;               // max over shells of t_hi: cheap reject
    int *idx[BQ_MAX_SHELLS];
    int *cnt[BQ_MAX_SHELLS];
    int use_tma;
};

template <int NS, bool DILATED>
__global__ void __launch_bounds__(BQ_THREADS)
ball_query_kernel(const float *__restrict__ xyz1, const float *__restrict__ xyz2, const BqParams p)
{
    extern __shared__ float4 dyn_smem[];
    float *tile = reinterpret_cast<float *>(dyn_smem);                 // [2][BQ_TILE*3]
    int *stage_idx = reinterpret_cast<int *>(tile + 2 * BQ_TILE * 3);  // [BQ_QPB][ktot]
    __shared__ unsigned long long full_bar[2];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int scene = blockIdx.y;
    const int n = p.n, m = p.m;
    const float *cand = xyz1 + (size_t)scene * n * 3;
    const int q0 = blockIdx.x * BQ_QPB + warp * BQ_QW;  // first query of this warp

    float qx[BQ_QW], qy[BQ_QW], qz[BQ_QW];
    int cnt[BQ_QW][NS];
#pragma unroll
    for (int q = 0; q < BQ_QW; q++) {
        const int qi = q0 + q;
        const bool valid = qi < m;
        const float *src = xyz2 + ((size_t)scene * m + (valid ? qi : 0)) * 3;
        qx[q] = src[0]; qy[q] = src[1]; qz[q] = src[2];
#pragma unroll
        for (int s = 0; s < NS; s++) cnt[q][s] = valid ? 0 : p.nsample[s];  // invalid queries count as full
    }
    int *my_stage = stage_idx + (size_t)(warp * BQ_QW) * p.ktot;

    const int ntiles = (n + BQ_TILE - 1) / BQ_TILE;
    if (tid == 0) {
        mbar_init(smem_u32(&full_bar[0]), p.use_tma ? 1 : BQ_THREADS);
        mbar_init(smem_u32(&full_bar[1]), p.use_tma ? 1 : BQ_THREADS);
        fence_mbar_init_cluster();
    }
    __syncthreads();

    auto load_tile = [&](int t) {
        const int stage = t & 1;
        const int base = t * BQ_TILE;
        const int npts = min(BQ_TILE, n - base);
        float *dst = tile + stage * BQ_TILE * 3;
        if (p.use_tma) {
            if (tid == 0) {
                const uint32_t bytes = (uint32_t)npts * 12u;
                mbar_arrive_expect_tx(smem_u32(&full_bar[stage]), bytes);
                bulk_g2s(smem_u32(dst), cand + (size_t)base * 3, bytes, smem_u32(&full_bar[stage]));
            }
        } else {
            for (int i = tid; i < npts * 3; i += BQ_THREADS) dst[i] = cand[(size_t)base * 3 + i];
            mbar_arrive(smem_u32(&full_bar[stage]));
        }
    };

    load_tile(0);
    if (ntiles > 1) load_tile(1);
    int issued = min(ntiles, 2);
    int consumed = 0;

    for (int t = 0; t < ntiles; t++) {
        const int stage = t & 1;
        mbar_wait_cta(smem_u32(&full_bar[stage]), (t >> 1) & 1);
        const float *pts = tile + stage * BQ_TILE * 3;
        const int base = t * BQ_TILE;
        const int npts = min(BQ_TILE, n - base);

        bool warp_done = true;
#pragma unroll
        for (int q = 0; q < BQ_QW; q++)
#pragma unroll
            for (int s = 0; s < NS; s++) warp_done = warp_done && (cnt[q][s] >= p.nsample[s]);

        if (!warp_done) {
            const int nsteps = (npts + 31) >> 5;
            // squared distances of one candidate (32 per step, one per lane) to the warp's 4 queries.  Packed fp32
            // (FADD2 / FMUL2 / FFMA2, sm_100): two queries per instruction, each lane-half an independent IEEE operation
            // -> same bits as the reference recipe t = dy*dy ; t = fma(dx,dx,t) ; t = fma(dz,dz,t)
            auto dist4 = [&](int li, float (&tt)[BQ_QW]) -> bool {
                const float cx = pts[li * 3], cy = pts[li * 3 + 1], cz = pts[li * 3 + 2];
                const float2 ncx = make_float2(-cx, -cx), ncy = make_float2(-cy, -cy), ncz = make_float2(-cz, -cz);
                bool near_any = false;
#pragma unroll
                for (int q = 0; q < BQ_QW; q += 2) {
                    const float2 dx = __fadd2_rn(make_float2(qx[q], qx[q + 1]), ncx);
                    const float2 dy = __fadd2_rn(make_float2(qy[q], qy[q + 1]), ncy);
                    const float2 dz = __fadd2_rn(make_float2(qz[q], qz[q + 1]), ncz);
                    float2 t = __fmul2_rn(dy, dy);
                    t = __ffma2_rn(dx, dx, t);
                    t = __ffma2_rn(dz, dz, t);
                    tt[q] = t.x; tt[q + 1] = t.y;
                    near_any = near_any || (DILATED ? (t.x < p.t_max) : !(t.x >= p.t_max)) ||
                               (DILATED ? (t.y < p.t_max) : !(t.y >= p.t_max));
                }
                return near_any;
            };
            for (int step2 = 0; step2 < nsteps; step2 += 2) {
                // two steps (64 candidates) per vote: in the common case neither holds a candidate inside any query's
                // largest ball and one __any_sync dismisses both
                float tta[BQ_QW], ttb[BQ_QW];
                const int la = step2 * 32 + lane, lb = la + 32;
                const bool ina = la < npts, inb = lb < npts;             // false only at the ragged end of a scene
                const bool neara = dist4(ina ? la : 0, tta) && ina;
                const bool nearb = dist4(inb ? lb : 0, ttb) && inb;
                if (!__any_sync(0xffffffffu, neara || nearb)) continue;
                bool full2 = false;
#pragma unroll
                for (int half = 0; half < 2 && !full2; half++) {
                    const float (&tt)[BQ_QW] = half ? ttb : tta;
                    const bool in = half ? inb : ina;
                    const int local = half ? lb : la;
                    if (!__any_sync(0xffffffffu, half ? nearb : neara)) continue;
                    const int k = base + local;
#pragma unroll
                    for (int q = 0; q < BQ_QW; q++) {
                        // most slow steps concern ONE of the warp's queries: a single vote skips the others' shells
                        const bool nearq = in && (DILATED ? (tt[q] < p.t_max) : !(tt[q] >= p.t_max));
                        if (!__any_sync(0xffffffffu, nearq)) continue;
#pragma unroll
                        for (int s = 0; s < NS; s++) {
                            const bool hit = in && (DILATED ? (tt[q] == 0.0f || (tt[q] >= p.t_lo[s] && tt[q] < p.t_hi[s]))
                                                            : !(tt[q] >= p.t_hi[s]));
                            const uint32_t hs = __ballot_sync(0xffffffffu, hit);
                            const int c0 = cnt[q][s];
                            const int ns = p.nsample[s];
                            if (hs != 0u && c0 < ns) {
                                int *row = my_stage + q * p.ktot + p.koff[s];
                                const int pos = c0 + __popc(hs & ((1u << lane) - 1u));
                                if (hit && pos < ns) row[pos] = k;
                                cnt[q][s] = min(ns, c0 + __popc(hs));
                            }
                        }
                    }
                    bool all_full = true;
#pragma unroll
                    for (int q = 0; q < BQ_QW; q++)
#pragma unroll
                        for (int s = 0; s < NS; s++) all_full = all_full && (cnt[q][s] >= p.nsample[s]);
                    if (all_full) { warp_done = true; full2 = true; }
                }
                if (full2) break;
            }
        }
        // everyone is done with this stage -> refill it; stop streaming when every warp is full
        const int all_done = __syncthreads_and(warp_done ? 1 : 0);
        consumed = t + 1;
        if (all_done) break;
        if (t + 2 < ntiles) { load_tile(t + 2); issued = t + 3; }
    }
    // never exit with a bulk copy still in flight towards this CTA's shared memory
    for (int u = consumed; u < issued; u++) mbar_wait_cta(smem_u32(&full_bar[u & 1]), (u >> 1) & 1);
    __syncwarp();

    // back-fill (first hit repeated, tf_grouping_g.cu:245-248) and write whole rows
#pragma unroll
    for (int q = 0; q < BQ_QW; q++) {
        const int qi = q0 + q;
        if (qi >= m) continue;
#pragma unroll
        for (int s = 0; s < NS; s++) {
            const int ns = p.nsample[s];
            const int c = cnt[q][s];
            const int *row = my_stage + q * p.ktot + p.koff[s];
            const int first = c > 0 ? row[0] : 0;
            int *dst = p.idx[s] + ((size_t)scene * m + qi) * ns;
            for (int l = lane; l < ns; l += 32) dst[l] = l < c ? row[l] : first;
            if (lane == 0) p.cnt[s][(size_t)scene * m + qi] = c;
        }
    }
}

// smallest float t >= 0 with sqrt_rn(t) >= r   (so  sqrt_rn(t) < r  <=>  t < T(r)  by monotonicity)
static float sq_threshold(float r)
{
    if (!(r > 0.0f)) return 0.0f;
    if (isinf(r)) return INFINITY;
    float t = (float)((double)r * (double)r);
    if (isinf(t)) t = 3.402823466e+38f;
    while (t > 0.0f && sqrtf(nextafterf(t, 0.0f)) >= r) t = nextafterf(t, 0.0f);
    while (!isinf(t) && sqrtf(t) < r) t = nextafterf(t, INFINITY);
    return t;
}

float bq_sq_threshold(float r) { return sq_threshold(r); }   // shared with ball_query_grid.cu

template <int NS>
static cudaError_t launch_bq(bool dilated, dim3 grid, size_t smem, cudaStream_t st, const float *xyz1, const float *xyz2,
                             const BqParams &p)
{
    cudaError_t e;
    if (dilated) {
        e = cudaFuncSetAttribute((const void *)ball_query_kernel<NS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) ball_query_kernel<NS, true><<<grid, BQ_THREADS, smem, st>>>(xyz1, xyz2, p);
    } else {
        e = cudaFuncSetAttribute((const void *)ball_query_kernel<NS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) ball_query_kernel<NS, false><<<grid, BQ_THREADS, smem, st>>>(xyz1, xyz2, p);
    }
    return e;
}

static int ball_query_multi(int b, int n, int m, int nq, int dilated, const float *min_r, const float *max_r,
                            const int *nsample, const float *xyz1, const float *xyz2, int *const *idx,
                            int *const *cnt, cudaStream_t st)
{
    SSD3D_REQUIRE(b >= 0 && n > 0 && m >= 0, "query_ball_point: bad shape b=%d n=%d m=%d", b, n, m);
    SSD3D_REQUIRE(nq >= 1 && nq <= BQ_MAX_SHELLS, "query_ball_point: 1..%d radius shells per call, got %d", BQ_MAX_SHELLS, nq);
    SSD3D_REQUIRE(xyz1 && xyz2, "query_ball_point: null pointer");
    BqParams p = {};
    p.n = n; p.m = m; p.nshell = nq;
    int ktot = 0;
    float tmax = 0.0f;
    for (int s = 0; s < nq; s++) {
        // attribute checks of tf_grouping.cpp:275-279 / :368-374
        SSD3D_REQUIRE(max_r[s] > 0.0f, "query_ball_point expects positive radius");
        SSD3D_REQUIRE(nsample[s] > 0, "query_ball_point expects positive nsample");
        SSD3D_REQUIRE(idx[s] && cnt[s], "query_ball_point: null output pointer");
        p.nsample[s] = nsample[s];
        p.koff[s] = ktot;
        ktot += nsample[s];
        p.t_hi[s] = sq_threshold(max_r[s]);
        p.t_lo[s] = dilated ? sq_threshold(min_r[s]) : 0.0f;
        if (!dilated && !(max_r[s] > 1e-20f)) p.t_hi[s] = -1.0f;  // max(d,1e-20) < r can never hold
        tmax = fmaxf(tmax, p.t_hi[s]);
        p.idx[s] = idx[s];
        p.cnt[s] = cnt[s];
    }
    p.ktot = ktot;
    p.t_max = tmax;
    if (b == 0 || m == 0) return 0;
    // bulk copies need 16-byte aligned sources and sizes: every scene base and every tile length
    p.use_tma = ((reinterpret_cast<uintptr_t>(xyz1) & 15u) == 0 && (n % 4) == 0) ? 1 : 0;
    const size_t smem = (size_t)2 * BQ_TILE * 3 * sizeof(float) + (size_t)BQ_QPB * ktot * sizeof(int);
    SSD3D_REQUIRE(smem <= 200 * 1024, "query_ball_point: sum of nsample (%d) too large for the staging buffer", ktot);
    dim3 grid((unsigned)ceil_div(m, BQ_QPB), (unsigned)b);
    cudaError_t e;
    switch (nq) {
        case 1: e = launch_bq<1>(dilated != 0, grid, smem, st, xyz1, xyz2, p); break;
        case 2: e = launch_bq<2>(dilated != 0, grid, smem, st, xyz1, xyz2, p); break;
        case 3: e = launch_bq<3>(dilated != 0, grid, smem, st, xyz1, xyz2, p); break;
        default: e = launch_bq<4>(dilated != 0, grid, smem, st, xyz1, xyz2, p); break;
    }
    if (e != cudaSuccess) return cuda_status(e, "ball_query_kernel shared-memory opt-in");
    SSD3D_LAUNCH_CHECK("ball_query_kernel");
}

}  // namespace ssd3d

using namespace ssd3d;

extern "C" int ssd3d_query_ball_point(int b, int n, int m, float radius, int nsample, const float *xyz1,
                                      const float *xyz2, int *idx, int *pts_cnt, ssd3d_stream_t stream)
{
    const float lo = 0.0f;
    return ball_query_multi(b, n, m, 1, 0, &lo, &radius, &nsample, xyz1, xyz2, &idx, &pts_cnt, (cudaStream_t)stream);
}

extern "C" int ssd3d_query_ball_point_dilated(int b, int n, int m, float min_radius, float max_radius, int nsample,
                                              const float *xyz1, const float *xyz2, int *idx, int *pts_cnt,
                                              ssd3d_stream_t stream)
{
    return ball_query_multi(b, n, m, 1, 1, &min_radius, &max_radius, &nsample, xyz1, xyz2, &idx, &pts_cnt,
                            (cudaStream_t)stream);
}

extern "C" int ssd3d_query_ball_point_multi(int b, int n, int m, int nqueries, int dilated, const float *min_radius,
                                            const float *max_radius, const int *nsample, const float *xyz1,
                                            const float *xyz2, int *const *idx, int *const *pts_cnt,
                                            ssd3d_stream_t stream)
{
    return ball_query_multi(b, n, m, nqueries, dilated, min_radius, max_radius, nsample, xyz1, xyz2, idx, pts_cnt,
                            (cudaStream_t)stream);
}
