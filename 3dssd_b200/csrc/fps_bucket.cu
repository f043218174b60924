// fps_bucket.cu -- D-FPS on xyz for large scenes (8192 < n <= 16384: 3DSSD layer 1) with SPATIAL PRUNING.
//
// Same function as fps3_direct_kernel (fps.cu), i.e. farthestpointsamplingKernel of
// /root/reference/lib/utils/tf_ops/sampling/tf_sampling_g.cu:124-178 for c == 3, same indices bit for bit.
//
// Why another kernel.  A round of FPS is  dist[k] = min(dist[k], d(k, last sample))  for every point, then an arg-max.
// The cluster kernel does the full update with the points spread over 4-8 SMs and pays a DSMEM exchange per round
// (~390 ns per round, 4095 rounds, 32-64 SMs busy per batch of 8 scenes).  But after a few dozen rounds a new sample
// can only LOWER the running distance of points in its own neighbourhood: dist[k] is already the distance to the
// nearest of j samples, so only points closer to the new sample than that change.  With the points grouped into
// spatially compact buckets of 32 (2-D Morton order of the two widest axes) and an axis-aligned box per bucket,
//     lower bound of d(any point of the box, s)  >=  max running distance inside the bucket
// proves that the round leaves the bucket untouched -- no distance needs to be computed, and its cached (max, arg-max)
// stays valid.  On KITTI-like scenes a round touches ~6 of the 512 buckets (tools/fps_bucket_sim.py).  A whole scene then
// fits ONE CTA: coordinates in shared memory (SoA, 192 KiB), running distances in registers (32 per thread), no
// cluster, no DSMEM; a round is  bucket test -> update of the (usually one) affected bucket of a warp -> one
// __syncthreads -> 16-entry arg-max.  The reductions carry (value, key) only, and the key word holds the point's place
// in bucket order below its tie-break fields, so the winner's coordinates are one shared-memory read away: a ballot +
// find-first to track lanes costs as much as the two REDUX of a stage (tools/ubench/warp_ops.cu).  One SM per scene
// instead of 4-8.
//
// Exactness.  Skipping is the only approximation-shaped step and it is one-sided: a bucket is skipped only when
// lb * (1 - 1e-5) >= bucket max, where lb is the squared distance from the sample to the box computed in fp32; the
// reference's fp32 distance of any point inside the box is >= lb * (1 - 8 * 2^-24) (every operation rounds to nearest
// and all terms are non-negative), so a skipped point satisfies d >= dist[k] and min() would not have changed it.
// Tiny values (lb < 1e-30, where denormal rounding breaks relative bounds) never skip.  Everything that IS computed
// uses the reference's contracted recipe d = fma(dz,dz, fma(dy,dy, dx*dx)) and the arg-max order
// (value desc, k mod 1024 asc, k asc) of fps.cu.  The bucket assignment itself cannot change a result.
//
// Resumable like fps3_direct_kernel (rounds [j0, j1)): running distances travel through temp[scene][0:n] in ORIGINAL
// point order, the bucket permutation through temp[scene][n:2n], so a resumed launch skips the sort.
#include "common.cuh"
#include "fps.cuh"

namespace ssd3d {

constexpr int FB_T = 512;                    // threads per CTA (one CTA per scene)
constexpr int FB_NW = FB_T / 32;             // 16 warps
constexpr int FB_SLOTS = 32;                 // buckets per warp: lane l OWNS the meta data of the warp's slot l
constexpr int FB_NBUCKET = FB_NW * FB_SLOTS; // 512
constexpr int FB_MAXN = FB_NBUCKET * 32;     // 16384 points
constexpr uint32_t FB_PAD_KEY = 0xFFFFFFFFu;

__device__ __forceinline__ uint32_t fb_spread9(uint32_t v)   // 9 bits -> every second bit
{
    v &= 0x1ffu;
    v = (v | (v << 8)) & 0x00ff00ffu;
    v = (v | (v << 4)) & 0x0f0f0f0fu;
    v = (v | (v << 2)) & 0x33333333u;
    v = (v | (v << 1)) & 0x55555555u;
    return v;
}

// position of (warp w, slot i, lane l) in bucket order: consecutive buckets belong to different warps, so the buckets a
// sample touches (neighbours in Morton order) are worked on in parallel
__device__ __forceinline__ int fb_pos(int w, int i, int lane) { return ((i * FB_NW + w) << 5) + lane; }

// Tie-break key of point `o` (original index, < 16384) WITH its position p in bucket order in the low bits: ordered like
// fps_key -- (o mod 1024, o div 1024) -- because those two fields are unique per point and sit above the position.  A
// min-reduction over these words therefore returns the reference's winner AND where its coordinates are; no lane or
// position has to be tracked through the stages (a ballot + find-first per stage cost as much as the stage's reductions).
__device__ __forceinline__ uint32_t fb_key(uint32_t o, uint32_t p) { return ((o & 1023u) << 21) | ((o >> 10) << 17) | p; }
__device__ __forceinline__ int fb_key_to_k(uint32_t key) { return (int)((((key >> 17) & 15u) << 10) | (key >> 21)); }

#define FB_CASE(I)                                                              \
    case I:                                                                     \
        nd = fminf(d, dist[I]);                                                 \
        dist[I] = nd;                                                           \
        break;

__global__ void __launch_bounds__(FB_T, 1)
fps3_bucket_kernel(int n, int m, const float *__restrict__ inp, int *__restrict__ out, const FpsIO io)
{
    extern __shared__ float4 fb_dyn[];
    float *xs = reinterpret_cast<float *>(fb_dyn);          // [FB_MAXN] sorted x          (first 64 KiB: sort keys during setup)
    float *ys = xs + FB_MAXN, *zs = ys + FB_MAXN;
    uint32_t *skey = reinterpret_cast<uint32_t *>(fb_dyn);
    __shared__ __align__(8) uint2 slots[2][FB_NW];          // per round parity: (max bits, key) of every warp's best point
    __shared__ uint32_t red[6][FB_NW];
    __shared__ uint16_t orig_of[FB_MAXN];                   // position in bucket order -> original index (0xffff: no point)

    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int scene = blockIdx.x;
    const float *data = inp + (size_t)scene * io.sa;
    int *idxs = out + (size_t)scene * io.ldo;
    const int jbeg = io.j0 > 1 ? io.j0 : 1, jend = io.j1 < m ? io.j1 : m;
    const bool resume = io.j0 > 0, save = io.j1 < m;
    float *tsave = io.temp ? io.temp + (size_t)scene * 2 * n : nullptr;
    uint32_t *perm = tsave ? reinterpret_cast<uint32_t *>(tsave + n) : nullptr;

    float dist[FB_SLOTS];

    if (!resume) {
        // ---- scene box -> 2-D Morton keys of the two widest axes -> bitonic sort (key = morton18 : index14)
        float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
        for (int k = tid; k < n; k += FB_T) {
#pragma unroll
            for (int a = 0; a < 3; a++) {
                const float v = __ldg(data + 3 * k + a);
                lo[a] = fminf(lo[a], v); hi[a] = fmaxf(hi[a], v);
            }
        }
#pragma unroll
        for (int a = 0; a < 3; a++) {
            const uint32_t mn = __reduce_min_sync(0xffffffffu, f2ord(lo[a])), mx = __reduce_max_sync(0xffffffffu, f2ord(hi[a]));
            if (lane == 0) { red[a][w] = mn; red[3 + a][w] = mx; }
        }
        __syncthreads();
        float ext[3];
#pragma unroll
        for (int a = 0; a < 3; a++) {
            uint32_t mn = 0xffffffffu, mx = 0u;
            for (int q = 0; q < FB_NW; q++) { mn = min(mn, red[a][q]); mx = max(mx, red[3 + a][q]); }
            lo[a] = ord2f(mn); hi[a] = ord2f(mx);
            ext[a] = hi[a] - lo[a];
        }
        // the two widest axes (a0 widest), square cells sized by the widest; non-finite extents just give poor buckets
        int a0 = 0, a1 = 1;
        if (ext[1] > ext[a0]) a0 = 1;
        if (ext[2] > ext[a0]) a0 = 2;
        a1 = a0 == 0 ? 1 : 0;
        for (int a = 0; a < 3; a++)
            if (a != a0 && ext[a] > ext[a1]) a1 = a;
        const float scale = ext[a0] > 0.0f ? 511.999f / ext[a0] : 0.0f;
        int np = 1024;
        while (np < n) np <<= 1;                                  // sort size (n <= FB_MAXN)
        for (int k = tid; k < np; k += FB_T) {
            uint32_t key = FB_PAD_KEY;
            if (k < n) {
                const float u = (__ldg(data + 3 * k + a0) - lo[a0]) * scale, v = (__ldg(data + 3 * k + a1) - lo[a1]) * scale;
                const uint32_t qu = (uint32_t)min(511, max(0, (int)u)), qv = (uint32_t)min(511, max(0, (int)v));
                key = ((fb_spread9(qu) | (fb_spread9(qv) << 1)) << 14) | (uint32_t)k;
            }
            skey[k] = key;
        }
        __syncthreads();
        for (int k = 2; k <= np; k <<= 1) {
            for (int jj = k >> 1; jj > 0; jj >>= 1) {
                for (int t = tid; t < (np >> 1); t += FB_T) {
                    const int l = ((t & ~(jj - 1)) << 1) | (t & (jj - 1));
                    const int h = l | jj;
                    const bool asc = (l & k) == 0;
                    const uint32_t a = skey[l], b2 = skey[h];
                    if ((a > b2) == asc) { skey[l] = b2; skey[h] = a; }
                }
                __syncthreads();
            }
        }
#pragma unroll
        for (int i = 0; i < FB_SLOTS; i++) {
            const int p = fb_pos(w, i, lane);
            uint32_t o = 0xffffu;                                  // 0xffff marks "no point" (n <= 16384 < 0xffff)
            if (p < n) o = skey[p] & 0x3fffu;
            orig_of[p] = (uint16_t)o;
            if (tsave != nullptr && p < n) perm[p] = o;
        }
        __syncthreads();                                           // sort buffer consumed: xs may be overwritten
    } else {
#pragma unroll
        for (int i = 0; i < FB_SLOTS; i++) {
            const int p = fb_pos(w, i, lane);
            orig_of[p] = (uint16_t)(p < n ? (perm[p] & 0xffffu) : 0xffffu);
        }
    }

    // ---- coordinates into bucket order, bucket boxes, running distances
    float bminx = 0, bminy = 0, bminz = 0, bmaxx = 0, bmaxy = 0, bmaxz = 0;   // box of the slot this lane owns
    uint32_t bmaxu = 0u, bkey = KEY_INVALID;                                  // its max (bits) and the key of the point holding it
#pragma unroll
    for (int i = 0; i < FB_SLOTS; i++) {
        const int p = fb_pos(w, i, lane);
        const uint32_t o = orig_of[p];                             // written by this thread above
        const bool valid = o != 0xffffu;
        float x = 0.0f, y = 0.0f, z = 0.0f;
        if (valid) { x = __ldg(data + 3 * o); y = __ldg(data + 3 * o + 1); z = __ldg(data + 3 * o + 2); }
        xs[p] = x; ys[p] = y; zs[p] = z;
        dist[i] = valid ? (resume ? tsave[o] : 1e38f) : -1.0f;    // tf_sampling_g.cu:136
        const uint32_t mnx = __reduce_min_sync(0xffffffffu, valid ? f2ord(x) : 0xffffffffu);
        const uint32_t mny = __reduce_min_sync(0xffffffffu, valid ? f2ord(y) : 0xffffffffu);
        const uint32_t mnz = __reduce_min_sync(0xffffffffu, valid ? f2ord(z) : 0xffffffffu);
        const uint32_t mxx = __reduce_max_sync(0xffffffffu, valid ? f2ord(x) : 0u);
        const uint32_t mxy = __reduce_max_sync(0xffffffffu, valid ? f2ord(y) : 0u);
        const uint32_t mxz = __reduce_max_sync(0xffffffffu, valid ? f2ord(z) : 0u);
        // arg-max of the slot as it stands (a fresh start has 1e38 everywhere: every bucket is "affected" in round 1)
        const uint32_t u = valid ? __float_as_uint(fmaxf(dist[i], 0.0f)) : 0u;
        const uint32_t key = valid ? fb_key(o, (uint32_t)p) : KEY_INVALID;
        uint32_t mx, kmin;
        warp_argmax(u, key, mx, kmin);
        if (lane == i) {
            bminx = ord2f(mnx); bminy = ord2f(mny); bminz = ord2f(mnz);
            bmaxx = ord2f(mxx); bmaxy = ord2f(mxy); bmaxz = ord2f(mxz);
            bmaxu = mx; bkey = kmin;
        }
    }

    int old0 = 0;
    if (resume) old0 = idxs[jbeg - 1] - io.ioff;                  // written by the previous launch of this scene
    else if (tid == 0) idxs[0] = io.ioff;
    float sx = __ldg(data + 3 * old0), sy = __ldg(data + 3 * old0 + 1), sz = __ldg(data + 3 * old0 + 2);
    // the warp's best over its 32 slots, cached between rounds (valid while none of its buckets changes)
    uint32_t wm = 0u, wk = KEY_INVALID;
    bool wdirty = true;
    __syncthreads();                                               // xs / ys / zs complete

    for (int j = jbeg; j < jend; j++) {
        const int par = j & 1;
        // ---- which of this warp's buckets can the new sample change?  (lane l tests slot l)
        const float gx = fmaxf(fmaxf(bminx - sx, sx - bmaxx), 0.0f);
        const float gy = fmaxf(fmaxf(bminy - sy, sy - bmaxy), 0.0f);
        const float gz = fmaxf(fmaxf(bminz - sz, sz - bmaxz), 0.0f);
        const float lb = gx * gx + gy * gy + gz * gz;
        const bool skip = bmaxu == 0u || (lb * 0.99999f >= __uint_as_float(bmaxu) && lb >= 1e-30f);
        uint32_t mask = __ballot_sync(0xffffffffu, !skip);
        wdirty = wdirty || mask != 0u;
        while (mask) {
            const int i = 31 - __clz(mask);                        // warp-uniform; any order (find-leading-one is the cheaper one)
            mask &= ~(1u << i);
            const int p = fb_pos(w, i, lane);
            const uint32_t kk = orig_of[p];
            const float dx = xs[p] - sx, dy = ys[p] - sy, dz = zs[p] - sz;
            float d = __fmul_rn(dx, dx);
            d = __fmaf_rn(dy, dy, d);
            d = __fmaf_rn(dz, dz, d);
            float nd;
            switch (i) {
                FB_CASE(0) FB_CASE(1) FB_CASE(2) FB_CASE(3) FB_CASE(4) FB_CASE(5) FB_CASE(6) FB_CASE(7)
                FB_CASE(8) FB_CASE(9) FB_CASE(10) FB_CASE(11) FB_CASE(12) FB_CASE(13) FB_CASE(14) FB_CASE(15)
                FB_CASE(16) FB_CASE(17) FB_CASE(18) FB_CASE(19) FB_CASE(20) FB_CASE(21) FB_CASE(22) FB_CASE(23)
                FB_CASE(24) FB_CASE(25) FB_CASE(26) FB_CASE(27) FB_CASE(28) FB_CASE(29) FB_CASE(30)
                default: nd = fminf(d, dist[31]); dist[31] = nd; break;
            }
            const bool valid = kk != 0xffffu;
            const uint32_t u = valid ? __float_as_uint(fmaxf(nd, 0.0f)) : 0u;
            const uint32_t key = valid ? fb_key(kk, (uint32_t)p) : KEY_INVALID;
            uint32_t mx, kmin;
            warp_argmax(u, key, mx, kmin);
            if (lane == i) { bmaxu = mx; bkey = kmin; }
        }
        if (wdirty) {                                              // warp-uniform
            warp_argmax(bmaxu, bkey, wm, wk);
            wdirty = false;
        }
        if (lane == 0) slots[par][w] = make_uint2(wm, wk);
        __syncthreads();
        // ---- scene-wide arg-max of the 16 warp candidates (every warp, redundantly: no second barrier); the winning key
        // carries the winner's place
        const uint2 c = slots[par][lane & (FB_NW - 1)];
        uint32_t m3, k3;
        warp_argmax(c.x, c.y, m3, k3);
        const int p = (int)(k3 & 0x3fffu);
        sx = xs[p]; sy = ys[p]; sz = zs[p];
        if (tid == 0) idxs[j] = fb_key_to_k(k3) + io.ioff;
    }

    if (save) {
#pragma unroll
        for (int i = 0; i < FB_SLOTS; i++) {
            const uint32_t o = orig_of[fb_pos(w, i, lane)];
            if (o != 0xffffu) tsave[o] = dist[i];
        }
    }
}

bool fps3_bucket_applies(int n, int m, const float *inp, long long sa, int flags)
{
    (void)inp; (void)sa;
    if (flags & 2) return false;                                   // caller forbids it (tests, experiments)
    if (n > FB_MAXN || n < 64 || m < 2) return false;
    if (flags & 4) return true;                                    // caller forces it (tests: any n in range)
    return n > 8192 && m >= 256;
}

int launch_fps3_bucket(int b, int n, int m, const float *inp, int *out, const FpsIO &io, cudaStream_t st)
{
    const size_t smem = (size_t)3 * FB_MAXN * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute((const void *)fps3_bucket_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    fps3_bucket_kernel<<<b, FB_T, smem, st>>>(n, m, inp, out, io);
    return (int)cudaGetLastError();
}

}  // namespace ssd3d
