// nms.cu -- per-scene greedy BEV non-maximum suppression on the GPU (SURVEY.md section 8f, row f2).
//
// Replaces the per-scene, per-class tf.image.non_max_suppression call of the reference's post-processor
// (/root/reference/lib/builder/postprocessor.py:76-88), which runs on the CPU in the middle of inference, together
// with the projections that feed it: box_3d_to_anchor (lib/utils/box_3d_utils.py:25-58) and project_to_bev
// (lib/utils/anchors_util.py:11-48).  Semantics kept: candidates in descending score order (ties: lower index
// first), a candidate is dropped when its axis-aligned BEV IoU with an already kept box is > iou_threshold, at most
// max_output boxes are kept.  Output is the fixed-size block the multi-GPU gather moves: [max_output, 9] =
// (x, y, z, l, h, w, ry, score, class) zero padded, plus the number of kept boxes.
//
// One CTA per scene: bitonic sort of (score, index) keys in shared memory, one thread per candidate builds its
// row of the "suppresses" bit matrix, one warp walks the rows greedily.
#include "common.cuh"

namespace ssd3d {

constexpr int NMS_THREADS = 256;
constexpr int NMS_MAX_N = 512;

__global__ void __launch_bounds__(NMS_THREADS)
bev_nms_kernel(int n, int npow2, const float *__restrict__ boxes, const float *__restrict__ scores, float iou_thr,
               int max_out, int cls_id, float *__restrict__ out_block, int *__restrict__ out_cnt)
{
    __shared__ unsigned long long keys[NMS_MAX_N];
    __shared__ float4 bev[NMS_MAX_N];                       // x1, z1, x2, z2 in sorted order
    __shared__ uint32_t sup[NMS_MAX_N][NMS_MAX_N / 32];     // sup[i] bit j: sorted box i suppresses sorted box j (j > i)
    __shared__ int kept[NMS_MAX_N];
    __shared__ int nkept;

    const int scene = blockIdx.x, tid = threadIdx.x;
    const float *bx = boxes + (size_t)scene * n * 7;
    const float *sc = scores + (size_t)scene * n;

    // ---- sort keys: (score desc, index asc)  ==  descending on (ord(score) << 32 | ~index)
    for (int i = tid; i < npow2; i += NMS_THREADS)
        keys[i] = i < n ? (((unsigned long long)f2ord(sc[i]) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)i)) : 0ull;
    __syncthreads();
    for (int k = 2; k <= npow2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < npow2; i += NMS_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], b = keys[ixj];
                    const bool desc = (i & k) == 0;
                    if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
    // ---- BEV extents of the sorted candidates
    for (int i = tid; i < n; i += NMS_THREADS) {
        const int src = (int)(0xffffffffu - (uint32_t)(keys[i] & 0xffffffffull));
        const float *b7 = bx + (size_t)src * 7;
        const float x = b7[0], z = b7[2], l = b7[3], w = b7[5], ry = b7[6];
        const float c = fabsf(cosf(ry)), s = fabsf(sinf(ry));
        const float dimx = l * c + w * s, dimz = w * c + l * s;         // box_3d_to_anchor
        bev[i] = make_float4(x - dimx * 0.5f, z - dimz * 0.5f, x + dimx * 0.5f, z + dimz * 0.5f);   // project_to_bev
    }
    __syncthreads();
    // ---- suppression rows
    const int nwords = (n + 31) / 32;
    for (int i = tid; i < n; i += NMS_THREADS) {
        const float4 a = bev[i];
        const float area_a = (a.z - a.x) * (a.w - a.y);
        for (int wd = 0; wd < nwords; wd++) {
            uint32_t bits = 0u;
            for (int t = 0; t < 32; t++) {
                const int j = wd * 32 + t;
                if (j <= i || j >= n) continue;
                const float4 b = bev[j];
                const float area_b = (b.z - b.x) * (b.w - b.y);
                if (area_a <= 0.0f || area_b <= 0.0f) continue;
                const float iw = fminf(a.z, b.z) - fmaxf(a.x, b.x), ih = fminf(a.w, b.w) - fmaxf(a.y, b.y);
                // disjoint rectangles (the common case): inter == 0, IoU == 0 (or NaN), never > threshold -- skip the divide
                if (iou_thr >= 0.0f && (!(iw > 0.0f) || !(ih > 0.0f))) continue;
                const float inter = fmaxf(iw, 0.0f) * fmaxf(ih, 0.0f);
                if (inter / (area_a + area_b - inter) > iou_thr) bits |= 1u << t;
            }
            sup[i][wd] = bits;
        }
    }
    __syncthreads();
    // ---- greedy walk (one warp; lane w owns word w of the "removed" mask)
    if (tid < 32) {
        uint32_t removed = 0u;                               // lane w: word w (n <= 512 -> 16 words)
        int cnt = 0;
        for (int i = 0; i < n && cnt < max_out; i++) {
            const uint32_t word = __shfl_sync(0xffffffffu, removed, i >> 5);
            if ((word >> (i & 31)) & 1u) continue;
            if (tid == 0) kept[cnt] = i;
            cnt++;
            if (tid < nwords) removed |= sup[i][tid];
        }
        if (tid == 0) nkept = cnt;
    }
    __syncthreads();
    // ---- fixed-size output block
    const int cnt = nkept;
    float *ob = out_block + (size_t)scene * max_out * 9;
    for (int e = tid; e < max_out * 9; e += NMS_THREADS) {
        const int k = e / 9, f = e - k * 9;
        float v = 0.0f;
        if (k < cnt) {
            const int src = (int)(0xffffffffu - (uint32_t)(keys[kept[k]] & 0xffffffffull));
            v = f < 7 ? bx[(size_t)src * 7 + f] : (f == 7 ? sc[src] : (float)cls_id);
        }
        ob[e] = v;
    }
    if (tid == 0) out_cnt[scene] = cnt;
}

}  // namespace ssd3d

using namespace ssd3d;

extern "C" int ssd3d_bev_nms(int b, int n, const float *boxes, const float *scores, float iou_threshold, int max_output,
                             int cls_id, float *out_block, int *out_cnt, ssd3d_stream_t stream)
{
    SSD3D_REQUIRE(b >= 0 && n > 0 && max_output > 0, "bev_nms: bad shape b=%d n=%d max_output=%d", b, n, max_output);
    SSD3D_REQUIRE(n <= NMS_MAX_N, "bev_nms: at most %d candidates per scene (got %d)", NMS_MAX_N, n);
    SSD3D_REQUIRE(boxes && scores && out_block && out_cnt, "bev_nms: null pointer");
    if (b == 0) return 0;
    int npow2 = 1;
    while (npow2 < n) npow2 <<= 1;
    bev_nms_kernel<<<b, NMS_THREADS, 0, (cudaStream_t)stream>>>(n, npow2, boxes, scores, iou_threshold, max_output, cls_id,
                                                               out_block, out_cnt);
    SSD3D_LAUNCH_CHECK("bev_nms_kernel");
}
