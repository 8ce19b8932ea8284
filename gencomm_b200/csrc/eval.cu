// Detection-to-ground-truth matching of the evaluation: eval_utils.caluclate_tp_fp (opencood/utils/eval_utils.py) with
// the polygon IoU of common_utils.compute_iou, batched over frames and thresholds, no host round trip (the reference
// copies every frame's boxes to the host and, in score order, intersects each detection's shapely polygon with every
// still-unmatched ground-truth polygon in a Python loop, once per IoU threshold).
//
//   k_eval_prep  : one CTA per frame: stable descending sort of the detections by score (bitonic sort of 64-bit keys
//                  order-preserving(score) << 32 | ~index, so equal scores keep their input order), sorted scores out,
//                  float64 bottom-face quads, AABBs and areas of the sorted detections and of the ground truths.
//   k_eval_iou   : many CTAs per frame, one thread per (detection, ground truth) pair: float32 IoU matrix [k][g] in the
//                  workspace (rotated_iou.cuh, bit-matched to oracle/nms_ref.c; disjoint AABBs skip the clipping, whose
//                  intersection is 0 there), plus a per-detection flag "some IoU >= the smallest threshold, or NaN".
//   k_eval_match : one warp per (frame, threshold): the greedy match in sorted order.  Unflagged detections are false
//                  positives at every threshold without reading their row; a flagged row is scanned lane-strided with
//                  numpy's max / argmax rules over the still-unmatched ground truths.  Lane l owns ground truths
//                  l, l + 32, ..., so the unmatched set is one 32-bit register per lane.
//
// Latency-bound geometry like the NMS (DESIGN §5i): sized so that a batch of frames fills the SMs.
#include <math.h>

#include "common.cuh"
#include "rotated_iou.cuh"

namespace gc {
namespace evalm {

constexpr int kMax = 1024;      // k_max, g_max limit (one sort key / one ground truth per thread of a 1024-thread CTA)
constexpr int kMaxThresh = 8;   // thresholds per call (one warp each in k_eval_match)

struct Thresholds {
    double v[kMaxThresh];
    double min;   // smallest of v[0..n): a detection whose IoUs are all below it (and not NaN) is a FP at every threshold
};

// Workspace of one call, carved from the caller's buffer (all arrays frame-major)
struct Ws {
    double *det_quad;   // [B][k_max][8] bottom-face corners 0..3 (x, y) of the sorted detections
    double *det_box;    // [B][k_max][5] xmin, ymin, xmax, ymax, |area|
    double *gt_quad;    // [B][g_max][8]
    double *gt_box;     // [B][g_max][5]
    int *counts;        // [B][2] clamped detection / ground-truth counts
    int *flag;          // [B][k_max] row has an IoU >= Thresholds::min or NaN
    float *iou;         // [B][k_max][g_max]
    size_t bytes;
};

inline Ws carve(void *base, int n_frames, int k_max, int g_max) {
    Ws w;
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    const size_t B = (size_t)n_frames;
    w.det_quad = (double *)take(B * k_max * 8 * sizeof(double));
    w.det_box = (double *)take(B * k_max * 5 * sizeof(double));
    w.gt_quad = (double *)take(B * g_max * 8 * sizeof(double));
    w.gt_box = (double *)take(B * g_max * 5 * sizeof(double));
    w.counts = (int *)take(B * 2 * sizeof(int));
    w.flag = (int *)take(B * k_max * sizeof(int));
    w.iou = (float *)take(B * k_max * g_max * sizeof(float));
    w.bytes = off;
    return w;
}

// float -> uint32 with the same order (-0.0 is folded onto +0.0: numpy compares them equal)
__device__ __forceinline__ uint32_t order_key(float s) {
    const uint32_t u = __float_as_uint(s == 0.0f ? 0.0f : s);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// bottom-face quad of one [8][3] box in float64, its AABB and its |area| (the value quad_iou uses)
__device__ __forceinline__ void box_geometry(const float *__restrict__ box, double *quad, double *aabb) {
    double q[8];
    double xmin = INFINITY, ymin = INFINITY, xmax = -INFINITY, ymax = -INFINITY;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const double x = (double)__ldg(box + 3 * c), y = (double)__ldg(box + 3 * c + 1);
        q[2 * c] = x; q[2 * c + 1] = y;
        xmin = fmin(xmin, x); xmax = fmax(xmax, x); ymin = fmin(ymin, y); ymax = fmax(ymax, y);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) quad[k] = q[k];
    aabb[0] = xmin; aabb[1] = ymin; aabb[2] = xmax; aabb[3] = ymax;
    aabb[4] = fabs(riou::poly_area(q, 4));
}

// ---- 1/3: one CTA per frame: stable score sort, sorted scores, geometry ----
__global__ void __launch_bounds__(kMax)
k_eval_prep(const float *__restrict__ det_boxes, const float *__restrict__ det_scores, const int *__restrict__ det_counts,
            int k_max, const float *__restrict__ gt_boxes, const int *__restrict__ gt_counts, int g_max, Ws ws,
            float *__restrict__ sorted_scores) {
    __shared__ unsigned long long s_keys[kMax];
    const int f = blockIdx.x, tid = threadIdx.x;
    const int k = min(max(det_counts[f], 0), k_max), g = min(max(gt_counts[f], 0), g_max);
    const float *scores = det_scores + (size_t)f * k_max;
    int width = 1;   // bitonic width: the next power of two >= k
    while (width < k) width <<= 1;
    if (tid < width) s_keys[tid] = tid < k ? ((unsigned long long)order_key(__ldg(scores + tid)) << 32) | (uint32_t)~tid : 0ull;
    __syncthreads();
    for (int s = 2; s <= width; s <<= 1) {
        for (int j = s >> 1; j > 0; j >>= 1) {
            const int partner = tid ^ j;
            if (tid < width && partner > tid) {
                const unsigned long long x = s_keys[tid], y = s_keys[partner];
                const bool desc = (tid & s) == 0;
                if (desc ? x < y : x > y) { s_keys[tid] = y; s_keys[partner] = x; }
            }
            __syncthreads();
        }
    }
    if (tid < k_max) {
        float sc = 0.0f;
        if (tid < k) {
            const int src = (int)~(uint32_t)(s_keys[tid] & 0xffffffffull);
            sc = __ldg(scores + src);
            const size_t row = (size_t)f * k_max + tid;
            box_geometry(det_boxes + ((size_t)f * k_max + src) * 24, ws.det_quad + row * 8, ws.det_box + row * 5);
            ws.flag[row] = 0;
        }
        sorted_scores[(size_t)f * k_max + tid] = sc;
    }
    if (tid < g) {
        const size_t row = (size_t)f * g_max + tid;
        box_geometry(gt_boxes + row * 24, ws.gt_quad + row * 8, ws.gt_box + row * 5);
    }
    if (tid == 0) { ws.counts[2 * f] = k; ws.counts[2 * f + 1] = g; }
}

// ---- 2/3: IoU matrix, one thread per (sorted detection i, ground truth j) of the frame ----
__global__ void __launch_bounds__(256)
k_eval_iou(Ws ws, int k_max, int g_max, double thr_min) {
    const int f = blockIdx.y;
    const int k = ws.counts[2 * f], g = ws.counts[2 * f + 1];
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= k * g) return;
    const int i = p / g, j = p - i * g;
    const size_t di = (size_t)f * k_max + i, gj = (size_t)f * g_max + j;
    const double *a = ws.det_box + di * 5, *b = ws.gt_box + gj * 5;
    float iou;
    if (b[0] > a[2] || b[2] < a[0] || b[1] > a[3] || b[3] < a[1]) {
        // no overlap: quad_iou's intersection is 0, leaving 0 / (|A| + |B| - 0)
        iou = (float)__ddiv_rn(0.0, riou::ds(riou::da(a[4], b[4]), 0.0));
    } else {
        double qa[8], qb[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) { qa[c] = ws.det_quad[di * 8 + c]; qb[c] = ws.gt_quad[gj * 8 + c]; }
        iou = riou::quad_iou(qa, qb);
    }
    ws.iou[di * g_max + j] = iou;
    if (isnan(iou) || (double)iou >= thr_min) ws.flag[di] = 1;
}

// numpy's max / argmax order over (iou, gt index): NaN beats any number, larger beats smaller, then the lower index
__device__ __forceinline__ bool beats(float v, int j, float w, int l) {
    const bool nv = isnan(v), nw = isnan(w);
    if (nv != nw) return nv;
    if (!nv && v != w) return v > w;
    return j < l;
}

// ---- 3/3: one warp per (frame, threshold): greedy matching in score order ----
__global__ void __launch_bounds__(32 * kMaxThresh)
k_eval_match(Ws ws, int k_max, int g_max, Thresholds th, int n_thresh, uint8_t *__restrict__ tp) {
    const int f = blockIdx.x, t = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (t >= n_thresh) return;
    const int k = ws.counts[2 * f], g = ws.counts[2 * f + 1];
    double thr = th.v[0];   // selected without a dynamic index, which would copy the parameter struct to local memory
#pragma unroll
    for (int u = 1; u < kMaxThresh; ++u) thr = u == t ? th.v[u] : thr;
    const float *iou = ws.iou + (size_t)f * k_max * g_max;
    const int *flag = ws.flag + (size_t)f * k_max;
    uint8_t *out = tp + ((size_t)f * n_thresh + t) * k_max;
    // bit m of `open`: ground truth 32 m + lane is still unmatched
    const int mine = g > lane ? (g - lane + 31) >> 5 : 0;
    uint32_t open = mine >= 32 ? 0xffffffffu : (1u << mine) - 1u;
    int base = 0;
    for (; base < k; base += 32) {
        const int i0 = base + lane;
        const bool flagged = i0 < k && flag[i0] != 0;
        uint32_t todo = __ballot_sync(0xffffffffu, flagged);
        uint8_t hit_mine = 0;
        while (todo) {
            const int s = __ffs(todo) - 1;
            todo &= todo - 1u;
            const float *row = iou + (size_t)(base + s) * g_max;
            float bv = -INFINITY;
            int bj = 0x7fffffff;   // none
#pragma unroll 4
            for (int m = 0; m < 32; ++m) {
                const int j = 32 * m + lane;
                if (j >= g) break;
                const float v = row[j];
                if (((open >> m) & 1u) && beats(v, j, bv, bj)) { bv = v; bj = j; }
            }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
                if (beats(ov, oj, bv, bj)) { bv = ov; bj = oj; }
            }
            // np.max(ious) < iou_thresh with the float32 max widened to double; NaN compares false -> TP
            const bool hit = bj != 0x7fffffff && !((double)bv < thr);
            if (hit) {
                if (lane == (bj & 31)) open &= ~(1u << (bj >> 5));
                if (lane == s) hit_mine = 1;
            }
        }
        if (i0 < k_max) out[i0] = hit_mine;
    }
    for (int i = base + lane; i < k_max; i += 32) out[i] = 0;   // padding rows beyond the count: no scan, stores only
}

}  // namespace evalm
}  // namespace gc

using namespace gc;

extern "C" size_t gc_eval_workspace_bytes(int n_frames, int k_max, int g_max) {
    if (n_frames < 1 || k_max < 1 || k_max > evalm::kMax || g_max < 1 || g_max > evalm::kMax) return 0;
    return evalm::carve(nullptr, n_frames, k_max, g_max).bytes;
}

extern "C" int gc_eval_match(const float *det_boxes, const float *det_scores, const int *det_counts, int k_max,
                             const float *gt_boxes, const int *gt_counts, int g_max, int n_frames, const double *iou_thresh,
                             int n_thresh, void *workspace, float *sorted_scores, uint8_t *tp, void *stream) {
    GC_REQUIRE(det_boxes && det_scores && det_counts && gt_boxes && gt_counts && iou_thresh && workspace && sorted_scores && tp,
               GC_EINVAL, "gc_eval_match: null pointer");
    GC_REQUIRE(n_frames >= 1 && n_frames <= 65535, GC_EINVAL, "gc_eval_match: n_frames must be in 1..65535");
    GC_REQUIRE(k_max >= 1 && k_max <= evalm::kMax, GC_EINVAL, "gc_eval_match: k_max must be in 1..%d", evalm::kMax);
    GC_REQUIRE(g_max >= 1 && g_max <= evalm::kMax, GC_EINVAL, "gc_eval_match: g_max must be in 1..%d", evalm::kMax);
    GC_REQUIRE(n_thresh >= 1 && n_thresh <= evalm::kMaxThresh, GC_EINVAL, "gc_eval_match: n_thresh must be in 1..%d",
               evalm::kMaxThresh);
    evalm::Thresholds th;
    th.min = iou_thresh[0];
    for (int t = 0; t < evalm::kMaxThresh; ++t) {
        th.v[t] = t < n_thresh ? iou_thresh[t] : 0.0;
        if (t < n_thresh) th.min = fmin(th.min, iou_thresh[t]);
    }
    cudaStream_t st = (cudaStream_t)stream;
    const evalm::Ws ws = evalm::carve(workspace, n_frames, k_max, g_max);
    evalm::k_eval_prep<<<n_frames, evalm::kMax, 0, st>>>(det_boxes, det_scores, det_counts, k_max, gt_boxes, gt_counts, g_max,
                                                         ws, sorted_scores);
    GC_LAUNCH_CHECK("k_eval_prep");
    const int pairs = k_max * g_max;
    evalm::k_eval_iou<<<dim3((pairs + 255) / 256, n_frames), 256, 0, st>>>(ws, k_max, g_max, th.min);
    GC_LAUNCH_CHECK("k_eval_iou");
    evalm::k_eval_match<<<n_frames, 32 * n_thresh, 0, st>>>(ws, k_max, g_max, th, n_thresh, tp);
    GC_LAUNCH_CHECK("k_eval_match");
    return GC_OK;
}
