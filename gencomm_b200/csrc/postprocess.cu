// Decode + rotated NMS of the detector heads (SURVEY.md 8f rank 3): VoxelPostprocessor.post_process
// (opencood/data_utils/post_processor/voxel_postprocessor.py:1084-1244) for the ego output of an intermediate-fusion
// model, one CTA chain per frame, no host round trip (the reference copies the candidates to the host and runs a
// Python / shapely O(K^2) loop, utils/box_utils.py:915-960).
//
//   k_post_decode : one thread per anchor: sigmoid(cls) > score_threshold -> delta_to_boxes3d (:1351-1396), direction
//                   classifier fix (:1156-1172), boxes_to_corners_3d + project_box3d (box_utils.py:152-203, :278-316),
//                   remove_large_pred_bbx / remove_bbx_abnormal_z (:1062-1112); survivors append a 64-bit key
//                   (score bits << 32 | anchor index) to the frame's candidate list.
//   k_post_select : one CTA per frame: top-1000 keys by a 64-step bisection on the key value (keys are unique, so the
//                   k-th largest is exact and independent of the append order), bitonic sort of those <= 1024 keys in shared
//                   memory, geometry (bottom-face quad + AABB) of the sorted candidates.
//   k_post_iou    : 128 CTAs per frame: convex-quad IoU (Sutherland-Hodgman in float64, the same operation order as the
//                   oracle's nms_ref.c, no FMA contraction) into a 1000 x 1000 suppression bit matrix.  (First version: one
//                   CTA per frame did all of it -- 0.84 ms of a 4.3 ms single-frame detector pass.)
//   k_post_greedy : one CTA per frame: a one-warp greedy pass over the bit matrix, then mask_boxes_outside_range
//                   (box_utils.py:384-421) and an order-preserving store.
//
// HBM traffic is negligible (three head maps read once: 20 x H x W floats per frame); the work is latency-bound integer /
// geometry bookkeeping, sized to one CTA per frame so that a batch of frames fills the SMs.
#include <math.h>

#include "common.cuh"
#include "rotated_iou.cuh"

namespace gc {
namespace post {

constexpr int kTopMax = 1024;      // shared-memory sort width (>= params.top)
constexpr int kThreads = 1024;

struct Box {
    float c[8][3];   // projected corners
    float score;
    bool keep;       // passed the score threshold and the size / z filters
};

// fp32 arithmetic in torch's order, no FMA contraction
__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }

__device__ __forceinline__ float limit_period(float v, float offset, float period) {   // common_utils.py:112
    return sub(v, mul(floorf(add(__fdiv_rn(v, period), offset)), period));
}

__device__ Box decode(const float *__restrict__ cls, const float *__restrict__ reg, const float *__restrict__ dir,
                      const float *__restrict__ anchors, const float *__restrict__ tfm, int n, int A, int H, int W,
                      const gcPostParams &p) {
    Box b;
    const int a = n % A, hw = n / A;
    const int HW = H * W;
    const float logit = __ldg(cls + (size_t)a * HW + hw);
    b.score = 1.0f / (1.0f + expf(-logit));
    b.keep = b.score > p.score_threshold;
    if (!b.keep) return b;
    float an[7], d[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        an[k] = __ldg(anchors + (size_t)n * 7 + k);
        d[k] = __ldg(reg + (size_t)(a * 7 + k) * HW + hw);
    }
    const float ad = __fsqrt_rn(add(mul(an[4], an[4]), mul(an[5], an[5])));
    const float cx = add(mul(d[0], ad), an[0]), cy = add(mul(d[1], ad), an[1]), cz = add(mul(d[2], an[3]), an[2]);
    const float s3 = mul(expf(d[3]), an[3]), s4 = mul(expf(d[4]), an[4]), s5 = mul(expf(d[5]), an[5]);
    float yaw = add(d[6], an[6]);
    if (dir != nullptr) {
        int label = 0;
        float best = __ldg(dir + (size_t)(a * p.num_bins) * HW + hw);
        for (int j = 1; j < p.num_bins; ++j) {
            const float v = __ldg(dir + (size_t)(a * p.num_bins + j) * HW + hw);
            if (v > best) { best = v; label = j; }
        }
        const float period = (float)(2.0 * M_PI / (double)p.num_bins);
        const float rot = limit_period(sub(yaw, p.dir_offset), 0.0f, period);
        yaw = add(add(rot, p.dir_offset), mul(period, (float)label));
        yaw = limit_period(yaw, 0.5f, (float)(2.0 * M_PI));
    }
    // boxes_to_corners_3d: 'hwl' order stores (h, w, l) in slots 3..5; the template multiplies (l, w, h)
    const float L = p.order_hwl ? s5 : s3, Wd = s4, Hh = p.order_hwl ? s3 : s5;
    const float co = cosf(yaw), si = sinf(yaw);
    float zmin = INFINITY, zmax = -INFINITY, xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float tx = (k == 0 || k == 1 || k == 4 || k == 5) ? 0.5f : -0.5f;
        const float ty = (k == 1 || k == 2 || k == 5 || k == 6) ? 0.5f : -0.5f;
        const float tz = k >= 4 ? 0.5f : -0.5f;
        const float x = mul(L, tx), y = mul(Wd, ty), z = mul(Hh, tz);
        const float xr = add(add(mul(x, co), mul(y, -si)), cx);
        const float yr = add(add(mul(x, si), mul(y, co)), cy);
        const float zr = add(z, cz);
        float px = xr, py = yr, pz = zr;
        if (tfm != nullptr) {
            px = add(add(add(mul(tfm[0], xr), mul(tfm[1], yr)), mul(tfm[2], zr)), tfm[3]);
            py = add(add(add(mul(tfm[4], xr), mul(tfm[5], yr)), mul(tfm[6], zr)), tfm[7]);
            pz = add(add(add(mul(tfm[8], xr), mul(tfm[9], yr)), mul(tfm[10], zr)), tfm[11]);
        }
        b.c[k][0] = px; b.c[k][1] = py; b.c[k][2] = pz;
        xmin = fminf(xmin, px); xmax = fmaxf(xmax, px);
        ymin = fminf(ymin, py); ymax = fmaxf(ymax, py);
        zmin = fminf(zmin, pz); zmax = fmaxf(zmax, pz);
    }
    const float x_len = sub(xmax, xmin), y_len = sub(ymax, ymin);
    // remove_large_pred_bbx: "z_len" is computed from axis 1 again and only used as a truth value (box_utils.py:1084-1089)
    const bool k1 = x_len <= 6.0f && y_len <= 6.0f && y_len != 0.0f;
    const bool k2 = zmin >= -3.0f && zmax <= 1.0f;                                    // remove_bbx_abnormal_z
    b.keep = k1 && k2;
    return b;
}

__global__ void __launch_bounds__(256)
k_post_decode(const float *__restrict__ cls, const float *__restrict__ reg, const float *__restrict__ dir,
              const float *__restrict__ anchors, const float *__restrict__ tfm, int A, int H, int W, gcPostParams p,
              unsigned long long *__restrict__ keys, int *__restrict__ cand_count) {
    const int N = A * H * W, f = blockIdx.y;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const Box b = decode(cls + (size_t)f * N, reg + (size_t)f * N * 7, dir ? dir + (size_t)f * N * p.num_bins : nullptr, anchors,
                         tfm ? tfm + (size_t)f * 16 : nullptr, n, A, H, W, p);
    if (!b.keep) return;
    const int slot = atomicAdd(cand_count + f, 1);
    keys[(size_t)f * N + slot] = ((unsigned long long)__float_as_uint(b.score) << 32) | (unsigned)n;
}

using riou::quad_iou;   // rotated_iou.cuh: float64 convex clipping, bit-matched to oracle/nms_ref.c

// Per-frame workspace of the NMS chain (global memory, L2 resident)
struct NmsFrame {
    unsigned long long keys[kTopMax];   // sorted, largest first
    double quad[kTopMax][8];            // bottom-face corners 0..3 (x, y) of the sorted candidates
    double aabb[kTopMax][4];            // xmin, ymin, xmax, ymax (quick reject: disjoint boxes have IoU 0)
    uint32_t mask[kTopMax][32];         // suppression bits
    int m;                              // candidates entering the NMS
};

// ---- NMS 1/3: one CTA per frame: top-`top` keys, sorted, and their geometry ----
__global__ void __launch_bounds__(kThreads)
k_post_select(const float *__restrict__ cls, const float *__restrict__ reg, const float *__restrict__ dir,
              const float *__restrict__ anchors, const float *__restrict__ tfm, int A, int H, int W, gcPostParams p,
              const unsigned long long *__restrict__ keys_all, const int *__restrict__ cand_count, NmsFrame *__restrict__ frames) {
    __shared__ unsigned long long s_keys[kTopMax];
    __shared__ int s_counter;
    const int N = A * H * W, f = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const unsigned long long *keys = keys_all + (size_t)f * N;
    NmsFrame &fr = frames[f];
    const int n = min(cand_count[f], N);
    const int top = min(p.top, kTopMax);
    if (n == 0) {
        if (tid == 0) fr.m = 0;
        return;
    }
    // threshold key T: the top-th largest key (0 when everything fits)
    unsigned long long T = 0ull;
    if (n > top) {
        unsigned long long lo = 0ull, hi = ~0ull;            // invariant: count(keys >= lo) >= top
        while (lo < hi) {
            const unsigned long long mid = lo + ((hi - lo) >> 1) + 1ull;
            if (tid == 0) s_counter = 0;
            __syncthreads();
            int c = 0;
            for (int i = tid; i < n; i += kThreads) c += keys[i] >= mid;
            for (int o = 16; o >= 1; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            if (lane == 0 && c) atomicAdd(&s_counter, c);
            __syncthreads();
            const int total = s_counter;
            __syncthreads();
            if (total >= top) lo = mid; else hi = mid - 1ull;
        }
        T = lo;
    }
    // gather the keys >= T (exactly min(n, top): keys are unique) and sort them, largest first
    if (tid == 0) s_counter = 0;
    s_keys[tid] = 0ull;
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
        const unsigned long long k = keys[i];
        if (k >= T) {
            const int slot = atomicAdd(&s_counter, 1);
            if (slot < kTopMax) s_keys[slot] = k;
        }
    }
    __syncthreads();
    const int m = min(min(s_counter, top), n);
    for (int k = 2; k <= kTopMax; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            const int partner = tid ^ j;
            if (partner > tid) {
                const unsigned long long x = s_keys[tid], y = s_keys[partner];
                const bool desc = (tid & k) == 0;
                if (desc ? x < y : x > y) { s_keys[tid] = y; s_keys[partner] = x; }
            }
            __syncthreads();
        }
    }
    fr.keys[tid] = s_keys[tid];
    if (tid == 0) fr.m = m;
    if (tid < m) {
        const Box b = decode(cls + (size_t)f * N, reg + (size_t)f * N * 7, dir ? dir + (size_t)f * N * p.num_bins : nullptr, anchors,
                             tfm ? tfm + (size_t)f * 16 : nullptr, (int)(s_keys[tid] & 0xffffffffull), A, H, W, p);
        double xmin = INFINITY, ymin = INFINITY, xmax = -INFINITY, ymax = -INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double x = (double)b.c[k][0], y = (double)b.c[k][1];
            fr.quad[tid][2 * k] = x; fr.quad[tid][2 * k + 1] = y;
            xmin = fmin(xmin, x); xmax = fmax(xmax, x); ymin = fmin(ymin, y); ymax = fmax(ymax, y);
        }
        fr.aabb[tid][0] = xmin; fr.aabb[tid][1] = ymin; fr.aabb[tid][2] = xmax; fr.aabb[tid][3] = ymax;
    }
}

// ---- NMS 2/3: suppression bits on a many-CTA grid: mask[i][w] bit j = IoU(i, 32 w + j) > nms_thresh for 32 w + j > i ----
__global__ void __launch_bounds__(256)
k_post_iou(NmsFrame *__restrict__ frames, float nms_thresh) {
    NmsFrame &fr = frames[blockIdx.y];
    const int m = fr.m;
    const int task = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = task >> 5, w = task & 31;
    if (i >= m) return;
    uint32_t bits = 0u;
    if (32 * w + 31 > i && 32 * w < m) {
        double qi[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) qi[k] = fr.quad[i][k];
        const double ax0 = fr.aabb[i][0], ay0 = fr.aabb[i][1], ax1 = fr.aabb[i][2], ay1 = fr.aabb[i][3];
        for (int j = max(32 * w, i + 1); j < min(32 * w + 32, m); ++j) {
            if (fr.aabb[j][0] > ax1 || fr.aabb[j][2] < ax0 || fr.aabb[j][1] > ay1 || fr.aabb[j][3] < ay0) continue;
            double qj[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) qj[k] = fr.quad[j][k];
            if (quad_iou(qi, qj) > nms_thresh) bits |= 1u << (j & 31);
        }
    }
    fr.mask[i][w] = bits;
}

// ---- NMS 3/3: one CTA per frame: greedy pass (one warp), range mask, order-preserving store ----
__global__ void __launch_bounds__(kThreads)
k_post_greedy(const float *__restrict__ cls, const float *__restrict__ reg, const float *__restrict__ dir,
              const float *__restrict__ anchors, const float *__restrict__ tfm, int A, int H, int W, gcPostParams p,
              const NmsFrame *__restrict__ frames, float *__restrict__ boxes_out, float *__restrict__ scores_out,
              int *__restrict__ counts_out) {
    __shared__ int s_pick[kTopMax];
    __shared__ int s_warp_cnt[32];
    __shared__ int s_n_pick;
    const int N = A * H * W, f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const NmsFrame &fr = frames[f];
    const int m = fr.m;
    if (m == 0) {
        if (tid == 0) counts_out[f] = 0;
        return;
    }
    const int words = (m + 31) >> 5;
    if (warp == 0) {   // lane l owns removed-word l; mask rows are prefetched eight at a time
        uint32_t removed = 0u;
        int np = 0;
        for (int base = 0; base < m; base += 8) {
            uint32_t row[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) row[u] = (base + u < m && lane < words) ? fr.mask[base + u][lane] : 0u;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = base + u;
                if (i >= m) break;
                const uint32_t r = __shfl_sync(0xffffffffu, removed, i >> 5);
                if (!((r >> (i & 31)) & 1u)) {
                    if (lane == 0) s_pick[np] = i;
                    ++np;
                    removed |= row[u];
                }
            }
        }
        if (lane == 0) s_n_pick = np;
    }
    __syncthreads();
    // range mask (all 8 corners inside gt_range) and order-preserving store
    const int np = s_n_pick;
    Box b;
    bool ok = false;
    if (tid < np) {
        b = decode(cls + (size_t)f * N, reg + (size_t)f * N * 7, dir ? dir + (size_t)f * N * p.num_bins : nullptr, anchors,
                   tfm ? tfm + (size_t)f * 16 : nullptr, (int)(fr.keys[s_pick[tid]] & 0xffffffffull), A, H, W, p);
        ok = true;
#pragma unroll
        for (int k = 0; k < 8; ++k)
#pragma unroll
            for (int ax = 0; ax < 3; ++ax)
                ok = ok && (double)b.c[k][ax] >= p.gt_range[ax] && (double)b.c[k][ax] <= p.gt_range[3 + ax];
    }
    const uint32_t ballot = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) s_warp_cnt[warp] = __popc(ballot);
    __syncthreads();
    int offset = 0, total = 0;
    for (int w2 = 0; w2 < 32; ++w2) {
        const int c = s_warp_cnt[w2];
        if (w2 < warp) offset += c;
        total += c;
    }
    if (ok) {
        const int pos = offset + __popc(ballot & ((1u << lane) - 1u));
        float *dst = boxes_out + ((size_t)f * p.top + pos) * 24;
#pragma unroll
        for (int k = 0; k < 8; ++k) { dst[3 * k] = b.c[k][0]; dst[3 * k + 1] = b.c[k][1]; dst[3 * k + 2] = b.c[k][2]; }
        scores_out[(size_t)f * p.top + pos] = b.score;
    }
    if (tid == 0) counts_out[f] = total;
}

}  // namespace post
}  // namespace gc

using namespace gc;

extern "C" size_t gc_postprocess_workspace_bytes(int n_frames, int n_anchors) {
    if (n_frames <= 0 || n_anchors <= 0) return 0;
    return align_up((size_t)n_frames * n_anchors * 8, 256) + align_up((size_t)n_frames * 4, 256) +
           align_up((size_t)n_frames * sizeof(post::NmsFrame), 256);
}

extern "C" int gc_postprocess(const float *cls, const float *reg, const float *dir, const float *anchors, const float *tfm,
                              int n_frames, int A, int H, int W, const gcPostParams *params, void *workspace, float *boxes,
                              float *scores, int *counts, void *stream) {
    GC_REQUIRE(n_frames >= 0 && n_frames <= 65535, GC_EINVAL, "gc_postprocess: bad frame count");
    if (n_frames == 0) return GC_OK;
    GC_REQUIRE(cls && reg && anchors && params && workspace && boxes && scores && counts, GC_EINVAL,
               "gc_postprocess: null pointer");
    GC_REQUIRE(A > 0 && H > 0 && W > 0 && (long long)A * H * W < (1ll << 31), GC_EINVAL, "gc_postprocess: bad head shape");
    GC_REQUIRE(params->top > 0 && params->top <= post::kTopMax, GC_EUNSUPPORTED,
               "gc_postprocess: top must be in 1..%d (the reference uses 1000)", post::kTopMax);
    GC_REQUIRE(dir == nullptr || params->num_bins >= 1, GC_EINVAL, "gc_postprocess: num_bins must be >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    const int N = A * H * W;
    char *ws = (char *)workspace;
    unsigned long long *keys = (unsigned long long *)ws;
    ws += align_up((size_t)n_frames * N * 8, 256);
    int *cand = (int *)ws;
    ws += align_up((size_t)n_frames * 4, 256);
    post::NmsFrame *frames = (post::NmsFrame *)ws;
    cudaError_t e = cudaMemsetAsync(cand, 0, (size_t)n_frames * 4, st);
    GC_REQUIRE(e == cudaSuccess, (int)e, "gc_postprocess: memset: %s", cudaGetErrorString(e));
    post::k_post_decode<<<dim3((N + 255) / 256, n_frames), 256, 0, st>>>(cls, reg, dir, anchors, tfm, A, H, W, *params, keys, cand);
    GC_LAUNCH_CHECK("k_post_decode");
    post::k_post_select<<<n_frames, post::kThreads, 0, st>>>(cls, reg, dir, anchors, tfm, A, H, W, *params, keys, cand, frames);
    GC_LAUNCH_CHECK("k_post_select");
    post::k_post_iou<<<dim3(post::kTopMax * 32 / 256, n_frames), 256, 0, st>>>(frames, params->nms_thresh);
    GC_LAUNCH_CHECK("k_post_iou");
    post::k_post_greedy<<<n_frames, post::kThreads, 0, st>>>(cls, reg, dir, anchors, tfm, A, H, W, *params, frames, boxes, scores,
                                                           counts);
    GC_LAUNCH_CHECK("k_post_greedy");
    return GC_OK;
}
