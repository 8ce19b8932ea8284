// Convex-quadrilateral IoU in float64 for the rotated NMS (postprocess.cu) and the detection matching (eval.cu).
//
// Sutherland-Hodgman clipping of one bottom-face quad against the other, with the operation order of the oracle's
// gc_ref_quad_iou (oracle/nms_ref.c) and explicit roundings (no FMA contraction), so the float32 IoU is bit-identical
// to the oracle's.  The reference computes the same quantity with shapely polygons (utils/common_utils.py:230-270);
// parity with shapely's area is unpinned (DESIGN §5g).
#pragma once
#include <math.h>

namespace gc {
namespace riou {

__device__ __forceinline__ double dm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double da(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double ds(double a, double b) { return __dsub_rn(a, b); }

// signed area of the polygon p[0..n) of (x, y) pairs (shoelace, counter-clockwise positive)
static __device__ double poly_area(const double *p, int n) {
    double acc = 0.0;
    for (int i = 0; i < n; ++i) {
        const int j = (i + 1 == n) ? 0 : i + 1;
        acc = da(acc, ds(dm(p[2 * i], p[2 * j + 1]), dm(p[2 * j], p[2 * i + 1])));
    }
    return dm(0.5, acc);
}

static __device__ void load_ccw(const double *src, double *dst) {
    if (poly_area(src, 4) < 0.0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { dst[2 * i] = src[2 * (3 - i)]; dst[2 * i + 1] = src[2 * (3 - i) + 1]; }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) dst[i] = src[i];
    }
}

static __device__ double quad_intersection_area(const double *p_in, const double *q_in) {
    double p[8], q[8], bufa[32], bufb[32], side[16];
    load_ccw(p_in, p);
    load_ccw(q_in, q);
    double *in = bufa, *out = bufb;
    int n = 4;
    for (int i = 0; i < 8; ++i) in[i] = p[i];
    for (int e = 0; e < 4 && n > 0; ++e) {
        const int e1 = (e + 1) & 3;
        const double ax = q[2 * e], ay = q[2 * e + 1];
        const double ex = ds(q[2 * e1], ax), ey = ds(q[2 * e1 + 1], ay);
        for (int k = 0; k < n; ++k) side[k] = ds(dm(ex, ds(in[2 * k + 1], ay)), dm(ey, ds(in[2 * k], ax)));
        int m = 0;
        for (int k = 0; k < n; ++k) {
            const int k1 = (k + 1 == n) ? 0 : k + 1;
            const double sc = side[k], sn = side[k1];
            if (sc >= 0.0) { out[2 * m] = in[2 * k]; out[2 * m + 1] = in[2 * k + 1]; ++m; }
            if ((sc >= 0.0) != (sn >= 0.0)) {
                const double t = __ddiv_rn(sc, ds(sc, sn));
                out[2 * m] = da(in[2 * k], dm(t, ds(in[2 * k1], in[2 * k])));
                out[2 * m + 1] = da(in[2 * k + 1], dm(t, ds(in[2 * k1 + 1], in[2 * k + 1])));
                ++m;
            }
        }
        double *t2 = in; in = out; out = t2;
        n = m;
    }
    return n < 3 ? 0.0 : fabs(poly_area(in, n));
}

// inter / (|p| + |q| - inter), rounded once to float32 (0 / 0 = NaN for two zero-area quads, as in the oracle)
__device__ __forceinline__ float quad_iou(const double *p, const double *q) {
    const double inter = quad_intersection_area(p, q);
    const double uni = ds(da(fabs(poly_area(p, 4)), fabs(poly_area(q, 4))), inter);
    return (float)__ddiv_rn(inter, uni);
}

}  // namespace riou
}  // namespace gc
