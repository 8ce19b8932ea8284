// Shared device code of the warp+fusion kernels (affine_grid + grid_sample numerics).
//
// Numerics (SURVEY.md App. A.4/A.5): the base grid and the 2x3 affine are evaluated in float64 and only the
// resulting grid coordinate is rounded to float32 -- exactly what F.affine_grid(theta_f64).to(src) does
// (models/sub_modules/torch_transformation_utils.py:329-331).  Unnormalisation, floor, the four weights and
// the tap accumulation order follow ATen's grid_sampler_2d CUDA kernel (align_corners=False, zeros padding).
#pragma once
#include <type_traits>
#include <utility>

#include "common.cuh"

namespace gc {

constexpr int kMaxN = GC_MAX_AGENTS_PER_FRAME;

// ---- helpers of the TMA-staged kernels (warp_fuse_tile.cu, warp_fuse_persist.cu) ----
template <int kCount>
__device__ __forceinline__ void consumer_sync() {   // named barrier 1: consumer warps only
    asm volatile("bar.sync 1, %0;" ::"n"(kCount) : "memory");
}
// shared-memory accesses by 32-bit shared address + compile-time byte offset (folds into the LDS/STS immediate)
template <int OFF>
__device__ __forceinline__ float lds(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(addr), "n"(OFF));
    return v;
}
template <int OFF>
__device__ __forceinline__ void sts(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0+%1], %2;" ::"r"(addr), "n"(OFF), "f"(v) : "memory");
}
template <int... Is, class F>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, Is...>, F &&f) {
    (f(std::integral_constant<int, Is>{}), ...);
}
template <int N, class F>
__device__ __forceinline__ void static_for(F &&f) {   // f(std::integral_constant<int, i>) for i = 0 .. N-1
    static_for_impl(std::make_integer_sequence<int, N>{}, static_cast<F &&>(f));
}

// ATen linspace(-1,1,n) * (n-1)/n, evaluated in float64 (AffineGridGenerator.cpp: linspace_from_neg_one).
__host__ __device__ __forceinline__ double base_coord(int i, int n) {
    if (n <= 1) return 0.0;
    const double step = 2.0 / (double)(n - 1);
    const double v = (i < n / 2) ? (-1.0 + step * (double)i) : (1.0 - step * (double)(n - 1 - i));
    return v * (double)(n - 1) / (double)n;
}

struct Tap {
    float w_nw, w_ne, w_sw, w_se;
    int off;          // y0 * W + x0 (may be out of range; guarded by the valid bits)
    unsigned valid;   // bit0 nw, bit1 ne, bit2 sw, bit3 se; taps with zero weight are dropped
};

// theta: 6 doubles (row-major 2x3).  (xs, ys): float64 base grid coordinates of the output pixel.
__device__ __forceinline__ Tap make_tap(const double *__restrict__ th, double xs, double ys, int H, int W) {
    // bmm of [xs, ys, 1] with theta^T (float64), then .to(float32)
    const float gx = (float)(xs * th[0] + ys * th[1] + th[2]);
    const float gy = (float)(xs * th[3] + ys * th[4] + th[5]);
    // grid_sampler_unnormalize, align_corners=False: ((coord + 1) * size - 1) / 2
    const float ix = __fmaf_rn(gx + 1.0f, (float)W, -1.0f) * 0.5f;
    const float iy = __fmaf_rn(gy + 1.0f, (float)H, -1.0f) * 0.5f;
    const float fx = floorf(ix), fy = floorf(iy);
    Tap t;
    // nw = (ix_se - ix)(iy_se - iy), ne = (ix - ix_sw)(iy_sw - iy), sw = (ix_ne - ix)(iy - iy_ne), se = (ix - ix_nw)(iy - iy_nw)
    const float ex = (fx + 1.0f) - ix, wx = ix - fx;
    const float sy = (fy + 1.0f) - iy, ny_ = iy - fy;
    t.w_nw = ex * sy;
    t.w_ne = wx * sy;
    t.w_sw = ex * ny_;
    t.w_se = wx * ny_;
    // clamp before the int conversion so absurd coordinates stay defined; they are out of range anyway
    const int x0 = (int)fminf(fmaxf(fx, -2.0f), (float)W);
    const int y0 = (int)fminf(fmaxf(fy, -2.0f), (float)H);
    const bool xin0 = x0 >= 0 && x0 < W, xin1 = x0 + 1 >= 0 && x0 + 1 < W;
    const bool yin0 = y0 >= 0 && y0 < H, yin1 = y0 + 1 >= 0 && y0 + 1 < H;
    // a tap whose weight is exactly 0 contributes +-0 and can be skipped (features are finite)
    t.valid = ((xin0 && yin0 && t.w_nw != 0.0f) ? 1u : 0u) | ((xin1 && yin0 && t.w_ne != 0.0f) ? 2u : 0u) |
              ((xin0 && yin1 && t.w_sw != 0.0f) ? 4u : 0u) | ((xin1 && yin1 && t.w_se != 0.0f) ? 8u : 0u);
    t.off = y0 * W + x0;
    if (!(ix == ix) || !(iy == iy)) t.valid = 0;   // NaN transform
    return t;
}

// ATen order: out = 0; out += nw_val*nw; += ne; += sw; += se   (each a fused multiply-add under nvcc)
__device__ __forceinline__ float sample(const float *__restrict__ plane, const Tap &t, int W) {
    const float *p = plane + t.off;
    const float a = (t.valid & 1u) ? __ldg(p) : 0.0f;
    const float b = (t.valid & 2u) ? __ldg(p + 1) : 0.0f;
    const float c = (t.valid & 4u) ? __ldg(p + W) : 0.0f;
    const float d = (t.valid & 8u) ? __ldg(p + W + 1) : 0.0f;
    float acc = a * t.w_nw;
    acc = __fmaf_rn(b, t.w_ne, acc);
    acc = __fmaf_rn(c, t.w_sw, acc);
    acc = __fmaf_rn(d, t.w_se, acc);
    return acc;
}

}  // namespace gc
