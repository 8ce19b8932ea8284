// Implicit-GEMM building blocks on tcgen05 shared by message_extractor.cu and enhancer.cu:
//   k_me_to_nhwc : NCHW fp32 -> channel-last bf16 value + residual planes
//   k_me_pack    : weights -> bf16 (value [+ residual]) B operands in UMMA core-matrix order
//   k_me_conv    : 3x3 (plain or deformable) convolution / 1x1 GEMM over the planes, fp32 accumulation in TMEM
// See message_extractor.cu for the design notes and the measurements behind the layout choices.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"
#include "ptx.cuh"

namespace gc {
namespace me {

using namespace ptx;

constexpr int kPix = 128;            // pixels per CTA = M
constexpr int kThreads = 256;          // threads that stage operands and run the epilogue
// Plain (non-deformable) layers add one warp that only feeds the tensor core: it issues the weight (B) bulk copies one
// stage ahead and the MMAs, so the 256 operand threads never meet at a block-wide barrier inside the K loop.
__host__ __device__ constexpr int conv_block_threads(bool deform) { return deform ? kThreads : kThreads + 32; }
// Input channels per stage (SC / 16 MMAs of K = 16): 64 for the deformable layer, 32 for the offset layer (its value +
// residual planes double the operand bytes; with 64-channel stages only two CTAs fit an SM and the layer was latency
// bound on its load -> store -> barrier -> MMA chain: 305 us at 28 % issue-active).
// A operand plane: [SC/8 channel groups][128 pixels][8 bf16], the group stride padded by 16 (32) bytes so that the lanes
// that build one pixel store to different bank quads (measured without the pad: 8-way conflicts, 32 wavefronts per
// STS.128, 70 M conflicts per launch).  UMMA no-swizzle K-major: LBO = group stride, SBO = 128 B.
__host__ __device__ constexpr int a_group_bytes(int SC) { return kPix * 16 + (SC == 64 ? 16 : 32); }
__host__ __device__ constexpr int a_plane_bytes(int SC) { return (SC / 8) * a_group_bytes(SC); }
// MT = 128-pixel M tiles per CTA that share one B (weight) stage (plain layers only)
__host__ __device__ constexpr int conv_smem_bytes(int NOUT, bool split, int SC, int MT = 1) {
    return 2 * (split ? 2 : 1) * (MT * a_plane_bytes(SC) + SC * NOUT * 2);
}
constexpr int kScOffset = 32, kScDeform = 64;

// ------------------------------------------------------------------------------------------------
// weights [NOUT_real][C][3][3] f32 -> bf16 B operand, per stage (tap, 64-channel chunk):
//   [k8 = SC/8 channel groups][n8 = NOUT/8][8 rows n][8 bf16 k]     (rows >= NOUT_real are zero)
// ------------------------------------------------------------------------------------------------
//   split: every stage is followed by its residual plane  lo = bf16(w - float(bf16(w)))  (the "bf16x3" offset layer)
__device__ __forceinline__ float bf16_residual(float v) { return v - __bfloat162float(__float2bfloat16_rn(v)); }

static __global__ void k_me_pack(const float *__restrict__ w, int n_real, int NOUT, int C, int SC, int taps, int split,
                          uint4 *__restrict__ out) {
    const int chunks = C / SC, groups = SC / 8;
    const int per_stage = groups * NOUT;       // uint4 (8 k values of one row n) per stage and plane
    const int total = taps * chunks * per_stage;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int n = i % NOUT;                // i = ((stage * groups + k8) * (NOUT/8) + n8) * 8 + (n % 8)  with n = n8 * 8 + n % 8
    const int k8 = (i / NOUT) % groups;
    const int stage = i / per_stage;
    const int tap = stage / chunks, chunk = stage % chunks;
    uint32_t p[4], q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int c = chunk * SC + k8 * 8 + 2 * j + e;
            v[e] = n < n_real ? w[((size_t)n * C + c) * taps + tap] : 0.0f;
        }
        p[j] = pack_bf16(v[0], v[1]);
        q[j] = pack_bf16(bf16_residual(v[0]), bf16_residual(v[1]));
    }
    const int within = i - stage * per_stage;
    if (split) {
        out[(size_t)stage * 2 * per_stage + within] = make_uint4(p[0], p[1], p[2], p[3]);
        out[(size_t)stage * 2 * per_stage + per_stage + within] = make_uint4(q[0], q[1], q[2], q[3]);
    } else {
        out[i] = make_uint4(p[0], p[1], p[2], p[3]);
    }
}

// ------------------------------------------------------------------------------------------------
// x [A][C][HW] f32 (NCHW)  ->  channel-last bf16 planes  xh = bf16(x),  xl = bf16(x - xh)   [A][HW][C]
// so that a bilinear corner of 8 channels is ONE 16-byte load and the 8 lanes that sample a pixel read 128 contiguous
// bytes.  (Measured before: sampling NCHW fp32 directly made the deformable layer L1-gather bound -- 4 loads per
// (pixel, tap, channel), l1tex 76 % busy, 0.64 ms of the 0.94 ms call.)   grid = (HW/64, C/64, A), 256 threads.
// ------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
k_me_to_nhwc(const float *__restrict__ x, int C, int HW, uint4 *__restrict__ xh, uint4 *__restrict__ xl) {
    __shared__ float t[64][65];
    const int tid = threadIdx.x, p0 = blockIdx.x * 64, c0 = blockIdx.y * 64, a = blockIdx.z;
    const float *src = x + ((size_t)a * C + c0) * HW + p0;
    {
        const int p = tid & 63, c_base = tid >> 6;   // 16 independent loads in flight per thread
        float v[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = (p0 + p < HW) ? __ldg(src + (size_t)(c_base + 4 * k) * HW + p) : 0.0f;
#pragma unroll
        for (int k = 0; k < 16; ++k) t[c_base + 4 * k][p] = v[k];
    }
    __syncthreads();
    for (int i = tid; i < 64 * 8; i += 256) {
        const int p = i >> 3, g = i & 7;
        if (p0 + p >= HW) continue;
        float v[8], r[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { v[k] = t[g * 8 + k][p]; r[k] = bf16_residual(v[k]); }
        const size_t o = ((size_t)a * HW + p0 + p) * (C / 8) + c0 / 8 + g;
        xh[o] = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        xl[o] = make_uint4(pack_bf16(r[0], r[1]), pack_bf16(r[2], r[3]), pack_bf16(r[4], r[5]), pack_bf16(r[6], r[7]));
    }
}

__device__ __forceinline__ float bf_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }
// torchvision bilinear_interpolate: val = hh*hw*v1 + hh*lw*v2 + lh*hw*v3 + lh*lw*v4 (left to right), two channels
// (packed fp32: one FMUL2 + three FFMA2 for the two channels of a 32-bit word, same roundings as scalar fmaf)
__device__ __forceinline__ uint32_t lerp2(const float4 &w, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    float2 r = __fmul2_rn(make_float2(w.x, w.x), make_float2(bf_lo(a), bf_hi(a)));
    r = __ffma2_rn(make_float2(w.y, w.y), make_float2(bf_lo(b), bf_hi(b)), r);
    r = __ffma2_rn(make_float2(w.z, w.z), make_float2(bf_lo(c), bf_hi(c)), r);
    r = __ffma2_rn(make_float2(w.w, w.w), make_float2(bf_lo(d), bf_hi(d)), r);
    return pack_bf16(r.x, r.y);
}

// ------------------------------------------------------------------------------------------------
// 3x3 (deformable) convolution as a tcgen05 implicit GEMM.  grid = (H*W/128, n_agents), 256 threads.
//   xh, xl [A][HW][C] bf16 (k_me_to_nhwc); offset [A][18][H][W] f32 (DEFORM; channel 2k = dy, 2k+1 = dx of tap k);
//   wp: k_me_pack output;  out [A][n_store][H][W] f32 (+ bias);
//   tile_sums [A][tiles*4][NOUT] (DEFORM): channel sums over 32-pixel groups
// ------------------------------------------------------------------------------------------------
// TAPS = 9: 3x3 convolution; TAPS = 1: 1x1 (a plain GEMM over the channel-last planes; used by the Enhancer's linear
// layers).  EPI = 0: bias; EPI = 1: bias + exact GELU; EPI = 2: bias + GELU written channel-last (all NOUT columns);
// EPI = 3: bias + ReLU; EPI = 5: bias + ReLU written as channel-last bf16 value + residual planes (oh, ol).  c_in = channels contracted (<= C, the channel count of the planes);
// the n_store output channels go to planes out_ch_off .. of an [A][out_ch_total][HW] f32 tensor.
__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }

template <int NOUT, bool DEFORM, int SC, int TAPS = 9, int EPI = 0, int MT = 1>
__global__ void __launch_bounds__(conv_block_threads(DEFORM))
k_me_conv(const uint4 *__restrict__ xh, const uint4 *__restrict__ xl, const float *__restrict__ offset,
          const uint4 *__restrict__ wp, const float *__restrict__ bias, int C, int c_in, int H, int W, int n_store,
          int out_ch_total, int out_ch_off, float *__restrict__ out, float *__restrict__ tile_sums, int H_in = 0,
          int W_in = 0, int stride = 1, uint4 *__restrict__ oh = nullptr, uint4 *__restrict__ ol = nullptr, int up = 1,
          int up_dy = 0, int up_dx = 0) {
    // The plain (offset) layer runs as "bf16x3": A and B are split into a bf16 value and a bf16 residual and three MMAs
    // (hi*hi + lo*hi + hi*lo) rebuild ~16 mantissa bits, because its output positions the deformable layer's taps:
    // a bf16-only offset (rel. error 4e-3) moves a tap by 0.02 px at 5 px, which on high-frequency features costs
    // more accuracy than the deformable layer's own bf16 rounding.
    constexpr bool SPLIT = !DEFORM;
    constexpr int kPlanes = SPLIT ? 2 : 1;
    constexpr int kAGroup = a_group_bytes(SC), kABytes = a_plane_bytes(SC), kGroups = SC / 8;
    constexpr int kBBytes = SC * NOUT * 2 * kPlanes;
    static_assert(MT == 1 || (!DEFORM && MT == 2 && NOUT * MT <= 512), "two M tiles per CTA: plain layers, <= 512 TMEM columns");
    constexpr int kATile = kABytes * kPlanes;   // one 128-pixel tile: value (+ residual) plane
    constexpr int kAStage = kATile * MT;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *a_s = smem;                      // [2][kPlanes][kABytes]
    uint8_t *b_s = smem + 2 * kAStage;        // [2][kPlanes][SC * NOUT * 2]
    __shared__ __align__(8) uint64_t s_empty[2], s_done, s_full[2], s_afull[2];
    __shared__ uint32_t s_tmem;
    // B stages arrive by one 1-D bulk copy (TMA) per stage instead of LDG + STS by every thread: the packed weights of a
    // stage are kBBytes contiguous bytes in global memory and land in the same order in shared memory.
    constexpr bool kBulkB = true;
    __shared__ __align__(16) int4 s_o[kPix];      // pixel index (y*W + x) of the four bilinear corners of the tap
    __shared__ __align__(16) float4 s_w[kPix];    // their weights (0 for a corner outside the image)

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the role branches
    const int agent = blockIdx.y, tile = blockIdx.x;
    const int HW = H * W;
    const int chunks = c_in / SC, stages = TAPS * chunks;
    const int C8 = C / 8;

    if (warp == 0) tmem_alloc<NOUT * MT>(&s_tmem);
    if (tid == 32) {
        mbar_init(smem_u32(&s_empty[0]), 1); mbar_init(smem_u32(&s_empty[1]), 1); mbar_init(smem_u32(&s_done), 1);
        mbar_init(smem_u32(&s_full[0]), 1); mbar_init(smem_u32(&s_full[1]), 1);
        mbar_init(smem_u32(&s_afull[0]), kThreads); mbar_init(smem_u32(&s_afull[1]), kThreads);
        mbar_init_fence();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const uint32_t a_base = smem_u32(a_s), b_base = smem_u32(b_s);
    constexpr uint32_t idesc = make_idesc(128, NOUT);
    // plain convolutions may be strided: H x W is the output grid, Hi x Wi the input grid the planes are laid out over
    const int Hi = H_in > 0 ? H_in : H, Wi = W_in > 0 ? W_in : W;
    const uint4 *xh_a = xh + (size_t)agent * Hi * Wi * C8;
    const uint4 *xl_a = xl + (size_t)agent * Hi * Wi * C8;

    if constexpr (!DEFORM) {
        // ---- plain 3x3 / 1x1 path: warp-specialised, no block-wide barrier in the K loop ----
        static_assert(SC == 32, "the plain path stages 32 channels (4 groups) per stage");
        constexpr uint32_t kBPlane = SC * NOUT * 2;
        if (warp == kThreads / 32) {
            // feeder warp (one elected lane): B(s+1) bulk copy as soon as its buffer is free, then the MMAs of stage s
            if (elect_one()) {
                bulk_load(smem_u32(b_s), wp, kBBytes, smem_u32(&s_full[0]));
                for (int s = 0; s < stages; ++s) {
                    const int b = s & 1;
                    if (s + 1 < stages) {
                        const int b1 = (s + 1) & 1;
                        if (s + 1 >= 2) mbar_wait(smem_u32(&s_empty[b1]), (uint32_t)(((s + 1) >> 1) - 1) & 1u);
                        bulk_load(smem_u32(b_s + b1 * kBBytes), wp + (size_t)(s + 1) * (kBBytes / 16), kBBytes, smem_u32(&s_full[b1]));
                    }
                    mbar_wait(smem_u32(&s_afull[b]), (uint32_t)(s >> 1) & 1u);
                    mbar_wait(smem_u32(&s_full[b]), (uint32_t)(s >> 1) & 1u);
                    tc_fence_after();
                    const uint32_t b_buf = b_base + (uint32_t)b * kBBytes;
#pragma unroll
                    for (int t = 0; t < MT; ++t) {
                        const uint32_t a_buf = a_base + (uint32_t)b * kAStage + (uint32_t)t * kATile, acc = tmem + (uint32_t)(t * NOUT);
#pragma unroll
                        for (int j = 0; j < SC / 16; ++j) {
                            const uint32_t a_off = (uint32_t)(2 * j) * (uint32_t)kAGroup, b_off = (uint32_t)(2 * j) * (NOUT * 16u);
                            const uint64_t a_hi = make_desc(a_buf + a_off, (uint32_t)kAGroup, 128u);
                            const uint64_t b_hi = make_desc(b_buf + b_off, NOUT * 16u, 128u);
                            const uint64_t a_lo = make_desc(a_buf + kABytes + a_off, (uint32_t)kAGroup, 128u);
                            const uint64_t b_lo = make_desc(b_buf + kBPlane + b_off, NOUT * 16u, 128u);
                            mma_bf16(acc, a_hi, b_hi, idesc, (s > 0 || j > 0) ? 1u : 0u);
                            mma_bf16(acc, a_lo, b_hi, idesc, 1u);
                            mma_bf16(acc, a_hi, b_lo, idesc, 1u);
                        }
                    }
                    mma_commit(smem_u32(&s_empty[b]));
                    if (s == stages - 1) mma_commit(smem_u32(&s_done));
                }
            }
        } else {
            // operand threads: two pixels (tid / 4 and 64 + tid / 4) of channel group tid & 3, value + residual plane;
            // the rows of stage s + 1 are in flight (registers) while stage s is stored
            const int g_loc = tid & 3;
            constexpr int kU = 2 * MT;      // pixels per thread: u * 64 + tid / 4 of the CTA's MT * 128 pixels
            int py[kU], px[kU];
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                const int pix = tile * (kPix * MT) + u * 64 + (tid >> 2);
                py[u] = pix / W;
                px[u] = pix - py[u] * W;
            }
            auto issue = [&](int s, uint4 (&q)[kU][2]) {
                const int tap = s / chunks, chunk = s - tap * chunks;
                const int ky = TAPS == 1 ? 1 : tap / 3, kx = TAPS == 1 ? 1 : tap - 3 * ky;
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int yy = py[u] * stride - 1 + ky, xx = px[u] * stride - 1 + kx;
                    const bool ok = yy >= 0 && yy < Hi && xx >= 0 && xx < Wi;
                    const size_t o = (size_t)(ok ? yy * Wi + xx : 0) * C8 + chunk * kGroups + g_loc;
                    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
                    q[u][0] = ok ? __ldg(xh_a + o) : z;
                    q[u][1] = ok ? __ldg(xl_a + o) : z;
                }
            };
            // four register sets rotate: the rows of stages s + 1 .. s + 3 are in flight while stage s is stored
            uint4 q0[kU][2], q1[kU][2], q2[kU][2], q3[kU][2];
            auto step = [&](int s, uint4 (&cur)[kU][2], uint4 (&ahead)[kU][2]) {
                if (s >= stages) return;
                const int b = s & 1;
                if (s + 3 < stages) issue(s + 3, ahead);
                if (s >= 2) mbar_wait(smem_u32(&s_empty[b]), (uint32_t)((s >> 1) - 1) & 1u);   // MMAs of stage s-2 retired
                uint8_t *dst = a_s + b * kAStage;
#pragma unroll
                for (int u = 0; u < kU; ++u) {   // pixel u * 64 + tid / 4 lives in tile u / 2, row (u % 2) * 64 + tid / 4
                    uint4 *d = reinterpret_cast<uint4 *>(dst + (u >> 1) * kATile + g_loc * kAGroup) + ((u & 1) * 64 + (tid >> 2));
                    d[0] = cur[u][0];
                    d[kABytes / 16] = cur[u][1];
                }
                fence_async_smem();
                mbar_arrive(smem_u32(&s_afull[b]));
            };
            issue(0, q0);
            if (stages > 1) issue(1, q1);
            if (stages > 2) issue(2, q2);
            for (int s = 0; s < stages; s += 4) {
                step(s, q0, q3);
                step(s + 1, q1, q0);
                step(s + 2, q2, q1);
                step(s + 3, q3, q2);
            }
        }
    } else
    for (int s = 0; s < stages; ++s) {
        const int b = s & 1;
        const int tap = s / chunks, chunk = s - tap * chunks;
        if (chunk == 0) {
            // sampling position of every pixel of the tile for this tap (torchvision deformable_im2col /
            // bilinear_interpolate), once per tap, shared through s_o / s_w.  Every thread is past its staging of the
            // previous tap (barrier at the end of the previous stage), so the arrays can be overwritten.
            if (tid < kPix) {
                const int pix = tile * kPix + tid;
                const int py = pix / W, px = pix - py * W;
                const int ky = TAPS == 1 ? 1 : tap / 3, kx = TAPS == 1 ? 1 : tap - 3 * ky;
                int4 o = make_int4(0, 0, 0, 0);
                float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
                if (DEFORM) {
                    const float *op = offset + ((size_t)agent * 18 + 2 * tap) * HW + pix;
                    const float hh_ = (float)(py - 1 + ky) + __ldg(op);
                    const float ww_ = (float)(px - 1 + kx) + __ldg(op + HW);
                    const bool inside = hh_ > -1.0f && hh_ < (float)H && ww_ > -1.0f && ww_ < (float)W;
                    const float hf = floorf(hh_), wf = floorf(ww_);
                    const int hl = (int)hf, wl = (int)wf, hh = hl + 1, wh = wl + 1;
                    const float lh = hh_ - hf, lw = ww_ - wf, uh = 1.0f - lh, uw = 1.0f - lw;
                    const bool t_ok = inside && hl >= 0, b_ok = inside && hh <= H - 1;
                    const bool l_ok = wl >= 0, r_ok = wh <= W - 1;
                    const int hlc = min(max(hl, 0), H - 1), hhc = min(max(hh, 0), H - 1);
                    const int wlc = min(max(wl, 0), W - 1), whc = min(max(wh, 0), W - 1);
                    o = make_int4(hlc * W + wlc, hlc * W + whc, hhc * W + wlc, hhc * W + whc);
                    w.x = (t_ok && l_ok) ? uh * uw : 0.0f;
                    w.y = (t_ok && r_ok) ? uh * lw : 0.0f;
                    w.z = (b_ok && l_ok) ? lh * uw : 0.0f;
                    w.w = (b_ok && r_ok) ? lh * lw : 0.0f;
                } else {
                    const int yy = py * stride - 1 + ky, xx = px * stride - 1 + kx;
                    const bool ok = yy >= 0 && yy < Hi && xx >= 0 && xx < Wi;
                    o.x = ok ? yy * Wi + xx : 0;
                    w.x = ok ? 1.0f : 0.0f;
                }
                s_o[tid] = o;
                s_w[tid] = w;
            }
            __syncthreads();
        }
        if (s >= 2) mbar_wait(smem_u32(&s_empty[b]), (uint32_t)((s >> 1) - 1) & 1u);   // MMAs of stage s-2 retired
        // ---- B stage: kBBytes contiguous bytes of the packed weights; the loads are issued here and stored after the
        // first batch of A loads is in flight (one round trip instead of two or three) ----
        constexpr int kBIter = kBulkB ? 1 : (kBBytes / 16 + kThreads - 1) / kThreads;
        uint4 bq[kBIter];
        if (kBulkB) {
            if (tid == 0) bulk_load(smem_u32(b_s + b * kBBytes), wp + (size_t)s * (kBBytes / 16), kBBytes, smem_u32(&s_full[b]));
        } else {
            const uint4 *src = wp + (size_t)s * (kBBytes / 16);
#pragma unroll
            for (int i = 0; i < kBIter; ++i)
                bq[i] = (i * kThreads + tid < kBBytes / 16) ? __ldg(src + i * kThreads + tid) : make_uint4(0u, 0u, 0u, 0u);
        }
        // ---- A stage: 128 pixels x 8 channel groups = 1024 16-byte rows, four per thread.  The eight lanes of a pixel
        // read 128 contiguous bytes per corner (one full line; spreading a warp over 8 pixels x 4 groups instead was
        // measured 1.9x slower: twice the L1 tags per request) ----
        {
            uint8_t *dst = a_s + b * kAStage;
            const int g_loc = tid & (kGroups - 1);
            const int cg = chunk * kGroups + g_loc;
#pragma unroll
            for (int pass = 0; pass < kGroups / 2; pass += 2) {
                uint4 q[2][4];
                float4 w[2];
                int p[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    p[u] = ((pass + u) * kThreads + tid) / kGroups;
                    const int4 o = s_o[p[u]];
                    w[u] = s_w[p[u]];
                    if (DEFORM) {
                        q[u][0] = __ldg(xh_a + (size_t)o.x * C8 + cg);
                        q[u][1] = __ldg(xh_a + (size_t)o.y * C8 + cg);
                        q[u][2] = __ldg(xh_a + (size_t)o.z * C8 + cg);
                        q[u][3] = __ldg(xh_a + (size_t)o.w * C8 + cg);
                    } else {
                        q[u][0] = __ldg(xh_a + (size_t)o.x * C8 + cg);
                        q[u][1] = __ldg(xl_a + (size_t)o.x * C8 + cg);
                    }
                }
                if (!kBulkB && pass == 0) {
                    uint4 *bd = reinterpret_cast<uint4 *>(b_s + b * kBBytes);
#pragma unroll
                    for (int i = 0; i < kBIter; ++i)
                        if (i * kThreads + tid < kBBytes / 16) bd[i * kThreads + tid] = bq[i];
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    uint4 *d = reinterpret_cast<uint4 *>(dst + g_loc * kAGroup) + p[u];
                    if (DEFORM) {
                        d[0] = make_uint4(lerp2(w[u], q[u][0].x, q[u][1].x, q[u][2].x, q[u][3].x),
                                          lerp2(w[u], q[u][0].y, q[u][1].y, q[u][2].y, q[u][3].y),
                                          lerp2(w[u], q[u][0].z, q[u][1].z, q[u][2].z, q[u][3].z),
                                          lerp2(w[u], q[u][0].w, q[u][1].w, q[u][2].w, q[u][3].w));
                    } else {
                        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
                        const bool ok = w[u].x != 0.0f;
                        d[0] = ok ? q[u][0] : z;
                        d[kABytes / 16] = ok ? q[u][1] : z;
                    }
                }
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp == 0 && elect_one()) {
            if (kBulkB) mbar_wait(smem_u32(&s_full[b]), (uint32_t)(s >> 1) & 1u);   // the stage's weights have landed
            tc_fence_after();
            const uint32_t a_buf = a_base + (uint32_t)b * kAStage, b_buf = b_base + (uint32_t)b * kBBytes;
            constexpr uint32_t kBPlane = SC * NOUT * 2;
#pragma unroll
            for (int j = 0; j < SC / 16; ++j) {   // K = 16: channel groups 2j and 2j+1
                const uint32_t a_off = (uint32_t)(2 * j) * (uint32_t)kAGroup, b_off = (uint32_t)(2 * j) * (NOUT * 16u);
                const uint64_t a_hi = make_desc(a_buf + a_off, (uint32_t)kAGroup, 128u);
                const uint64_t b_hi = make_desc(b_buf + b_off, NOUT * 16u, 128u);
                mma_bf16(tmem, a_hi, b_hi, idesc, (s > 0 || j > 0) ? 1u : 0u);
                if (SPLIT) {
                    const uint64_t a_lo = make_desc(a_buf + kABytes + a_off, (uint32_t)kAGroup, 128u);
                    const uint64_t b_lo = make_desc(b_buf + kBPlane + b_off, NOUT * 16u, 128u);
                    mma_bf16(tmem, a_lo, b_hi, idesc, 1u);
                    mma_bf16(tmem, a_hi, b_lo, idesc, 1u);
                }
            }
            mma_commit(smem_u32(&s_empty[b]));
            if (s == stages - 1) mma_commit(smem_u32(&s_done));
        }
    }
    mbar_wait(smem_u32(&s_done), 0u);
    tc_fence_after();

    // ---- epilogue: warp w reads TMEM lanes 32 (w % 4) .. +31 (= pixels) and columns (w / 4) * NOUT/2 .. ----
    if (warp < kThreads / 32)
#pragma unroll 1
    for (int mt = 0; mt < MT; ++mt) {
        const int q = warp & 3, ch0 = (warp >> 2) * (NOUT / 2);
        const int p_out = tile * (kPix * MT) + mt * kPix + q * 32 + lane;
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(mt * NOUT + ch0);
        // NCHW stores may be "pixel-shuffled": output pixel (y * up + up_dy, x * up + up_dx) of an up-sampled grid -- one
        // phase of a ConvTranspose2d with kernel == stride == up evaluated as a 1x1 GEMM over the input pixels
        const int pyo = p_out / W, pxo = p_out - pyo * W;
        const size_t hw_store = (size_t)HW * up * up;
        const size_t p_store = (size_t)(pyo * up + up_dy) * (W * up) + pxo * up + up_dx;
#pragma unroll
        for (int c16 = 0; c16 < NOUT / 2; c16 += 16) {
            float v[16];
            tmem_ld16(taddr + (uint32_t)c16, v);
            if (EPI == 5) {   // bias + ReLU -> channel-last bf16 value + residual planes [A][HW * up * up][out_ch_total]: the
                              // next layer's A operand, no fp32 NCHW round trip and no layout conversion between layers
                uint32_t h[8], l[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float a = fmaxf(v[2 * i] + (bias ? __ldg(bias + ch0 + c16 + 2 * i) : 0.0f), 0.0f);
                    const float b = fmaxf(v[2 * i + 1] + (bias ? __ldg(bias + ch0 + c16 + 2 * i + 1) : 0.0f), 0.0f);
                    h[i] = pack_bf16(a, b);
                    l[i] = pack_bf16(bf16_residual(a), bf16_residual(b));
                }
                if (ch0 + c16 < n_store) {
                    const size_t o = ((size_t)agent * hw_store + p_store) * (out_ch_total >> 3) + ((out_ch_off + ch0 + c16) >> 3);
                    oh[o] = make_uint4(h[0], h[1], h[2], h[3]); oh[o + 1] = make_uint4(h[4], h[5], h[6], h[7]);
                    ol[o] = make_uint4(l[0], l[1], l[2], l[3]); ol[o + 1] = make_uint4(l[4], l[5], l[6], l[7]);
                }
                continue;
            }
            if (EPI == 2) {   // bias + GELU, fp32 channel-last [A][HW][out_ch_total]: 64 contiguous bytes per lane
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = gelu_erf(v[i] + (bias ? __ldg(bias + ch0 + c16 + i) : 0.0f));
                float4 *dst = reinterpret_cast<float4 *>(out + ((size_t)agent * HW + p_out) * out_ch_total + out_ch_off + ch0 + c16);
#pragma unroll
                for (int i = 0; i < 4; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                continue;
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int ch = ch0 + c16 + i;
                if (ch < n_store) {
                    float r = v[i] + (bias ? __ldg(bias + ch) : 0.0f);
                    if (EPI == 1) r = gelu_erf(r);
                    if (EPI == 3) r = fmaxf(r, 0.0f);
                    out[((size_t)agent * out_ch_total + out_ch_off + ch) * hw_store + p_store] = r;
                    if (DEFORM) {
                        float t = r;
#pragma unroll
                        for (int d = 16; d >= 1; d >>= 1) t += __shfl_xor_sync(0xffffffffu, t, d);
                        if (lane == 0) tile_sums[((size_t)agent * gridDim.x * 4 + tile * 4 + q) * NOUT + ch] = t;
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free<NOUT * MT>(tmem);
}

}  // namespace me
}  // namespace gc
