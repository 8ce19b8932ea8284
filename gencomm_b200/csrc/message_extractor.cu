// MessageExtractorv2 for sm_100a (SURVEY.md section 8f, rank 1): the module that turns an agent's BEV feature into the
// 2-channel message GenComm's sampler is conditioned on.
//
// Replaces (paths relative to /root/reference/opencood):
//   models/gencomm_modules/message_extractor_v2.py:70-120  (BEVDeformableExtractor / MessageExtractorv2)
//     offset1 = Conv2d(C -> 18, 3x3)            :74,  :97
//     dcn1    = torchvision DeformConv2d(C -> 64, 3x3, padding 1)   :78, :101   (deformable im2col + GEMM)
//     attn    = AvgPool -> 1x1 (64 -> 32) -> ReLU -> 1x1 (32 -> 64) -> Sigmoid   :88-94, :108
//     fuse    = 1x1 (64 -> 64) -> ReLU -> 1x1 (64 -> 2)                            :82-86, :111
//
// Both 3x3 convolutions are real dense contractions (K = 9 C = 1152 at C = 128): they run as ONE tcgen05 implicit-GEMM
// kernel template, k_me_conv<NOUT, DEFORM>:
//   * A pre-pass writes the features once as channel-last bf16 (value + residual planes).
//   * CTA = 128 consecutive pixels (M = 128) of one agent, 256 threads.  Per tap the four bilinear corners + weights
//     of every pixel are evaluated once (torchvision's bilinear_interpolate, zero outside the image; the plain
//     convolution is the same code with one corner of weight 1).  Eight lanes then build one pixel's row of the A
//     operand: per corner ONE coalesced 16-byte load of 8 channels each, interpolation in fp32, rounding to bf16,
//     one 16-byte store into K-major no-swizzle core matrices -- the deformable im2col never exists in global memory.
//   * K is walked in stages of one tap x 64 channels (four K = 16 MMAs), double buffered: the gather of stage s+1
//     overlaps the MMAs of stage s; stage reuse is guarded by tcgen05.commit -> mbarrier.
//   * B operand: the weights, pre-packed once to bf16 core-matrix order (gc_me_pack_weights), 8 KB per stage from L2.
//   * D: fp32 accumulators in TMEM (NOUT columns), epilogue tcgen05.ld.32x32b (lane = pixel -> coalesced NCHW stores),
//     bias, and -- for the deformable layer -- the per-tile channel sums the average pool needs (deterministic order).
// The tail (global average pool -> squeeze/excite -> two 1x1 convolutions) is 1 % of the FLOPs: CUDA-core fp32 kernels,
// the excitation folded into the first 1x1's weights per agent (two threads per pixel with 32 accumulators each were
// measured slower: 117 -> 167 us, shared-memory weight reads lose their warp-wide broadcast).
//
// Arithmetic: bf16 operands, fp32 accumulation for the two 3x3 layers; everything else fp32.  Tolerance vs the fp32
// reference is written in tests/test_message_extractor_gpu.py.
#include <cuda_bf16.h>

#include <stdlib.h>

#include "common.cuh"
#include "conv_layer.cuh"
#include "implicit_gemm.cuh"

namespace gc {
namespace me {

// ------------------------------------------------------------------------------------------------
// offset1 fast path for W % 128 == 0 (every shipped configuration: 64 x 128 maps): a tile is 128 pixels of ONE image
// row, so the three taps kx = 0, 1, 2 of a kernel row are the same staged pixels shifted by one 16-byte operand row.
// Stage (ky, 32-channel chunk) = 130 pixels x0-1 .. x0+128 of input row y-1+ky, copied once from the channel-last
// planes (zero outside the image); the taps are addressed by moving the descriptor start by kx * 16 bytes (the conv_in
// scheme of denoiser_tc.cu).  3 x C/32 stages of 18 MMAs instead of 9 x C/32 stages of 6: a third of the loads, stores
// and barriers of the generic kernel (ncu: that one spends the offset layer waiting on its per-stage
// load -> store -> barrier -> MMA chain).  bf16x3 like the generic path.  grid = (H*W/128, n_agents), 256 threads.
// ------------------------------------------------------------------------------------------------
constexpr int kR3Pix = 130;
constexpr int kR3Group = kR3Pix * 16;                  // 2080 B = 32 (mod 128): the 4-lane pixel rows store conflict-free
constexpr int kR3Plane = 4 * kR3Group;
constexpr int kR3BBlk = 32 * 32 * 2 * 2;               // one tap's B: value + residual planes (= one packed stage, SC = 32)
constexpr int kR3Stage = 2 * kR3Plane + 3 * kR3BBlk;
constexpr int kR3Smem = 2 * kR3Stage;

__global__ void __launch_bounds__(kThreads)
k_me_offset_row3(const uint4 *__restrict__ xh, const uint4 *__restrict__ xl, const uint4 *__restrict__ wp,
                 const float *__restrict__ bias, int C, int H, int W, float *__restrict__ out) {
    constexpr int NOUT = 32, n_store = 18;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t s_empty[2], s_done;
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int agent = blockIdx.y, tile = blockIdx.x;
    const int HW = H * W, C8 = C / 8, chunks = C / 32, stages = 3 * chunks;
    const int pix0 = tile * kPix, py = pix0 / W, x0 = pix0 - py * W;

    if (warp == 0) tmem_alloc<NOUT>(&s_tmem);
    if (tid == 32) {
        mbar_init(smem_u32(&s_empty[0]), 1); mbar_init(smem_u32(&s_empty[1]), 1); mbar_init(smem_u32(&s_done), 1);
        mbar_init_fence();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const uint32_t s_base = smem_u32(smem);
    constexpr uint32_t idesc = make_idesc(128, NOUT);
    const uint4 *xh_a = xh + (size_t)agent * HW * C8;
    const uint4 *xl_a = xl + (size_t)agent * HW * C8;

    for (int s = 0; s < stages; ++s) {
        const int b = s & 1;
        const int ky = s / chunks, chunk = s - ky * chunks;
        if (s >= 2) mbar_wait(smem_u32(&s_empty[b]), (uint32_t)((s >> 1) - 1) & 1u);   // MMAs of stage s-2 retired
        uint8_t *a_buf = smem + b * kR3Stage, *b_buf = a_buf + 2 * kR3Plane;
        // ---- all nine 16-byte loads of this thread are issued before the first store (one L2 round trip per stage;
        // load -> store pairs in sequence made the layer wait five round trips per stage: ncu, 57 % of the stall
        // samples on the STS instructions) ----
        {
            // B: the three taps of kernel row ky (4 KB each, value + residual): 768 rows, three per thread
            uint4 bq[3];
#pragma unroll
            for (int kx = 0; kx < 3; ++kx)
                bq[kx] = __ldg(wp + (size_t)((ky * 3 + kx) * chunks + chunk) * (kR3BBlk / 16) + tid);
            // A: 130 pixels x 4 channel groups, value and residual planes
            const int yy = py - 1 + ky;
            const bool row_ok = yy >= 0 && yy < H;
            const uint4 z = make_uint4(0u, 0u, 0u, 0u);
            uint4 hi[3], lo[3];
#pragma unroll
            for (int it = 0; it < 3; ++it) {
                const int item = it * kThreads + tid;
                const int p = item >> 2, g = item & 3, xx = x0 - 1 + p;
                const bool ok = item < kR3Pix * 4 && row_ok && xx >= 0 && xx < W;
                const size_t idx = ok ? (size_t)(yy * W + xx) * C8 + chunk * 4 + g : 0;
                hi[it] = ok ? __ldg(xh_a + idx) : z;
                lo[it] = ok ? __ldg(xl_a + idx) : z;
            }
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) reinterpret_cast<uint4 *>(b_buf)[kx * (kR3BBlk / 16) + tid] = bq[kx];
#pragma unroll
            for (int it = 0; it < 3; ++it) {
                const int item = it * kThreads + tid;
                if (item < kR3Pix * 4) {
                    uint4 *d = reinterpret_cast<uint4 *>(a_buf + (item & 3) * kR3Group) + (item >> 2);
                    d[0] = hi[it];
                    d[kR3Plane / 16] = lo[it];
                }
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (leader_of_warp0()) {
            tc_fence_after();
            const uint32_t a_addr = s_base + (uint32_t)b * kR3Stage, b_addr = a_addr + 2u * kR3Plane;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {   // K = 16: channel groups 2j and 2j+1
                    const uint32_t a_off = (uint32_t)(2 * j) * kR3Group + (uint32_t)kx * 16u;
                    const uint32_t b_off = (uint32_t)kx * kR3BBlk + (uint32_t)(2 * j) * (NOUT * 16u);
                    const uint64_t a_hi = make_desc(a_addr + a_off, kR3Group, 128u);
                    const uint64_t a_lo = make_desc(a_addr + kR3Plane + a_off, kR3Group, 128u);
                    const uint64_t b_hi = make_desc(b_addr + b_off, NOUT * 16u, 128u);
                    const uint64_t b_lo = make_desc(b_addr + kR3BBlk / 2 + b_off, NOUT * 16u, 128u);
                    mma_bf16(tmem, a_hi, b_hi, idesc, (s > 0 || kx > 0 || j > 0) ? 1u : 0u);
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
    {
        const int q = warp & 3, ch0 = (warp >> 2) * (NOUT / 2);
        const int p_out = tile * kPix + q * 32 + lane;
        float v[16];
        tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)ch0, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int ch = ch0 + i;
            if (ch < n_store) out[((size_t)agent * n_store + ch) * HW + p_out] = v[i] + __ldg(bias + ch);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free<NOUT>(tmem);
}

// ------------------------------------------------------------------------------------------------
// tail parameters (device blob, floats), see include/gencomm_b200.h
// ------------------------------------------------------------------------------------------------
constexpr int kOffBias = 0;                      // offset1.bias [18]
constexpr int kDcnBias = 32;                     // dcn1.bias [64]
constexpr int kAttn1W = kDcnBias + 64;           // attn.1.weight [32][64]
constexpr int kAttn1B = kAttn1W + 32 * 64;       // attn.1.bias [32]
constexpr int kAttn2W = kAttn1B + 32;            // attn.3.weight [64][32]
constexpr int kAttn2B = kAttn2W + 64 * 32;       // attn.3.bias [64]
constexpr int kFuse1W = kAttn2B + 64;            // fuse.0.weight [64][64]
constexpr int kFuse1B = kFuse1W + 64 * 64;       // fuse.0.bias [64]
constexpr int kFuse2W = kFuse1B + 64;            // fuse.2.weight [2][64]
constexpr int kFuse2B = kFuse2W + 2 * 64;        // fuse.2.bias [2]
constexpr int kTailFloats = kFuse2B + 2 + 6;     // padded to a multiple of 8

// global average pool (fixed summation order) + squeeze/excite.  grid = n_agents, 64 threads.
__global__ void __launch_bounds__(64)
k_me_attn(const float *__restrict__ tile_sums, int groups, int HW, const float *__restrict__ prm, float *__restrict__ attn) {
    __shared__ float s_mean[64], s_hid[32];
    const int a = blockIdx.x, c = threadIdx.x;
    const float *ts = tile_sums + (size_t)a * groups * 64;
    float s = 0.0f;
    for (int g = 0; g < groups; ++g) s += ts[(size_t)g * 64 + c];
    s_mean[c] = s / (float)HW;
    __syncthreads();
    if (c < 32) {
        float h = prm[kAttn1B + c];
        for (int k = 0; k < 64; ++k) h = fmaf(prm[kAttn1W + c * 64 + k], s_mean[k], h);
        s_hid[c] = fmaxf(h, 0.0f);
    }
    __syncthreads();
    float z = prm[kAttn2B + c];
    for (int k = 0; k < 32; ++k) z = fmaf(prm[kAttn2W + c * 32 + k], s_hid[k], z);
    attn[a * 64 + c] = 1.0f / (1.0f + expf(-z));
}

// enhanced = b1 * attn; out = fuse.2(relu(fuse.0(enhanced))).  grid = (H*W/128, n_agents), 128 threads (thread = pixel).
// The excitation is folded into fuse.0's weights per agent: W'[o][c] = W[o][c] * attn[c].
__global__ void __launch_bounds__(128)
k_me_tail(const float *__restrict__ b1, const float *__restrict__ attn, const float *__restrict__ prm, int HW,
          float *__restrict__ out) {
    __shared__ __align__(16) float s_w[64][64];   // [c][o]
    __shared__ float s_b[64], s_w2[2][64];
    const int a = blockIdx.y, tid = threadIdx.x;
    for (int i = tid; i < 64 * 64; i += 128) {
        const int o = i >> 6, c = i & 63;
        s_w[c][o] = prm[kFuse1W + i] * attn[a * 64 + c];
    }
    if (tid < 64) { s_b[tid] = prm[kFuse1B + tid]; s_w2[0][tid] = prm[kFuse2W + tid]; s_w2[1][tid] = prm[kFuse2W + 64 + tid]; }
    __syncthreads();
    const int p = blockIdx.x * 128 + tid;
    if (p >= HW) return;
    float2 acc[32];   // packed fp32 (FFMA2): two output channels per instruction, same roundings as scalar fmaf
#pragma unroll
    for (int o = 0; o < 32; ++o) acc[o] = make_float2(0.0f, 0.0f);
    const float *src = b1 + (size_t)a * 64 * HW + p;
#pragma unroll 1
    for (int c0 = 0; c0 < 64; c0 += 8) {
        float v8[8];   // eight plane-strided loads in flight (two at a time left the kernel latency bound: 24 % issue-active)
#pragma unroll
        for (int k = 0; k < 8; ++k) v8[k] = __ldg(src + (size_t)(c0 + k) * HW);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float2 vv = make_float2(v8[k], v8[k]);
            const float4 *wr = reinterpret_cast<const float4 *>(&s_w[c0 + k][0]);
#pragma unroll
            for (int o4 = 0; o4 < 16; ++o4) {
                const float4 w = wr[o4];
                acc[2 * o4 + 0] = __ffma2_rn(make_float2(w.x, w.y), vv, acc[2 * o4 + 0]);
                acc[2 * o4 + 1] = __ffma2_rn(make_float2(w.z, w.w), vv, acc[2 * o4 + 1]);
            }
        }
    }
    float r0 = prm[kFuse2B], r1 = prm[kFuse2B + 1];
#pragma unroll
    for (int o = 0; o < 32; ++o) {
        const float h0 = fmaxf(acc[o].x + s_b[2 * o], 0.0f), h1 = fmaxf(acc[o].y + s_b[2 * o + 1], 0.0f);
        r0 = fmaf(s_w2[0][2 * o], h0, r0);
        r1 = fmaf(s_w2[1][2 * o], h0, r1);
        r0 = fmaf(s_w2[0][2 * o + 1], h1, r0);
        r1 = fmaf(s_w2[1][2 * o + 1], h1, r1);
    }
    out[((size_t)a * 2 + 0) * HW + p] = r0;
    out[((size_t)a * 2 + 1) * HW + p] = r1;
}

// The same tail with fuse.0 (64 -> 64) on the tensor cores: one M = 128 pixels, N = 64, K = 64 GEMM per CTA in
// "bf16x3" (value + residual planes of both operands, three MMAs per K = 16 step, ~16 mantissa bits), the excitation
// folded into the A operand, ReLU + fuse.2 (64 -> 2) in the TMEM epilogue.  Replaces 2048 FFMA2 + 1024 LDS per pixel
// (k_me_tail: 117 us, latency bound) by 12 MMAs per 128 pixels.  grid = (H*W/128, n_agents), 128 threads (thread = pixel).
constexpr int kTtGroup = kPix * 16 + 16;        // [8 channel groups][128 pixels][16 B], padded group stride
constexpr int kTtPlane = 8 * kTtGroup;
constexpr int kTtBPlane = 64 * 64 * 2;          // [8 k groups][64 n][16 B]
constexpr int kTtSmem = 2 * kTtPlane + 2 * kTtBPlane;

__global__ void __launch_bounds__(128)
k_me_tail_tc(const float *__restrict__ b1, const float *__restrict__ attn, const float *__restrict__ prm, int HW,
             float *__restrict__ out) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *a_hi = smem, *a_lo = smem + kTtPlane, *b_hi = smem + 2 * kTtPlane, *b_lo = b_hi + kTtBPlane;
    __shared__ __align__(8) uint64_t s_done;
    __shared__ uint32_t s_tmem;
    __shared__ float s_attn[64], s_b[64], s_w2[2][64];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int a = blockIdx.y, p = blockIdx.x * kPix + tid;

    if (warp == 0) tmem_alloc<64>(&s_tmem);
    if (tid == 32) {
        mbar_init(smem_u32(&s_done), 1);
        mbar_init_fence();
    }
    if (tid < 64) {
        s_attn[tid] = attn[a * 64 + tid];
        s_b[tid] = prm[kFuse1B + tid];
        s_w2[0][tid] = prm[kFuse2W + tid];
        s_w2[1][tid] = prm[kFuse2W + 64 + tid];
    }
    // B: fuse.0.weight [n][k] -> value / residual planes in core-matrix order [k8][n][8 k]
    for (int i = tid; i < 64 * 8; i += 128) {
        const int n = i & 63, k8 = i >> 6;
        const float4 w0 = __ldg(reinterpret_cast<const float4 *>(prm + kFuse1W + n * 64 + k8 * 8));
        const float4 w1 = __ldg(reinterpret_cast<const float4 *>(prm + kFuse1W + n * 64 + k8 * 8 + 4));
        const float v[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            h[j] = pack_bf16(v[2 * j], v[2 * j + 1]);
            l[j] = pack_bf16(bf16_residual(v[2 * j]), bf16_residual(v[2 * j + 1]));
        }
        reinterpret_cast<uint4 *>(b_hi)[k8 * 64 + n] = make_uint4(h[0], h[1], h[2], h[3]);
        reinterpret_cast<uint4 *>(b_lo)[k8 * 64 + n] = make_uint4(l[0], l[1], l[2], l[3]);
    }
    // A: this thread's pixel, 64 plane-strided loads in flight
    float x[64];
    {
        const float *src = b1 + (size_t)a * 64 * HW + (p < HW ? p : 0);
#pragma unroll
        for (int c = 0; c < 64; ++c) x[c] = __ldg(src + (size_t)c * HW);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float v0 = x[8 * g + 2 * j] * s_attn[8 * g + 2 * j], v1 = x[8 * g + 2 * j + 1] * s_attn[8 * g + 2 * j + 1];
            h[j] = pack_bf16(v0, v1);
            l[j] = pack_bf16(bf16_residual(v0), bf16_residual(v1));
        }
        reinterpret_cast<uint4 *>(a_hi + g * kTtGroup)[tid] = make_uint4(h[0], h[1], h[2], h[3]);
        reinterpret_cast<uint4 *>(a_lo + g * kTtGroup)[tid] = make_uint4(l[0], l[1], l[2], l[3]);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    const uint32_t tmem = s_tmem;
    if (leader_of_warp0()) {
        tc_fence_after();
        constexpr uint32_t idesc = make_idesc(128, 64);
        const uint32_t ah = smem_u32(a_hi), al = smem_u32(a_lo), bh = smem_u32(b_hi), bl = smem_u32(b_lo);
#pragma unroll
        for (int j = 0; j < 4; ++j) {   // K = 16: channel groups 2j and 2j+1
            const uint32_t a_off = (uint32_t)(2 * j) * kTtGroup, b_off = (uint32_t)(2 * j) * (64 * 16u);
            const uint64_t d_ah = make_desc(ah + a_off, kTtGroup, 128u), d_al = make_desc(al + a_off, kTtGroup, 128u);
            const uint64_t d_bh = make_desc(bh + b_off, 64 * 16u, 128u), d_bl = make_desc(bl + b_off, 64 * 16u, 128u);
            mma_bf16(tmem, d_ah, d_bh, idesc, j > 0 ? 1u : 0u);
            mma_bf16(tmem, d_al, d_bh, idesc, 1u);
            mma_bf16(tmem, d_ah, d_bl, idesc, 1u);
        }
        mma_commit(smem_u32(&s_done));
    }
    mbar_wait(smem_u32(&s_done), 0u);
    tc_fence_after();
    {
        const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
        float r0 = prm[kFuse2B], r1 = prm[kFuse2B + 1];
#pragma unroll
        for (int c16 = 0; c16 < 64; c16 += 16) {
            float v[16];
            tmem_ld16(taddr + (uint32_t)c16, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float h = fmaxf(v[i] + s_b[c16 + i], 0.0f);
                r0 = fmaf(s_w2[0][c16 + i], h, r0);
                r1 = fmaf(s_w2[1][c16 + i], h, r1);
            }
        }
        if (p < HW) {
            out[((size_t)a * 2 + 0) * HW + p] = r0;
            out[((size_t)a * 2 + 1) * HW + p] = r1;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free<64>(tmem);
}

struct Workspace {
    float *offset;      // [A][18][HW]
    float *b1;          // [A][64][HW]
    float *tile_sums;   // [A][HW/32][64]
    float *attn;        // [A][64]
    uint4 *xh, *xl;     // [A][HW][C] bf16: value and residual planes of the input, channel-last
    size_t bytes;
};
static Workspace carve(void *base, int A, int C, int HW) {
    Workspace w;
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align_up(bytes, 256);
        return (float *)p;
    };
    w.offset = take((size_t)A * 18 * HW * 4);
    w.b1 = take((size_t)A * 64 * HW * 4);
    w.tile_sums = take((size_t)A * (HW / 32) * 64 * 4);
    w.attn = take((size_t)A * 64 * 4);
    w.xh = (uint4 *)take((size_t)A * HW * C * 2);
    w.xl = (uint4 *)take((size_t)A * HW * C * 2);
    w.bytes = off;
    return w;
}
static inline size_t packed_off_bytes(int C) { return (size_t)9 * C * 32 * 2 * 2; }   // value + residual planes
static inline size_t packed_dcn_bytes(int C) { return (size_t)9 * C * 64 * 2; }

}  // namespace me
}  // namespace gc

using namespace gc;

extern "C" size_t gc_me_param_floats(void) { return me::kTailFloats; }
extern "C" size_t gc_me_packed_bytes(int C) {
    return C > 0 ? align_up(me::packed_off_bytes(C), 256) + me::packed_dcn_bytes(C) : 0;
}
extern "C" size_t gc_me_workspace_bytes(int total_agents, int C, int H, int W) {
    if (total_agents <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
    return me::carve(nullptr, total_agents, C, H * W).bytes;
}

extern "C" int gc_me_pack_weights(const float *w_offset, const float *w_dcn, int C, void *packed, void *stream) {
    GC_REQUIRE(w_offset && w_dcn && packed, GC_EINVAL, "gc_me_pack_weights: null pointer");
    GC_REQUIRE(C > 0 && C % 64 == 0, GC_EUNSUPPORTED, "gc_me_pack_weights: C must be a multiple of 64 (got %d)", C);
    cudaStream_t st = (cudaStream_t)stream;
    uint4 *p_off = (uint4 *)packed;
    uint4 *p_dcn = (uint4 *)((char *)packed + align_up(me::packed_off_bytes(C), 256));
    const int n_off = 9 * (C / 8) * 32, n_dcn = 9 * (C / 8) * 64;
    me::k_me_pack<<<(n_off + 255) / 256, 256, 0, st>>>(w_offset, 18, 32, C, me::kScOffset, 9, 1, p_off);
    GC_LAUNCH_CHECK("k_me_pack(offset1)");
    me::k_me_pack<<<(n_dcn + 255) / 256, 256, 0, st>>>(w_dcn, 64, 64, C, me::kScDeform, 9, 0, p_dcn);
    GC_LAUNCH_CHECK("k_me_pack(dcn1)");
    return GC_OK;
}

extern "C" int gc_message_extractor(const float *x, int total_agents, int C, int H, int W, const void *packed,
                                    const float *params, void *workspace, float *message, void *stream) {
    GC_REQUIRE(total_agents >= 0 && total_agents <= 65535, GC_EINVAL, "gc_message_extractor: bad agent count");
    if (total_agents == 0) return GC_OK;
    GC_REQUIRE(x && packed && params && workspace && message, GC_EINVAL, "gc_message_extractor: null pointer");
    GC_REQUIRE(C > 0 && C % 64 == 0, GC_EUNSUPPORTED, "gc_message_extractor: C must be a multiple of 64 (got %d)", C);
    GC_REQUIRE(H > 0 && W > 0 && (H * W) % me::kPix == 0, GC_EUNSUPPORTED,
               "gc_message_extractor: H*W must be a multiple of 128 (got %dx%d)", H, W);
    cudaStream_t st = (cudaStream_t)stream;
    const int HW = H * W, tiles = HW / me::kPix;
    const me::Workspace ws = me::carve(workspace, total_agents, C, HW);
    const uint4 *p_off = (const uint4 *)packed;
    const uint4 *p_dcn = (const uint4 *)((const char *)packed + align_up(me::packed_off_bytes(C), 256));
    static bool attr_done = false;
    constexpr int kSmemOff = me::conv_smem_bytes(32, true, me::kScOffset), kSmemDcn = me::conv_smem_bytes(64, false, me::kScDeform);
    if (!attr_done) {
        cudaFuncSetAttribute(me::k_me_conv<32, false, me::kScOffset>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemOff);
        cudaFuncSetAttribute(me::k_me_conv<64, true, me::kScDeform>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemDcn);
        cudaFuncSetAttribute(me::k_me_offset_row3, cudaFuncAttributeMaxDynamicSharedMemorySize, me::kR3Smem);
        cudaFuncSetAttribute(me::k_me_tail_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, me::kTtSmem);
        attr_done = true;
    }
    const dim3 grid(tiles, total_agents);
    if (int rc = to_planes(st, x, total_agents, C, HW, ws.xh, ws.xl)) return rc;
    if (W % me::kPix == 0 && !getenv("GC_ME_GENERIC_OFFSET")) {   // a tile is 128 pixels of one image row
        me::k_me_offset_row3<<<grid, me::kThreads, me::kR3Smem, st>>>(ws.xh, ws.xl, p_off, params + me::kOffBias, C, H, W,
                                                                      ws.offset);
        GC_LAUNCH_CHECK("k_me_offset_row3");
    } else {
        me::k_me_conv<32, false, me::kScOffset><<<grid, me::conv_block_threads(false), kSmemOff, st>>>(ws.xh, ws.xl, nullptr, p_off,
                                                                                   params + me::kOffBias, C, C, H, W, 18, 18,
                                                                                   0, ws.offset, nullptr);
        GC_LAUNCH_CHECK("k_me_conv<offset1>");
    }
    me::k_me_conv<64, true, me::kScDeform><<<grid, me::kThreads, kSmemDcn, st>>>(ws.xh, ws.xl, ws.offset, p_dcn, params + me::kDcnBias, C, C,
                                                                  H, W, 64, 64, 0, ws.b1, ws.tile_sums);
    GC_LAUNCH_CHECK("k_me_conv<dcn1>");
    me::k_me_attn<<<total_agents, 64, 0, st>>>(ws.tile_sums, tiles * 4, HW, params, ws.attn);
    GC_LAUNCH_CHECK("k_me_attn");
    if (!getenv("GC_ME_FP32_TAIL")) {
        me::k_me_tail_tc<<<grid, 128, me::kTtSmem, st>>>(ws.b1, ws.attn, params, HW, message);
        GC_LAUNCH_CHECK("k_me_tail_tc");
    } else {   // CUDA-core fp32 tail (A/B)
        me::k_me_tail<<<grid, 128, 0, st>>>(ws.b1, ws.attn, params, HW, message);
        GC_LAUNCH_CHECK("k_me_tail");
    }
    return GC_OK;
}
