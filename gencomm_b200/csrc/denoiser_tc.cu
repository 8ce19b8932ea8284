// tcgen05 (5th-gen tensor core) implicit-GEMM kernels for the two GEMM-shaped layers of the GenComm
// denoiser: conv_in ((C+2) -> 8, K = 9(C+2)) and norm_out+swish+conv_out (8 -> C, K = 72), which carry
// 63 % of the denoiser FLOPs (SURVEY.md App. A.7).  bf16 operands, fp32 accumulation in TMEM.
//
// Reference semantics: models/gencomm_modules/unet.py:315 (conv_in), :341-343 (norm_out, swish,
// conv_out); the sampler update fused into conv_out's epilogue is cond_diff.py:272-279, :310-313.
//
// Implicit GEMM without im2col.  D[M = 128 pixels of one image row, N] += A[M, K] * B[K, N].
// A is the activation row in "NHWC8 bf16" form in shared memory: pixel p = 16 bytes = 8 channels, which
// is exactly one row of a K-major no-swizzle UMMA core matrix (8 rows x 16 bytes, rows 16 bytes apart).
// With SBO = 128 B the 16 row-groups of an M = 128 operand are 128 consecutive pixels, so the A operand
// of tap (ky, kx) is simply the staged row y+ky-1 starting at pixel x0+kx-1: a descriptor whose start
// address is shifted by kx * 16 bytes.  The two K core matrices of one K = 16 MMA are
//   * conv_in : two 8-channel groups at the same tap        (LBO = distance between channel-group planes)
//   * conv_out: taps kx and kx+1 of the same row            (LBO = 16 B: the next pixel; the fourth
//               "tap" kx = 3 of each row has zero weights, K = 3 * 32 = 96)
// so the staged rows are read in place by the tensor core for all nine taps.
//
// One elected thread issues tcgen05.mma; completion is tracked with tcgen05.commit -> mbarrier; the
// epilogue reads TMEM with tcgen05.ld.32x32b (lane = pixel, so per-channel global stores are coalesced).
#include <cuda_bf16.h>

#include "common.cuh"
#include "denoiser_tc.cuh"
#include "ptx.cuh"

namespace gc {
namespace tc {

using namespace ptx;

__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
    return make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}
__device__ __forceinline__ float swish(float v) { return __fdividef(v, 1.0f + __expf(-v)); }

// GroupNorm(4 groups of 2 channels) coefficients of one 8-channel NHWC8 tensor from per-tile partial sums
// (same arithmetic as gn_coeff<8> in denoiser.cu: fixed order, float64).
__device__ __forceinline__ void gn_coeff8(int c, int agent, const float *__restrict__ st, int tiles, int hw, float gamma,
                                          float beta, float *ga, float *gb) {
    st += (size_t)agent * tiles * 8;
    const int p = c >> 1;
    double s = 0.0, ss = 0.0;
    for (int t = 0; t < tiles; ++t) { s += st[t * 8 + 2 * p]; ss += st[t * 8 + 2 * p + 1]; }
    const double cnt = (double)hw * 2.0;
    const double mean = s / cnt;
    double var = ss / cnt - mean * mean;
    var = var < 0.0 ? 0.0 : var;
    const double rstd = 1.0 / sqrt(var + 1e-6);
    *ga = (float)((double)gamma * rstd);
    *gb = (float)((double)beta - mean * (double)gamma * rstd);
}

// ------------------------------------------------------------------------------------------------
// One-time (per call) repack of the fp32 conv weights into the bf16 UMMA B-operand byte layouts, so that every CTA
// copies its B operand with coalesced 16-byte loads instead of converting scattered fp32 weights itself.
//   conv_out: [12 k-chunks (ky*4+kx, kx == 3 zero)][C rows][8 bf16]          from w [C][9][8] (cout, tap, cin)
//   conv_in : [chunks][9 taps][2 groups][8 cout][8 bf16]                     from w [C+2][9][8] (cin, tap, cout)
// ------------------------------------------------------------------------------------------------
__global__ void k_pack_conv_out_w(const float *__restrict__ w, int C, uint4 *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 12 * C) return;
    const int n = i % C, kc = i / C, ky = kc >> 2, kx = kc & 3;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (kx < 3) {
        const float4 *src = reinterpret_cast<const float4 *>(w + ((size_t)n * 9 + ky * 3 + kx) * 8);
        const float4 lo = __ldg(src), hi = __ldg(src + 1);
        v = make_uint4(pack_bf16(lo.x, lo.y), pack_bf16(lo.z, lo.w), pack_bf16(hi.x, hi.y), pack_bf16(hi.z, hi.w));
    }
    out[i] = v;
}

__global__ void k_pack_conv_in_w(const float *__restrict__ w, int C, int chunks, uint4 *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= chunks * 9 * 2 * 8) return;
    const int n = i & 7, gsel = (i >> 3) & 1, tap = (i >> 4) % 9, q = (i >> 4) / 9;
    const int g = 2 * q + gsel;
    float f[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const int kc = 8 * g + c;                       // GEMM channel: x_0..x_{C-1}, cond_0, cond_1, zeros
        const int cin = kc < C ? kc + 2 : kc - C;       // reference channel (cond first)
        f[c] = kc < C + 2 ? __ldg(w + ((size_t)cin * 9 + tap) * 8 + n) : 0.0f;
    }
    out[i] = pack8(f);
}

// ------------------------------------------------------------------------------------------------
// norm_out + swish + conv_out on tensor cores.  grid = (W/128, H, A * C/NT), 128 threads.
//   in  [A][H][W][8] f32 (NHWC8) + GroupNorm partial sums;  w [C][9][8] f32 (cout, tap, cin); bias [C]
//   mode 0: pred = x0;  mode 1: x <- (c1*x0 + c2*x) + sigma*noise   (NCHW f32)
// ------------------------------------------------------------------------------------------------
constexpr int kOutRowPx = 132;   // staged pixels per row: x0-1 .. x0+130 (taps kx = 0..3 of pixel 127 reach 130)
constexpr int kOutRows = 4;      // image rows per CTA

template <int NT>
__global__ void __launch_bounds__(128)
k_conv_out_tc(const float *__restrict__ in, const float *__restrict__ st_in, int tiles_in, const uint4 *__restrict__ wp,
              const float *__restrict__ bias, Affine8 aff, int C, int H, int W, int mode, float c1, float c2, float sigma,
              const float *__restrict__ noise, float *__restrict__ x, float *__restrict__ pred, int materialize) {
    extern __shared__ __align__(128) uint8_t smem[];
    // [B: 12 k-chunks][NT rows][16 B]  |  [A rows: 3][132 px][16 B]  |  [A materialised: 12][128][16 B] (debug mode)
    uint4 *b_s = reinterpret_cast<uint4 *>(smem);
    uint4 *a_rows = b_s + 12 * NT;
    uint4 *a_mat = a_rows + 3 * kOutRowPx;
    __shared__ float s_ga[8], s_gb[8], s_bias[NT];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ uint32_t s_tmem;

    const int tid = threadIdx.x, warp = tid >> 5;
    const int splits = C / NT;
    const int agent = blockIdx.z / splits, co0 = (blockIdx.z % splits) * NT;
    // kOutRows image rows per CTA: the weights (24 KB at NT = 128), bias and GroupNorm coefficients are loaded once per CTA instead of
    // once per row (round 2; one row per CTA spent most of its time in that set-up: 16 warps per SM, long-scoreboard bound)
    const int x0 = blockIdx.x * 128, y_first = blockIdx.y * kOutRows;

    if (warp == 0) tmem_alloc<NT>(&s_tmem);
    if (tid == 32) { mbar_init(smem_u32(&s_bar), 1); mbar_init_fence(); }
    if (tid >= 64 && tid < 72) {
        const int c = tid - 64;
        gn_coeff8(c, agent, st_in, tiles_in, H * W, aff.gamma[c], aff.beta[c], &s_ga[c], &s_gb[c]);
    }
    for (int i = tid; i < NT; i += 128) s_bias[i] = __ldg(bias + co0 + i);
    // ---- B operand: pre-packed bf16 K-major core matrices [kc][C][16 B]; this CTA's NT rows of every k-chunk ----
    for (int i = tid; i < 12 * NT; i += 128) {
        const int n = i % NT, kc = i / NT;
        b_s[i] = __ldg(wp + (size_t)kc * C + co0 + n);
    }
    __syncthreads();
    const size_t plane = (size_t)H * W;
    const uint32_t tmem_base = s_tmem;
#pragma unroll 1
    for (int yr = 0; yr < kOutRows; ++yr) {
    const int y = y_first + yr;
    if (y >= H) break;
    // epilogue operands of this row's first 16 channels: in flight while the row is staged and multiplied
    size_t idx = ((size_t)agent * C + co0) * plane + (size_t)y * W + x0 + tid;
    float xv[16], nz[16];
    if (mode != 0) {
#pragma unroll
        for (int i = 0; i < 16; ++i) { xv[i] = x[idx + (size_t)i * plane]; nz[i] = __ldg(noise + idx + (size_t)i * plane); }
    }
    // ---- A rows: GroupNorm + swish -> bf16; zero outside the image (padding applies AFTER the activation) ----
    for (int i = tid; i < 3 * kOutRowPx; i += 128) {
        const int r = i / kOutRowPx, px = i % kOutRowPx;
        const int gy = y - 1 + r, gx = x0 - 1 + px;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (px < 130 && gy >= 0 && gy < H && gx >= 0 && gx < W) {
            const float4 *src = reinterpret_cast<const float4 *>(in + (((size_t)agent * H + gy) * W + gx) * 8);
            const float4 lo = __ldg(src), hi = __ldg(src + 1);
            float f[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
#pragma unroll
            for (int c = 0; c < 8; ++c) f[c] = swish(fmaf(f[c], s_ga[c], s_gb[c]));
            v = pack8(f);
        }
        a_rows[i] = v;
    }
    if (materialize) {   // debug/validation variant: explicit im2col blocks, no overlapping operand windows
        __syncthreads();
        for (int kc = 0; kc < 12; ++kc) a_mat[kc * 128 + tid] = a_rows[(kc >> 2) * kOutRowPx + tid + (kc & 3)];
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base;

    if (leader_of_warp0()) {
        constexpr uint32_t idesc = make_idesc(128, NT);
#pragma unroll
        for (int j = 0; j < 6; ++j) {   // K = 16 slices: row ky = j/2, taps kx = 2*(j%2), 2*(j%2)+1
            const uint64_t adesc = materialize
                ? make_desc(smem_u32(a_mat + (2 * j) * 128), 2048u, 128u)
                : make_desc(smem_u32(a_rows + (j >> 1) * kOutRowPx + (j & 1) * 2), 16u, 128u);
            const uint64_t bdesc = make_desc(smem_u32(b_s + (2 * j) * NT), (uint32_t)NT * 16u, 128u);
            mma_bf16(tmem, adesc, bdesc, idesc, j > 0 ? 1u : 0u);
        }
        mma_commit(smem_u32(&s_bar));
    }
    mbar_wait(smem_u32(&s_bar), (uint32_t)yr & 1u);
    tc_fence_after();

    // ---- epilogue: lane = pixel; 16 channels per TMEM load; per-channel stores are 128 B per warp; the x / noise values of the
    // next 16 channels are loaded before the current 16 are combined and stored ----
    const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
    for (int c0 = 0; c0 < NT; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + (uint32_t)c0, v);
        if (mode == 0) {
#pragma unroll
            for (int i = 0; i < 16; ++i) pred[idx + (size_t)i * plane] = v[i] + s_bias[c0 + i];
        } else {
            float xn[16], nn[16];
            if (c0 + 16 < NT) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    xn[i] = x[idx + (size_t)(16 + i) * plane];
                    nn[i] = __ldg(noise + idx + (size_t)(16 + i) * plane);
                }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float mean = __fadd_rn(__fmul_rn(c1, v[i] + s_bias[c0 + i]), __fmul_rn(c2, xv[i]));
                x[idx + (size_t)i * plane] = __fadd_rn(mean, __fmul_rn(sigma, nz[i]));
            }
            if (c0 + 16 < NT) {
#pragma unroll
                for (int i = 0; i < 16; ++i) { xv[i] = xn[i]; nz[i] = nn[i]; }
            }
        }
        idx += 16 * plane;
    }
    // the next row overwrites the staged rows and the accumulator: every thread is past its TMEM reads
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    }   // rows
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free<NT>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// conv_in on tensor cores: cat[cond(2), x_t(C)] (NCHW f32) -> 8 channels (NHWC8 f32) + GroupNorm partial sums.
// grid = (W/128, ceil(H/4), A), 128 threads.  K is walked in chunks of 16 input channels (two 8-channel
// groups; GEMM channel order = x_0..x_{C-1}, cond_0, cond_1, zero padding), double buffered: while the
// tensor core consumes chunk q (9 taps x 4 rows = 36 MMAs of 128 x 16 x 16) the threads stage chunk q+1.
// M = 128 needs N % 16 == 0: the B descriptor uses SBO = 0, so output columns 8..15 alias 0..7 and are ignored.
//   w [C+2][9][8] f32 (cin in the reference's cat order, tap, cout)
// ------------------------------------------------------------------------------------------------
constexpr int kInRows = 4;                 // output rows per CTA
constexpr int kInStaged = kInRows + 2;     // staged input rows
constexpr int kInRowPx = 130;              // x0-1 .. x0+128
constexpr int kInGroupU4 = kInStaged * kInRowPx;   // uint4 per channel group per buffer

__global__ void __launch_bounds__(128)
k_conv_in_tc(const float *__restrict__ cond, const float *__restrict__ x, const uint4 *__restrict__ wp, Bias8 bias, int C,
             int H, int W, float *__restrict__ out, float *__restrict__ stats_out) {
    extern __shared__ __align__(128) uint8_t smem[];
    // [A: 2 buffers][2 groups][6 rows][130 px][16 B]  |  [B: chunks][9 taps][2 groups][8 cout][16 B]
    uint4 *a_s = reinterpret_cast<uint4 *>(smem);
    uint4 *b_s = a_s + 2 * 2 * kInGroupU4;
    __shared__ __align__(8) uint64_t s_empty[2], s_done;
    __shared__ uint32_t s_tmem;
    __shared__ float s_part[4][8];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int agent = blockIdx.z, x0 = blockIdx.x * 128, y0 = blockIdx.y * kInRows;
    const int groups = C / 8 + 1, chunks = (groups + 1) / 2;
    const size_t plane = (size_t)H * W;

    if (warp == 0) tmem_alloc<64>(&s_tmem);
    if (tid == 32) {
        mbar_init(smem_u32(&s_empty[0]), 1); mbar_init(smem_u32(&s_empty[1]), 1); mbar_init(smem_u32(&s_done), 1);
        mbar_init_fence();
    }
    // ---- B operand for every chunk: pre-packed [q][tap][gsel][n][8 bf16] ----
    for (int i = tid; i < chunks * 9 * 2 * 8; i += 128) b_s[i] = __ldg(wp + i);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const uint32_t a_base = smem_u32(a_s), b_base = smem_u32(b_s);
    constexpr uint32_t idesc = make_idesc(128, 16);
    constexpr uint32_t kGroupBytes = kInGroupU4 * 16u, kBufBytes = 2u * kGroupBytes;

    for (int q = 0; q < chunks; ++q) {
        const int b = q & 1;
        if (q >= 2) mbar_wait(smem_u32(&s_empty[b]), (uint32_t)((q >> 1) - 1) & 1u);   // MMAs of chunk q-2 retired
        uint4 *buf = a_s + b * 2 * kInGroupU4;
        // ---- stage chunk q: thread = pixel column; per channel group all 6 rows x 8 channels are loaded first
        // (48 independent loads in flight per thread), then packed to bf16 and stored ----
        for (int px = tid; px < kInRowPx; px += 128) {
            const int gx = x0 - 1 + px;
            const bool xin = gx >= 0 && gx < W;
#pragma unroll
            for (int gsel = 0; gsel < 2; ++gsel) {
                const int g = 2 * q + gsel;
                float f[kInStaged][8];
                if (xin && g < C / 8) {
                    const float *src = x + ((size_t)agent * C + 8 * g) * plane + gx;
#pragma unroll
                    for (int r = 0; r < kInStaged; ++r) {
                        const int gy = y0 - 1 + r;
                        const bool yin = gy >= 0 && gy < H;
                        const float *sr = src + (size_t)(yin ? gy : 0) * W;
#pragma unroll
                        for (int c = 0; c < 8; ++c) f[r][c] = yin ? __ldg(sr + (size_t)c * plane) : 0.0f;
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < kInStaged; ++r) {
                        const int gy = y0 - 1 + r;
                        const bool ok = xin && g == C / 8 && gy >= 0 && gy < H;
                        const float *sr = cond + (size_t)agent * 2 * plane + (size_t)(ok ? gy : 0) * W + (ok ? gx : 0);
                        f[r][0] = ok ? __ldg(sr) : 0.0f;
                        f[r][1] = ok ? __ldg(sr + plane) : 0.0f;
#pragma unroll
                        for (int c = 2; c < 8; ++c) f[r][c] = 0.0f;
                    }
                }
#pragma unroll
                for (int r = 0; r < kInStaged; ++r) buf[(gsel * kInStaged + r) * kInRowPx + px] = pack8(f[r]);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (leader_of_warp0()) {
            tc_fence_after();
            const uint32_t a_buf = a_base + (uint32_t)b * kBufBytes;
#pragma unroll 1
            for (int tap = 0; tap < 9; ++tap) {
                const int ky = tap / 3, kx = tap % 3;
                const uint64_t bdesc = make_desc(b_base + (uint32_t)((q * 9 + tap) * 2) * 128u, 128u, 0u);
#pragma unroll
                for (int r = 0; r < kInRows; ++r) {
                    const uint64_t adesc = make_desc(a_buf + (uint32_t)((r + ky) * kInRowPx + kx) * 16u, kGroupBytes, 128u);
                    mma_bf16(tmem + (uint32_t)(r * 16), adesc, bdesc, idesc, (q > 0 || tap > 0) ? 1u : 0u);
                }
            }
            mma_commit(smem_u32(&s_empty[b]));
            if (q == chunks - 1) mma_commit(smem_u32(&s_done));
        }
    }
    mbar_wait(smem_u32(&s_done), 0u);
    tc_fence_after();

    // ---- epilogue: thread = pixel; bias, NHWC8 store, GroupNorm partial sums of the tile ----
    const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
    float q8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) q8[i] = 0.0f;
#pragma unroll
    for (int r = 0; r < kInRows; ++r) {
        float v[8];
        tmem_ld8(taddr + (uint32_t)(r * 16), v);
        const int yy = y0 + r;
        if (yy < H) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += bias.b[i];
            float4 *dst = reinterpret_cast<float4 *>(out + (((size_t)agent * H + yy) * W + x0 + tid) * 8);
            dst[0] = make_float4(v[0], v[1], v[2], v[3]);
            dst[1] = make_float4(v[4], v[5], v[6], v[7]);
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                q8[2 * p] += v[2 * p] + v[2 * p + 1];
                q8[2 * p + 1] += v[2 * p] * v[2 * p] + v[2 * p + 1] * v[2 * p + 1];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) q8[i] += __shfl_xor_sync(0xffffffffu, q8[i], m);
    }
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s_part[warp][i] = q8[i];
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 8) {
        const float t = (s_part[0][tid] + s_part[1][tid]) + (s_part[2][tid] + s_part[3][tid]);
        const int tiles = gridDim.x * gridDim.y, tile = blockIdx.y * gridDim.x + blockIdx.x;
        stats_out[((size_t)agent * tiles + tile) * 8 + tid] = t;
    }
    if (warp == 0) tmem_free<64>(tmem);
}


// ------------------------------------------------------------------------------------------------
// conv_in, second version ("input-row stationary", the formulation of denoiser_cluster.cu): one CTA = 8 output rows x 128
// pixels of one agent.  Per chunk of 16 input channels the 10 input rows are staged ONCE as bf16 pixel vectors
// (thread = 4 pixels x 8 channels: eight coalesced 16-byte loads, an in-register transpose, four 16-byte stores) and
// every staged row feeds the three output rows it contributes to with ONE MMA per tap kx:
//   D[128 px of input row i, 32] += A_i[128, 16 ch] * B_kx[16 ch, 4 blocks x 8 cout]   (block j = tap row ky = 2 - j)
// into TMEM columns 8 i .. 8 i + 31 (the accumulator of output row r lives at column 8 (r + 2)): 30 MMAs per chunk for 8
// output rows instead of 72, input rows read 1.25x instead of 1.5x, and 256 CTAs for 32 agents = one wave at 2 CTAs/SM
// (the first version ran 512 CTAs on 444 slots: r01 112 us for 139 MB).
//   wp2: [chunk][kx 3][k group 2][block 4][cout 8][8 bf16] packed by k_pack_conv_in_w2
// ------------------------------------------------------------------------------------------------
constexpr int kIn2Rows = 8, kIn2Staged = kIn2Rows + 2, kIn2RowPx = 130, kIn2Threads = 256;
constexpr int kIn2PlaneU4 = kIn2Staged * kIn2RowPx;                 // uint4 per channel-group plane
constexpr int kIn2BufBytes = 2 * kIn2PlaneU4 * 16;                  // one chunk: two planes = 41600 B

__global__ void k_pack_conv_in_w2(const float *__restrict__ w, int C, int chunks, uint4 *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= chunks * 3 * 2 * 4 * 8) return;
    const int n = i & 7, j = (i >> 3) & 3, gsel = (i >> 5) & 1, kx = (i >> 6) % 3, q = (i >> 6) / 3;
    const int g = 2 * q + gsel;
    float f[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const int kc = 8 * g + c;                       // GEMM channel: x_0..x_{C-1}, cond_0, cond_1, zeros
        const int cin = kc < C ? kc + 2 : kc - C;       // reference channel (cond first)
        f[c] = (j < 3 && kc < C + 2) ? __ldg(w + ((size_t)cin * 9 + (2 - j) * 3 + kx) * 8 + n) : 0.0f;
    }
    out[i] = pack8(f);
}

__global__ void __launch_bounds__(kIn2Threads)
k_conv_in_tc2(const float *__restrict__ cond, const float *__restrict__ x, const uint4 *__restrict__ wp2, Bias8 bias, int C, int H,
              int W, float *__restrict__ out, float *__restrict__ stats_out) {
    extern __shared__ __align__(128) uint8_t smem[];
    // [A: 2 buffers][2 groups][10 rows][130 px][16 B]  |  [B: chunks][3 kx][2 groups][4 blocks][8 cout][16 B]
    uint4 *a_s = reinterpret_cast<uint4 *>(smem);
    uint4 *b_s = reinterpret_cast<uint4 *>(smem + 2 * kIn2BufBytes);
    __shared__ __align__(8) uint64_t s_empty[2], s_done, s_wbar;
    __shared__ uint32_t s_tmem;
    __shared__ float s_part[kIn2Threads / 32][8];

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int agent = blockIdx.y, y0 = blockIdx.x * kIn2Rows;            // W == 128: one tile per row band
    const int groups = C / 8 + 1, chunks = (groups + 1) / 2;
    const size_t plane = (size_t)H * W;

    if (warp == 0) tmem_alloc<128>(&s_tmem);
    if (tid == 32) {
        mbar_init(smem_u32(&s_empty[0]), 1); mbar_init(smem_u32(&s_empty[1]), 1); mbar_init(smem_u32(&s_done), 1);
        mbar_init(smem_u32(&s_wbar), 1);
        mbar_init_fence();
    }
    // x halo columns (pixels -1 and 128) are outside the image for W == 128: zero once, staging never touches them
    for (int i = tid; i < 2 * 2 * kIn2Staged * 2; i += kIn2Threads) {
        const int side = i & 1, r = (i >> 1) % kIn2Staged, pl = (i >> 1) / kIn2Staged;
        a_s[(pl * kIn2Staged + r) * kIn2RowPx + (side ? kIn2RowPx - 1 : 0)] = make_uint4(0u, 0u, 0u, 0u);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = __shfl_sync(0xffffffffu, s_tmem, 0);
    if (tid == 0) bulk_load(smem_u32(b_s), wp2, (uint32_t)chunks * 3u * 1024u, smem_u32(&s_wbar));
    if (warp < 4) {   // zero the 8 (10 + 3) accumulator columns
        const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll
        for (int j = 0; j < 13; ++j)
            tmem_zero8(ta + 8u * j);
        tmem_wait_st();
    }
    const uint32_t a_base = smem_u32(a_s), b_base = smem_u32(b_s);
    constexpr uint32_t idesc = make_idesc(128, 32);
    constexpr uint32_t kPlaneBytes = kIn2PlaneU4 * 16u;

    for (int q = 0; q < chunks; ++q) {
        const int b = q & 1;
        if (q >= 2) mbar_wait(smem_u32(&s_empty[b]), (uint32_t)((q >> 1) - 1) & 1u);   // MMAs of chunk q - 2 retired
        uint4 *buf = a_s + b * 2 * kIn2PlaneU4;
        // ---- stage chunk q: item = (group, row, 4-pixel quad); 2 x 10 x 32 = 640 items ----
        for (int it = tid; it < 2 * kIn2Staged * 32; it += kIn2Threads) {
            const int quad = it & 31, r = (it >> 5) % kIn2Staged, gsel = (it >> 5) / kIn2Staged;
            const int g = 2 * q + gsel, gy = y0 - 1 + r;
            if (gy < 0 || gy >= H) continue;                    // row outside the image: its MMAs are skipped
            float4 v[8];
            if (g < C / 8) {
                const float *src = x + ((size_t)agent * C + 8 * g) * plane + (size_t)gy * W + quad * 4;
#pragma unroll
                for (int c = 0; c < 8; ++c) v[c] = __ldg(reinterpret_cast<const float4 *>(src + (size_t)c * plane));
            } else {
#pragma unroll
                for (int c = 0; c < 8; ++c) v[c] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g == C / 8) {
                    const float *src = cond + (size_t)agent * 2 * plane + (size_t)gy * W + quad * 4;
                    v[0] = __ldg(reinterpret_cast<const float4 *>(src));
                    v[1] = __ldg(reinterpret_cast<const float4 *>(src + plane));
                }
            }
            uint4 *dst = buf + (gsel * kIn2Staged + r) * kIn2RowPx + 1 + quad * 4;
            { const float f[8] = {v[0].x, v[1].x, v[2].x, v[3].x, v[4].x, v[5].x, v[6].x, v[7].x}; dst[0] = pack8(f); }
            { const float f[8] = {v[0].y, v[1].y, v[2].y, v[3].y, v[4].y, v[5].y, v[6].y, v[7].y}; dst[1] = pack8(f); }
            { const float f[8] = {v[0].z, v[1].z, v[2].z, v[3].z, v[4].z, v[5].z, v[6].z, v[7].z}; dst[2] = pack8(f); }
            { const float f[8] = {v[0].w, v[1].w, v[2].w, v[3].w, v[4].w, v[5].w, v[6].w, v[7].w}; dst[3] = pack8(f); }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
            tc_fence_after();
            if (q == 0) mbar_wait(smem_u32(&s_wbar), 0u);       // weights landed (bulk copy)
            const uint32_t a_buf = a_base + (uint32_t)b * (uint32_t)kIn2BufBytes;
            for (int i = 0; i < kIn2Staged; ++i) {
                const int gy = y0 - 1 + i;
                if (gy < 0 || gy >= H) continue;
                const uint64_t a0 = make_desc(a_buf + (uint32_t)(i * kIn2RowPx) * 16u, kPlaneBytes, 128u);
                const uint64_t b0 = make_desc(b_base + (uint32_t)(q * 3) * 1024u, 512u, 128u);
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) mma_bf16_elect(tmem + 8u * i, a0 + (uint64_t)kx, b0 + (uint64_t)(kx * 64), idesc);
            }
            commit_elect(smem_u32(&s_empty[b]));
            if (q == chunks - 1) commit_elect(smem_u32(&s_done));
        }
    }
    mbar_wait(smem_u32(&s_done), 0u);
    tc_fence_after();

    // ---- epilogue: thread = pixel x of 4 output rows; bias, NHWC8 store, GroupNorm partial sums of the band ----
    const int qd = warp & 3, hsel = warp >> 2, px = qd * 32 + lane, r0 = hsel * 4;
    float q8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) q8[i] = 0.0f;
    {
        float acc[32];
        const uint32_t ta = tmem + ((uint32_t)(qd * 32) << 16) + 8u * (r0 + 2);
        {
            float t0[16], t1[16];
            tmem_ld16(ta, t0);
            tmem_ld16(ta + 16u, t1);
#pragma unroll
            for (int i = 0; i < 16; ++i) { acc[i] = t0[i]; acc[16 + i] = t1[i]; }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            float *v = acc + 8 * r;
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += bias.b[i];
            float4 *dst = reinterpret_cast<float4 *>(out + (((size_t)agent * H + y0 + r0 + r) * W + px) * 8);
            dst[0] = make_float4(v[0], v[1], v[2], v[3]);
            dst[1] = make_float4(v[4], v[5], v[6], v[7]);
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                q8[2 * p] += v[2 * p] + v[2 * p + 1];
                q8[2 * p + 1] += v[2 * p] * v[2 * p] + v[2 * p + 1] * v[2 * p + 1];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) q8[i] += __shfl_xor_sync(0xffffffffu, q8[i], m);
    }
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s_part[warp][i] = q8[i];
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 8) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < kIn2Threads / 32; ++w) t += s_part[w][tid];
        stats_out[((size_t)agent * gridDim.x + blockIdx.x) * 8 + tid] = t;
    }
    if (warp == 0) tmem_free<128>(tmem);
}

// ------------------------------------------------------------------------------------------------
// Width-8 middle layers on tensor cores: 3x3 conv, CIN (8 or 16) -> 8 channels on NHWC8 fp32 tensors, tf32 operands
// (fp32 storage, no conversion pass), fp32 accumulation in TMEM.  unet.py:117-138 (ResnetBlock), :40-56 (Upsample).
// grid = (W/128, ceil(H/4), A), 128 threads; H, W are the OUTPUT dims (kUp: the input is H/2 x W/2).
//
// For 32-bit operands a K-major core matrix is 8 rows x 4 elements, so the 8 channels of a pixel are staged as two
// 16-byte halves in two planes [half][row][pixel]; one K = 8 MMA reads the two halves of one channel group
// (LBO = plane stride) at the tap's shifted start address.  GroupNorm + swish are applied while staging (padding is
// zero AFTER the activation); bias / timestep embedding, the residual or the 1x1 nin_shortcut and the GroupNorm
// partial sums of the output are the epilogue.  N = 16 with SBO = 0 on B (columns 8..15 alias 0..7, ignored).
// ------------------------------------------------------------------------------------------------
constexpr int kMidRows = 4, kMidStaged = kMidRows + 2, kMidRowPx = 130;
constexpr int kMidPlaneU4 = kMidStaged * kMidRowPx;   // uint4 (16-byte pixel halves) per plane

template <int CIN, bool PRE_GN, int GEOM, int RES>
__global__ void __launch_bounds__(128)
k_conv_c8_tc(const float *__restrict__ in_a, const float *__restrict__ in_b, const float *__restrict__ st_a,
             const float *__restrict__ st_b, int tiles_a, int tiles_b, const float *__restrict__ res_a,
             const float *__restrict__ res_b, float *__restrict__ out, float *__restrict__ stats_out, int H, int W,
             const __grid_constant__ C8Params prm) {
    constexpr int CG = CIN / 8;                       // channel groups of 8
    extern __shared__ __align__(128) uint8_t smem[];
    // [A: CG groups x 2 halves planes][6 rows][130 px][16 B]  |  [B: 9 taps][CG][2 halves][8 cout][16 B]
    float4 *a_s = reinterpret_cast<float4 *>(smem);
    float4 *b_s = a_s + CG * 2 * kMidPlaneU4;
    __shared__ __align__(8) uint64_t s_done;
    __shared__ uint32_t s_tmem;
    __shared__ float s_ga[16], s_gb[16], s_part[4][8];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int agent = blockIdx.z, x0 = blockIdx.x * 128, y0 = blockIdx.y * kMidRows;
    const int Hin = GEOM == kUp ? H / 2 : H, Win = GEOM == kUp ? W / 2 : W;

    if (warp == 0) tmem_alloc<kMidRows * 16 <= 32 ? 32 : 64>(&s_tmem);
    if (tid == 32) { mbar_init(smem_u32(&s_done), 1); mbar_init_fence(); }
    if (PRE_GN && tid >= 64 && tid < 64 + CIN) {
        // GroupNorm(4 groups) coefficients from per-tile partial sums (same fixed-order float64 combination as
        // gn_coeff<CIN> in denoiser.cu): CIN == 8: one channel pair per group; CIN == 16: two pairs of one tensor
        const int c = tid - 64, cc = c & 7;
        const int tiles = c < 8 ? tiles_a : tiles_b;
        const float *st = (c < 8 ? st_a : st_b) + (size_t)agent * tiles * 8;
        double sum = 0.0, ssq = 0.0;
        if (CIN == 8) {
            const int pr = cc >> 1;
            for (int t = 0; t < tiles; ++t) { sum += st[t * 8 + 2 * pr]; ssq += st[t * 8 + 2 * pr + 1]; }
        } else {
            const int pr = (cc >> 2) * 2;
            for (int t = 0; t < tiles; ++t) {
                sum += (double)st[t * 8 + 2 * pr] + (double)st[t * 8 + 2 * pr + 2];
                ssq += (double)st[t * 8 + 2 * pr + 1] + (double)st[t * 8 + 2 * pr + 3];
            }
        }
        const double cnt = (double)Hin * Win * (CIN == 8 ? 2.0 : 4.0);
        const double mean = sum / cnt;
        double var = ssq / cnt - mean * mean;
        var = var < 0.0 ? 0.0 : var;
        const double rstd = 1.0 / sqrt(var + 1e-6);
        s_ga[c] = (float)((double)prm.gamma[c] * rstd);
        s_gb[c] = (float)((double)prm.beta[c] - mean * (double)prm.gamma[c] * rstd);
    }
    // ---- B operand: [tap][cg][half][n] = w[tap][cg*8 + half*4 .. +3][n] ----
    for (int i = tid; i < 9 * CG * 2 * 8; i += 128) {
        const int n = i & 7, half = (i >> 3) & 1, cg = (i >> 4) % CG, tap = (i >> 4) / CG;
        const int c = cg * 8 + half * 4;
        b_s[i] = make_float4(prm.w[tap][c][n], prm.w[tap][c + 1][n], prm.w[tap][c + 2][n], prm.w[tap][c + 3][n]);
    }
    __syncthreads();
    // ---- A operand: thread = pixel column, 6 rows; all loads of a channel group first, then activation + store ----
    for (int px = tid; px < kMidRowPx; px += 128) {
        const int gx = x0 - 1 + px;
        const bool xin = gx >= 0 && gx < W;
        const int ix = GEOM == kUp ? gx >> 1 : gx;      // nearest x2 upsample (unet.py:52-53)
#pragma unroll
        for (int cg = 0; cg < CG; ++cg) {
            const float *src = (cg == 0 ? in_a : in_b) + (size_t)agent * Hin * Win * 8;
            float4 v[kMidStaged][2];
#pragma unroll
            for (int r = 0; r < kMidStaged; ++r) {
                const int gy = y0 - 1 + r;
                const bool ok = xin && gy >= 0 && gy < H;
                const int iy = GEOM == kUp ? gy >> 1 : gy;
                const float4 *q = reinterpret_cast<const float4 *>(src + ((size_t)(ok ? iy : 0) * Win + (ok ? ix : 0)) * 8);
                v[r][0] = ok ? __ldg(q) : make_float4(0.f, 0.f, 0.f, 0.f);
                v[r][1] = ok ? __ldg(q + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int r = 0; r < kMidStaged; ++r) {
                const int gy = y0 - 1 + r;
                const bool ok = xin && gy >= 0 && gy < H;
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    float4 u = v[r][half];
                    if (PRE_GN && ok) {
                        const int c = cg * 8 + half * 4;
                        u.x = swish(fmaf(u.x, s_ga[c + 0], s_gb[c + 0]));
                        u.y = swish(fmaf(u.y, s_ga[c + 1], s_gb[c + 1]));
                        u.z = swish(fmaf(u.z, s_ga[c + 2], s_gb[c + 2]));
                        u.w = swish(fmaf(u.w, s_ga[c + 3], s_gb[c + 3]));
                    }
                    a_s[((cg * 2 + half) * kMidStaged + r) * kMidRowPx + px] = u;
                }
            }
        }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    if (leader_of_warp0()) {
        constexpr uint32_t idesc = make_idesc_tf32(128, 16);
        constexpr uint32_t kPlaneBytes = kMidPlaneU4 * 16u;
        const uint32_t a_base = smem_u32(a_s), b_base = smem_u32(b_s);
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
            const int ky = tap / 3, kx = tap % 3;
#pragma unroll
            for (int cg = 0; cg < CG; ++cg) {
                const uint64_t bdesc = make_desc(b_base + (uint32_t)((tap * CG + cg) * 2) * 128u, 128u, 0u);
#pragma unroll
                for (int r = 0; r < kMidRows; ++r) {
                    const uint64_t adesc = make_desc(a_base + (uint32_t)(cg * 2) * kPlaneBytes + (uint32_t)((r + ky) * kMidRowPx + kx) * 16u,
                                                     kPlaneBytes, 128u);
                    mma_tf32(tmem + (uint32_t)(r * 16), adesc, bdesc, idesc, (tap > 0 || cg > 0) ? 1u : 0u);
                }
            }
        }
        mma_commit(smem_u32(&s_done));
    }
    mbar_wait(smem_u32(&s_done), 0u);
    tc_fence_after();

    // ---- epilogue: thread = pixel ----
    const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
    float q8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) q8[i] = 0.0f;
#pragma unroll
    for (int r = 0; r < kMidRows; ++r) {
        float acc[8];
        tmem_ld8(taddr + (uint32_t)(r * 16), acc);
        const int yy = y0 + r;
        if (yy < H) {
            const size_t pix = ((size_t)agent * H + yy) * W + x0 + tid;
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += prm.bias[i];
            if (RES != kNone) {
                const float4 a0 = __ldg(reinterpret_cast<const float4 *>(res_a + pix * 8));
                const float4 a1 = __ldg(reinterpret_cast<const float4 *>(res_a + pix * 8 + 4));
                if (RES == kIdent) {
                    acc[0] += a0.x; acc[1] += a0.y; acc[2] += a0.z; acc[3] += a0.w;
                    acc[4] += a1.x; acc[5] += a1.y; acc[6] += a1.z; acc[7] += a1.w;
                } else {
                    const float4 b0 = __ldg(reinterpret_cast<const float4 *>(res_b + pix * 8));
                    const float4 b1 = __ldg(reinterpret_cast<const float4 *>(res_b + pix * 8 + 4));
                    const float xr[16] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w,
                                          b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                    for (int o = 0; o < 8; ++o) {
                        float sh = prm.nin_b[o];
#pragma unroll
                        for (int ci = 0; ci < 16; ++ci) sh = fmaf(xr[ci], prm.nin_w[ci][o], sh);
                        acc[o] += sh;
                    }
                }
            }
            float4 *dst = reinterpret_cast<float4 *>(out + pix * 8);
            dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
            dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
#pragma unroll
            for (int pr = 0; pr < 4; ++pr) {
                q8[2 * pr] += acc[2 * pr] + acc[2 * pr + 1];
                q8[2 * pr + 1] += acc[2 * pr] * acc[2 * pr] + acc[2 * pr + 1] * acc[2 * pr + 1];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) q8[i] += __shfl_xor_sync(0xffffffffu, q8[i], m);
    }
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s_part[warp][i] = q8[i];
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 8) {
        const float t = (s_part[0][tid] + s_part[1][tid]) + (s_part[2][tid] + s_part[3][tid]);
        const int tiles = gridDim.x * gridDim.y, tile = blockIdx.y * gridDim.x + blockIdx.x;
        stats_out[((size_t)agent * tiles + tile) * 8 + tid] = t;
    }
    if (warp == 0) tmem_free<kMidRows * 16 <= 32 ? 32 : 64>(tmem);
}

}  // namespace tc

// ------------------------------------------------------------------------------------------------
// host launchers (called from denoiser.cu)
// ------------------------------------------------------------------------------------------------
bool conv_in_tc_eligible(int C, int H, int W) {
    (void)H;
    if (W % 128 != 0 || C % 8 != 0 || C < 8) return false;
    const int chunks = (C / 8 + 1 + 1) / 2;
    const size_t smem = (size_t)2 * 2 * tc::kInGroupU4 * 16 + (size_t)chunks * 9 * 2 * 128;
    return smem <= 200 * 1024;
}

int conv_in_tc_tiles(int H, int W) { return (W / 128) * ((H + tc::kInRows - 1) / tc::kInRows); }

static size_t conv_tc_packed_v1_bytes(int C) {   // conv_in B operand (v1 layout), then conv_out B operand
    const size_t chunks = (size_t)(C / 8 + 1 + 1) / 2;
    return align_up(align_up(chunks * 9 * 2 * 8 * 16, 256) + (size_t)12 * C * 16, 256);
}

size_t conv_tc_packed_bytes(int C) {   // + conv_in B operand in the input-row-stationary layout (k_conv_in_tc2)
    const size_t chunks = (size_t)(C / 8 + 1 + 1) / 2;
    return conv_tc_packed_v1_bytes(C) + chunks * 3 * 1024;
}

int conv_tc_pack_weights(cudaStream_t st, const float *w_in, const float *w_out, int C, void *packed) {
    const int chunks = (C / 8 + 1 + 1) / 2;
    uint4 *pin = reinterpret_cast<uint4 *>(packed);
    uint4 *pout = reinterpret_cast<uint4 *>(reinterpret_cast<char *>(packed) + align_up((size_t)chunks * 9 * 2 * 8 * 16, 256));
    tc::k_pack_conv_in_w<<<(chunks * 9 * 2 * 8 + 127) / 128, 128, 0, st>>>(w_in, C, chunks, pin);
    tc::k_pack_conv_out_w<<<(12 * C + 127) / 128, 128, 0, st>>>(w_out, C, pout);
    uint4 *pin2 = reinterpret_cast<uint4 *>(reinterpret_cast<char *>(packed) + conv_tc_packed_v1_bytes(C));
    tc::k_pack_conv_in_w2<<<(chunks * 3 * 64 + 127) / 128, 128, 0, st>>>(w_in, C, chunks, pin2);
    GC_LAUNCH_CHECK("conv_tc_pack_weights");
    return GC_OK;
}

int conv_in_tc(cudaStream_t st, int A, const float *cond, const float *x, const void *packed, const Bias8 &bias, int C, int H,
               int W, float *out, float *stats_out) {
    const uint4 *w = reinterpret_cast<const uint4 *>(packed);
    const int chunks = (C / 8 + 1 + 1) / 2;
    const size_t smem = (size_t)2 * 2 * tc::kInGroupU4 * 16 + (size_t)chunks * 9 * 2 * 128;
    static size_t configured = 0;
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(tc::k_conv_in_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { (void)cudaGetLastError(); set_error("k_conv_in_tc: cudaFuncSetAttribute failed (%d)", (int)e); return (int)e; }
        configured = smem;
    }
    const dim3 grid(W / 128, (H + tc::kInRows - 1) / tc::kInRows, A);
    tc::k_conv_in_tc<<<grid, 128, smem, st>>>(cond, x, w, bias, C, H, W, out, stats_out);
    GC_LAUNCH_CHECK("k_conv_in_tc");
    return GC_OK;
}

static int pick_nt(int C) {
    if (C % 256 == 0) return 256;
    if (C % 128 == 0) return 128;
    if (C % 64 == 0) return 64;
    return 0;
}

// conv_in v2: W == 128, H % 8 == 0, C % 8 == 0; shared memory: two operand buffers + the whole B operand
bool conv_in_tc2_eligible(int C, int H, int W) {
    if (W != 128 || H % tc::kIn2Rows != 0 || C % 8 != 0 || C < 8) return false;
    const int chunks = (C / 8 + 1 + 1) / 2;
    return (size_t)2 * tc::kIn2BufBytes + (size_t)chunks * 3 * 1024 <= 220 * 1024;
}

int conv_in_tc2_tiles(int H) { return H / tc::kIn2Rows; }

int conv_in_tc2(cudaStream_t st, int A, const float *cond, const float *x, const void *packed, const Bias8 &bias, int C, int H,
                int W, float *out, float *stats_out) {
    const int chunks = (C / 8 + 1 + 1) / 2;
    const uint4 *w = reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(packed) + conv_tc_packed_v1_bytes(C));
    const size_t smem = (size_t)2 * tc::kIn2BufBytes + (size_t)chunks * 3 * 1024;
    static size_t configured = 0;
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(tc::k_conv_in_tc2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { (void)cudaGetLastError(); set_error("k_conv_in_tc2: cudaFuncSetAttribute failed (%d)", (int)e); return (int)e; }
        configured = smem;
    }
    tc::k_conv_in_tc2<<<dim3(H / tc::kIn2Rows, A), tc::kIn2Threads, smem, st>>>(cond, x, w, bias, C, H, W, out, stats_out);
    GC_LAUNCH_CHECK("k_conv_in_tc2");
    return GC_OK;
}

bool conv_out_tc_eligible(int C, int H, int W) {
    (void)H;
    return W % 128 == 0 && pick_nt(C) != 0;
}

template <int NT>
static int launch_out(cudaStream_t st, int A, const float *in, const float *st_in, int tiles_in, const uint4 *w,
                      const float *bias, const Affine8 &aff, int C, int H, int W, int mode, float c1, float c2, float sigma,
                      const float *noise, float *x, float *pred, int materialize) {
    const size_t smem = (size_t)12 * NT * 16 + (size_t)3 * tc::kOutRowPx * 16 + (size_t)12 * 128 * 16;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(tc::k_conv_out_tc<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { (void)cudaGetLastError(); set_error("k_conv_out_tc: cudaFuncSetAttribute failed (%d)", (int)e); return (int)e; }
        configured = true;
    }
    const dim3 grid(W / 128, (H + tc::kOutRows - 1) / tc::kOutRows, A * (C / NT));
    tc::k_conv_out_tc<NT><<<grid, 128, smem, st>>>(in, st_in, tiles_in, w, bias, aff, C, H, W, mode, c1, c2, sigma, noise, x,
                                                   pred, materialize);
    GC_LAUNCH_CHECK("k_conv_out_tc");
    return GC_OK;
}

int conv_out_tc(cudaStream_t st, int A, const float *in, const float *st_in, int tiles_in, const void *packed, const float *bias,
                const Affine8 &aff, int C, int H, int W, int mode, float c1, float c2, float sigma, const float *noise,
                float *x, float *pred, int materialize) {
    const int chunks = (C / 8 + 1 + 1) / 2;
    const uint4 *w = reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(packed) + align_up((size_t)chunks * 9 * 2 * 8 * 16, 256));
    switch (pick_nt(C)) {
        case 256: return launch_out<256>(st, A, in, st_in, tiles_in, w, bias, aff, C, H, W, mode, c1, c2, sigma, noise, x, pred, materialize);
        case 128: return launch_out<128>(st, A, in, st_in, tiles_in, w, bias, aff, C, H, W, mode, c1, c2, sigma, noise, x, pred, materialize);
        case 64: return launch_out<64>(st, A, in, st_in, tiles_in, w, bias, aff, C, H, W, mode, c1, c2, sigma, noise, x, pred, materialize);
        default: break;
    }
    set_error("conv_out_tc: unsupported channel count %d", C);
    return GC_EUNSUPPORTED;
}

bool conv_c8_tc_eligible(int geom, int H, int W) {
    (void)H;
    return W % 128 == 0 && (geom == kSame || geom == kUp) && (geom != kUp || (H % 2 == 0));
}

template <int CIN, bool PRE_GN, int GEOM, int RES>
static int launch_c8_tc(cudaStream_t st, int A, const float *in_a, const float *in_b, const float *st_a, const float *st_b,
                        int tiles_a, int tiles_b, const float *res_a, const float *res_b, float *out, float *stats_out, int H,
                        int W, const C8Params &prm) {
    constexpr int CG = CIN / 8;
    const size_t smem = (size_t)CG * 2 * tc::kMidPlaneU4 * 16 + (size_t)9 * CG * 2 * 128;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(tc::k_conv_c8_tc<CIN, PRE_GN, GEOM, RES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { (void)cudaGetLastError(); set_error("k_conv_c8_tc: cudaFuncSetAttribute failed (%d)", (int)e); return (int)e; }
        configured = true;
    }
    const dim3 grid(W / 128, (H + tc::kMidRows - 1) / tc::kMidRows, A);
    tc::k_conv_c8_tc<CIN, PRE_GN, GEOM, RES><<<grid, 128, smem, st>>>(in_a, in_b, st_a, st_b, tiles_a, tiles_b, res_a, res_b, out,
                                                                      stats_out, H, W, prm);
    GC_LAUNCH_CHECK("k_conv_c8_tc");
    return GC_OK;
}

int conv_c8_tc(cudaStream_t st, int A, int cin, bool pre_gn, int geom, int res, const float *in_a, const float *in_b,
               const float *st_a, const float *st_b, int tiles_a, int tiles_b, const float *res_a, const float *res_b,
               float *out, float *stats_out, int H, int W, const C8Params &prm, int *tiles_out) {
    *tiles_out = (W / 128) * ((H + tc::kMidRows - 1) / tc::kMidRows);
#define GC_C8(CIN, PRE, GEOM, RES)                                                                                   \
    if (cin == CIN && pre_gn == PRE && geom == GEOM && res == RES)                                                   \
        return launch_c8_tc<CIN, PRE, GEOM, RES>(st, A, in_a, in_b, st_a, st_b, tiles_a, tiles_b, res_a, res_b, out, \
                                                 stats_out, H, W, prm);
    GC_C8(8, true, kSame, kNone)
    GC_C8(8, true, kSame, kIdent)
    GC_C8(8, true, kSame, kNin)
    GC_C8(16, true, kSame, kNone)
    GC_C8(8, false, kUp, kNone)
#undef GC_C8
    set_error("conv_c8_tc: unsupported layer variant (cin %d, geom %d, res %d)", cin, geom, res);
    return GC_EUNSUPPORTED;
}

}  // namespace gc
