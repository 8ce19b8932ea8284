// GenComm conditional-diffusion sampler + DiffusionUNet denoiser for sm_100a (fp32 path).
//
// Replaces (paths relative to /root/reference/opencood):
//   models/gencomm_modules/cond_diff.py:331-383  GenComm.forward (eval), :262-264 q_sample,
//        :272-279 q_posterior, :281-329 p_mean_variance / p_sample / p_sample_loop
//   models/gencomm_modules/unet.py:307-344 DiffusionUNet.forward, :81-138 ResnetBlock,
//        :59-78 Downsample, :40-56 Upsample, :36-37 GroupNorm(4, eps 1e-6), :31-33 swish
// for the only shipped denoiser shape: ch=8, ch_mult=[1,1], num_res_blocks=2, no attention blocks
// (SURVEY.md App. A.7: curr_res never reaches attn_resolutions).
//
// Design (DESIGN.md section 5).  The reference runs ~200 cuDNN/ATen launches per sampler step on
// 8-channel tensors.  Here every 3x3 convolution is ONE kernel that
//   * applies GroupNorm + swish of its input while staging the halo tile into shared memory
//     (statistics come from per-tile partial sums written by the producer's epilogue and are
//     combined in a fixed order in float64 -> deterministic, no atomics),
//   * adds bias + timestep embedding (pre-tabulated on the host per step), the residual /
//     1x1 nin_shortcut, and writes per-tile partial statistics for the next GroupNorm,
//   * reads the concatenated skip tensor through two pointers (no torch.cat),
//   * folds nearest-upsample / pad(0,1,0,1)+stride-2 into its addressing.
// 8-channel activations live in NHWC8 (32 B per pixel) so each thread moves its pixel with two
// 128-bit accesses.  conv_in ((C+2)->8) and conv_out (8->C) are implicit GEMMs over the NCHW
// boundary tensors; the sampler arithmetic (q_posterior + noise) is fused into conv_out's
// epilogue, q_sample is one elementwise kernel.  28 launches per step, 0 host syncs.
#include <stdlib.h>

#include "common.cuh"
#include "denoiser_cluster.cuh"
#include "denoiser_tc.cuh"

namespace gc {

constexpr int kTH = 8, kTW = 32;   // output tile per CTA (256 threads, one pixel each)
constexpr int kC8Layers = 26;      // 3x3 convs with 8 outputs per UNet evaluation, execution order

__device__ __forceinline__ float swish(float v) { return __fdividef(v, 1.0f + __expf(-v)); }

// GroupNorm(4 groups) scale/offset of channel c of a CIN-channel input made of one or two NHWC8 tensors.
// stats: [A][tiles][8] = per channel pair p: (sum, sum of squares) at [2p], [2p+1].
template <int CIN>
__device__ __forceinline__ void gn_coeff(int c, int agent, const float *__restrict__ st_a,
                                         const float *__restrict__ st_b, int tiles_a, int tiles_b, int hw,
                                         float gamma, float beta, float *ga, float *gb) {
    const int tiles = c < 8 ? tiles_a : tiles_b;   // the two tensors may come from kernels with different tilings
    const float *st = (c < 8 ? st_a : st_b) + (size_t)agent * tiles * 8;
    const int cc = c & 7;
    double s = 0.0, ss = 0.0;
    if (CIN == 8) {            // 4 groups of 2 channels: one pair
        const int p = cc >> 1;
        for (int t = 0; t < tiles; ++t) { s += st[t * 8 + 2 * p]; ss += st[t * 8 + 2 * p + 1]; }
    } else {                   // 16 channels, 4 groups of 4: two pairs of the same tensor
        const int p = (cc >> 2) * 2;
        for (int t = 0; t < tiles; ++t) {
            s += (double)st[t * 8 + 2 * p] + (double)st[t * 8 + 2 * p + 2];
            ss += (double)st[t * 8 + 2 * p + 1] + (double)st[t * 8 + 2 * p + 3];
        }
    }
    const double cnt = (double)hw * (CIN == 8 ? 2.0 : 4.0);
    const double mean = s / cnt;
    double var = ss / cnt - mean * mean;
    var = var < 0.0 ? 0.0 : var;
    const double rstd = 1.0 / sqrt(var + 1e-6);
    *ga = (float)((double)gamma * rstd);
    *gb = (float)((double)beta - mean * (double)gamma * rstd);
}

// per-CTA partial statistics of an 8-channel output tile -> stats_out[(agent*tiles + tile)*8 + 0..7]
__device__ __forceinline__ void write_tile_stats(const float (&v)[8], float *__restrict__ stats_out, int agent) {
    __shared__ float s_part[8][8];
    float q[8];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        q[2 * p] = v[2 * p] + v[2 * p + 1];
        q[2 * p + 1] = v[2 * p] * v[2 * p] + v[2 * p + 1] * v[2 * p + 1];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) q[i] += __shfl_xor_sync(0xffffffffu, q[i], m);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s_part[warp][i] = q[i];
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += s_part[w][threadIdx.x];
        const int tiles = gridDim.x * gridDim.y;
        const int tile = blockIdx.y * gridDim.x + blockIdx.x;
        stats_out[((size_t)agent * tiles + tile) * 8 + threadIdx.x] = t;
    }
}

// ------------------------------------------------------------------------------------------------
// 3x3 conv, CIN (8 or 16) -> 8 channels on NHWC8 tensors.  H, W are the OUTPUT dims.
// ------------------------------------------------------------------------------------------------
template <int CIN, bool PRE_GN, int GEOM, int RES>
__global__ void __launch_bounds__(256)
k_conv_c8(const float *__restrict__ in_a, const float *__restrict__ in_b, const float *__restrict__ st_a,
          const float *__restrict__ st_b, int tiles_in, int tiles_in_b, const float *__restrict__ res_a,
          const float *__restrict__ res_b, float *__restrict__ out, float *__restrict__ stats_out, int H, int W,
          const __grid_constant__ C8Params prm) {
    constexpr int Q = CIN / 4;
    constexpr int TR = GEOM == kDown ? 2 * kTH + 1 : kTH + 2;   // staged rows
    constexpr int TC = GEOM == kDown ? 2 * kTW + 1 : kTW + 2;   // staged cols
    __shared__ float4 tile[Q][TR][TC];
    __shared__ float s_ga[16], s_gb[16];

    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int x0 = blockIdx.x * kTW, y0 = blockIdx.y * kTH, agent = blockIdx.z;
    const int Hin = GEOM == kDown ? H * 2 : (GEOM == kUp ? H / 2 : H);
    const int Win = GEOM == kDown ? W * 2 : (GEOM == kUp ? W / 2 : W);

    if (PRE_GN) {
        if (tid < CIN) gn_coeff<CIN>(tid, agent, st_a, st_b, tiles_in, tiles_in_b, Hin * Win, prm.gamma[tid], prm.beta[tid],
                                     &s_ga[tid], &s_gb[tid]);
        __syncthreads();
    }
    // ---- stage the halo tile (GroupNorm + swish applied here; padding is zero AFTER the activation)
    for (int i = tid; i < TR * TC * Q; i += 256) {
        const int q = i / (TR * TC), rem = i % (TR * TC), r = rem / TC, c = rem % TC;
        int iy, ix;
        bool ok;
        if (GEOM == kDown) {          // pad (0,1,0,1), stride 2: input pixel (2y+ky, 2x+kx)
            iy = 2 * y0 + r; ix = 2 * x0 + c;
            ok = iy < Hin && ix < Win;
        } else {                      // padding 1 in output-resolution coordinates
            const int gy = y0 - 1 + r, gx = x0 - 1 + c;
            ok = gy >= 0 && gy < H && gx >= 0 && gx < W;
            iy = GEOM == kUp ? gy >> 1 : gy;      // nearest x2 upsample (unet.py:52-53)
            ix = GEOM == kUp ? gx >> 1 : gx;
        }
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) {
            const float *src = (q < 2 ? in_a : in_b) + (((size_t)agent * Hin + iy) * Win + ix) * 8 + (q & 1) * 4;
            v = __ldg(reinterpret_cast<const float4 *>(src));
            if (PRE_GN) {
                v.x = swish(fmaf(v.x, s_ga[4 * q + 0], s_gb[4 * q + 0]));
                v.y = swish(fmaf(v.y, s_ga[4 * q + 1], s_gb[4 * q + 1]));
                v.z = swish(fmaf(v.z, s_ga[4 * q + 2], s_gb[4 * q + 2]));
                v.w = swish(fmaf(v.w, s_ga[4 * q + 3], s_gb[4 * q + 3]));
            }
        }
        tile[q][r][c] = v;
    }
    __syncthreads();

    float acc[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = prm.bias[o];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int r = GEOM == kDown ? 2 * ty + ky : ty + ky;
            const int c = GEOM == kDown ? 2 * tx + kx : tx + kx;
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                const float4 v = tile[q][r][c];
                const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
#pragma unroll
                    for (int o = 0; o < 8; ++o) acc[o] = fmaf(vv[i], prm.w[ky * 3 + kx][4 * q + i][o], acc[o]);
                }
            }
        }
    }
    const int y = y0 + ty, x = x0 + tx;
    const bool inb = y < H && x < W;
    const size_t pix = ((size_t)agent * H + y) * W + x;
    if (RES != kNone && inb) {
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
    if (!inb) {
#pragma unroll
        for (int o = 0; o < 8; ++o) acc[o] = 0.0f;
    } else {
        float4 *dst = reinterpret_cast<float4 *>(out + pix * 8);
        dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
        dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
    write_tile_stats(acc, stats_out, agent);
}

// ------------------------------------------------------------------------------------------------
// conv_in: cat[cond(2), x_t(C)] (NCHW) -> 8 channels (NHWC8), 3x3 pad 1.  unet.py:315
// weights: device [C+2][9][8] (cin, tap, cout).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_conv_in(const float *__restrict__ cond, const float *__restrict__ x, const float *__restrict__ w, Bias8 bias,
          int C, int H, int W, float *__restrict__ out, float *__restrict__ stats_out) {
    __shared__ float in_t[8][kTH + 2][kTW + 4];
    __shared__ __align__(16) float w_t[8][9][8];
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int x0 = blockIdx.x * kTW, y0 = blockIdx.y * kTH, agent = blockIdx.z;
    const size_t plane = (size_t)H * W;
    const int cin = C + 2;
    float acc[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = bias.b[o];

    for (int c0 = 0; c0 < cin; c0 += 8) {
        for (int i = tid; i < 8 * (kTH + 2) * (kTW + 2); i += 256) {
            const int ci = i / ((kTH + 2) * (kTW + 2)), rem = i % ((kTH + 2) * (kTW + 2));
            const int r = rem / (kTW + 2), c = rem % (kTW + 2);
            const int gy = y0 - 1 + r, gx = x0 - 1 + c, ch = c0 + ci;
            float v = 0.0f;
            if (ch < cin && gy >= 0 && gy < H && gx >= 0 && gx < W) {
                const float *src = ch < 2 ? cond + ((size_t)agent * 2 + ch) * plane
                                          : x + ((size_t)agent * C + (ch - 2)) * plane;
                v = __ldg(src + (size_t)gy * W + gx);
            }
            in_t[ci][r][c] = v;
        }
        for (int i = tid; i < 8 * 72; i += 256) {
            const int ci = i / 72;
            (&w_t[0][0][0])[i] = (c0 + ci < cin) ? __ldg(w + (size_t)c0 * 72 + i) : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int ci = 0; ci < 8; ++ci) {
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const float v = in_t[ci][ty + ky][tx + kx];
                    const float4 w0 = *reinterpret_cast<const float4 *>(&w_t[ci][ky * 3 + kx][0]);
                    const float4 w1 = *reinterpret_cast<const float4 *>(&w_t[ci][ky * 3 + kx][4]);
                    acc[0] = fmaf(v, w0.x, acc[0]); acc[1] = fmaf(v, w0.y, acc[1]);
                    acc[2] = fmaf(v, w0.z, acc[2]); acc[3] = fmaf(v, w0.w, acc[3]);
                    acc[4] = fmaf(v, w1.x, acc[4]); acc[5] = fmaf(v, w1.y, acc[5]);
                    acc[6] = fmaf(v, w1.z, acc[6]); acc[7] = fmaf(v, w1.w, acc[7]);
                }
            }
        }
        __syncthreads();
    }
    const int y = y0 + ty, xx = x0 + tx;
    if (y < H && xx < W) {
        float4 *dst = reinterpret_cast<float4 *>(out + (((size_t)agent * H + y) * W + xx) * 8);
        dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
        dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    } else {
#pragma unroll
        for (int o = 0; o < 8; ++o) acc[o] = 0.0f;
    }
    write_tile_stats(acc, stats_out, agent);
}

// ------------------------------------------------------------------------------------------------
// norm_out + swish + conv_out: 8 (NHWC8) -> C channels (NCHW), with the sampler update fused into
// the epilogue.  unet.py:341-343, cond_diff.py:272-279, :310-313.
//   mode 0 (t == 0):  pred = x0
//   mode 1 (t  > 0):  x_t <- (c1*x0 + c2*x_t) + sigma*noise        (in place, x_{t-1})
// weights: device [C][9][8] (cout, tap, cin), bias device [C].  grid.z = agent * (C/64) + split.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_conv_out(const float *__restrict__ in, const float *__restrict__ st_in, int tiles_in,
           const float *__restrict__ w, const float *__restrict__ bias, Affine8 aff, int C, int H, int W, int mode,
           float c1, float c2, float sigma, const float *__restrict__ noise, float *__restrict__ x,
           float *__restrict__ pred) {
    __shared__ float4 tile[2][kTH + 2][kTW + 2];
    __shared__ __align__(16) float w_s[64][72];
    __shared__ float b_s[64];
    __shared__ float s_ga[8], s_gb[8];
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int splits = (C + 63) / 64;
    const int agent = blockIdx.z / splits, co0 = (blockIdx.z % splits) * 64;
    const int x0 = blockIdx.x * kTW, y0 = blockIdx.y * kTH;
    const int nco = min(64, C - co0);

    if (tid < 8) gn_coeff<8>(tid, agent, st_in, st_in, tiles_in, tiles_in, H * W, aff.gamma[tid], aff.beta[tid], &s_ga[tid], &s_gb[tid]);
    for (int i = tid; i < nco * 72; i += 256) (&w_s[0][0])[i] = __ldg(w + (size_t)co0 * 72 + i);
    if (tid < nco) b_s[tid] = __ldg(bias + co0 + tid);
    __syncthreads();
    for (int i = tid; i < 2 * (kTH + 2) * (kTW + 2); i += 256) {
        const int q = i / ((kTH + 2) * (kTW + 2)), rem = i % ((kTH + 2) * (kTW + 2));
        const int r = rem / (kTW + 2), c = rem % (kTW + 2);
        const int gy = y0 - 1 + r, gx = x0 - 1 + c;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            v = __ldg(reinterpret_cast<const float4 *>(in + (((size_t)agent * H + gy) * W + gx) * 8 + q * 4));
            v.x = swish(fmaf(v.x, s_ga[4 * q + 0], s_gb[4 * q + 0]));
            v.y = swish(fmaf(v.y, s_ga[4 * q + 1], s_gb[4 * q + 1]));
            v.z = swish(fmaf(v.z, s_ga[4 * q + 2], s_gb[4 * q + 2]));
            v.w = swish(fmaf(v.w, s_ga[4 * q + 3], s_gb[4 * q + 3]));
        }
        tile[q][r][c] = v;
    }
    __syncthreads();

    float4 inr[9][2];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            inr[ky * 3 + kx][0] = tile[0][ty + ky][tx + kx];
            inr[ky * 3 + kx][1] = tile[1][ty + ky][tx + kx];
        }
    }
    const int y = y0 + ty, xx = x0 + tx;
    if (y >= H || xx >= W) return;   // no barriers below
    const size_t plane = (size_t)H * W;
    size_t idx = ((size_t)agent * C + co0) * plane + (size_t)y * W + xx;
#pragma unroll 1
    for (int o = 0; o < nco; ++o, idx += plane) {
        const float4 *wr = reinterpret_cast<const float4 *>(&w_s[o][0]);
        float acc = b_s[o];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const float4 wa = wr[2 * t], wb = wr[2 * t + 1];
            acc = fmaf(inr[t][0].x, wa.x, acc); acc = fmaf(inr[t][0].y, wa.y, acc);
            acc = fmaf(inr[t][0].z, wa.z, acc); acc = fmaf(inr[t][0].w, wa.w, acc);
            acc = fmaf(inr[t][1].x, wb.x, acc); acc = fmaf(inr[t][1].y, wb.y, acc);
            acc = fmaf(inr[t][1].z, wb.z, acc); acc = fmaf(inr[t][1].w, wb.w, acc);
        }
        if (mode == 0) {
            pred[idx] = acc;
        } else {
            const float mean = __fadd_rn(__fmul_rn(c1, acc), __fmul_rn(c2, x[idx]));
            x[idx] = __fadd_rn(mean, __fmul_rn(sigma, __ldg(noise + idx)));
        }
    }
}

// q_sample of the ego feature of each agent's frame: x_T = sa * ego + sb * noise0.  cond_diff.py:333-337, :372
__global__ void __launch_bounds__(256)
k_q_sample(const float *__restrict__ feat, const int32_t *__restrict__ agent_offsets, int n_frames,
           const float *__restrict__ noise0, float sa, float sb, size_t per_agent, float *__restrict__ x) {
    const int agent = blockIdx.y;
    int lo = 0, hi = n_frames;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(agent_offsets + mid) <= agent) lo = mid; else hi = mid;
    }
    const float4 *ego = reinterpret_cast<const float4 *>(feat + (size_t)__ldg(agent_offsets + lo) * per_agent);
    const float4 *nz = reinterpret_cast<const float4 *>(noise0 + (size_t)agent * per_agent);
    float4 *dst = reinterpret_cast<float4 *>(x + (size_t)agent * per_agent);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_agent / 4; i += (size_t)gridDim.x * blockDim.x) {
        const float4 e = __ldg(ego + i), n = __ldg(nz + i);
        float4 r;
        r.x = __fadd_rn(__fmul_rn(sa, e.x), __fmul_rn(sb, n.x));
        r.y = __fadd_rn(__fmul_rn(sa, e.y), __fmul_rn(sb, n.y));
        r.z = __fadd_rn(__fmul_rn(sa, e.z), __fmul_rn(sb, n.z));
        r.w = __fadd_rn(__fmul_rn(sa, e.w), __fmul_rn(sb, n.w));
        dst[i] = r;
    }
}

// ------------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------------
struct Act {          // NHWC8 activation + per-tile statistics
    float *data, *stats;
    int H, W, tiles;
};

struct UnetWorkspace {
    float *x;                 // [A][C][H][W] current x_t (NCHW)
    void *tc_packed;          // bf16 B operands of conv_in / conv_out (denoiser_tc.cu)
    Act p[12], q[15];
    size_t bytes;
};

static inline int tiles_of(int H, int W) { return ((W + kTW - 1) / kTW) * ((H + kTH - 1) / kTH); }

static UnetWorkspace carve_unet(void *base, int A, int C, int H, int W) {
    UnetWorkspace ws;
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align_up(bytes, 256);
        return (float *)p;
    };
    ws.x = take((size_t)A * C * H * W * 4);
    ws.tc_packed = take(conv_tc_packed_bytes(C));
    auto mk = [&](int h, int w) {
        Act a;
        a.H = h; a.W = w; a.tiles = tiles_of(h, w);
        a.data = take((size_t)A * h * w * 8 * 4);
        a.stats = take((size_t)A * a.tiles * 8 * 4);
        return a;
    };
    for (auto &a : ws.p) a = mk(H, W);
    for (auto &a : ws.q) a = mk(H / 2, W / 2);
    ws.bytes = off;
    return ws;
}

static int g_precision = 0;   // set by unet_eval for the launch helpers below (host-side, per call)

template <int CIN, bool PRE_GN, int GEOM, int RES>
static void launch_c8(cudaStream_t st, int A, const Act &ia, const Act *ib, const Act *ra, const Act *rb, Act &o,
                      const C8Params &prm) {
    if ((g_precision & GC_PREC_TC_MIDDLE) && conv_c8_tc_eligible(GEOM, o.H, o.W)) {   // tf32 tensor cores
        int tiles = 0;
        if (conv_c8_tc(st, A, CIN, PRE_GN, GEOM, RES, ia.data, ib ? ib->data : ia.data, ia.stats, ib ? ib->stats : ia.stats,
                       ia.tiles, ib ? ib->tiles : ia.tiles, ra ? ra->data : nullptr, rb ? rb->data : nullptr, o.data, o.stats,
                       o.H, o.W, prm, &tiles) == GC_OK) {
            o.tiles = tiles;
            return;
        }
    }
    o.tiles = tiles_of(o.H, o.W);
    const dim3 grid((o.W + kTW - 1) / kTW, (o.H + kTH - 1) / kTH, A);
    k_conv_c8<CIN, PRE_GN, GEOM, RES><<<grid, 256, 0, st>>>(
        ia.data, ib ? ib->data : ia.data, ia.stats, ib ? ib->stats : ia.stats, ia.tiles, ib ? ib->tiles : ia.tiles,
        ra ? ra->data : nullptr,
        rb ? rb->data : nullptr, o.data, o.stats, o.H, o.W, prm);
}

// ResnetBlock (unet.py:117-138) on an 8-channel input
static void resblock8(cudaStream_t st, int A, const Act &x, Act &h1, Act &o, const C8Params *prm) {
    launch_c8<8, true, kSame, kNone>(st, A, x, nullptr, nullptr, nullptr, h1, prm[0]);
    launch_c8<8, true, kSame, kIdent>(st, A, h1, nullptr, &x, nullptr, o, prm[1]);
}
// ResnetBlock on cat([h, skip]) (16 channels) with nin_shortcut
static void resblock16(cudaStream_t st, int A, const Act &h, const Act &skip, Act &h1, Act &o, const C8Params *prm) {
    launch_c8<16, true, kSame, kNone>(st, A, h, &skip, nullptr, nullptr, h1, prm[0]);
    launch_c8<8, true, kSame, kNin>(st, A, h1, nullptr, &h, &skip, o, prm[1]);
}

struct HostTail {     // trailing part of the host weight blob, after T * kC8Layers C8Params
    float conv_in_bias[8];
    float norm_out_gamma[8], norm_out_beta[8];
};

// Tensor k of the layer trace of gc_unet_trace: hs0 (k = 0) or the output of middle layer k - 1, [A][h][w][8]; layers
// 4 .. 18 (k = 5 .. 19) are half resolution.
static size_t trace_offset(int k, int A, int H, int W) {
    const int half = k < 5 ? 0 : (k > 20 ? 15 : k - 5);
    return (size_t)A * ((size_t)(k - half) * H * W * 8 + (size_t)half * (H / 2) * (W / 2) * 8);
}
static void trace_copy(cudaStream_t st, const Act &a, int k, int A, int H, int W, float *trace) {
    cudaMemcpyAsync(trace + trace_offset(k, A, H, W), a.data, (size_t)A * a.H * a.W * 8 * 4, cudaMemcpyDeviceToDevice, st);
}

// One DiffusionUNet evaluation; the result goes through k_conv_out's epilogue.  trace (gc_unet_trace, else NULL): every
// layer's output is also written there.
static int unet_eval(cudaStream_t st, int A, int C, int H, int W, const float *cond, UnetWorkspace &ws,
                     const C8Params *prm, const HostTail &tail, const float *w_in, const float *w_out,
                     const float *b_out, int mode, float c1, float c2, float sigma, const float *noise, float *pred,
                     int precision, const float *rec_dev, float *trace = nullptr) {
    Act *p = ws.p, *q = ws.q;
    g_precision = precision;
    // cluster-resident middle (denoiser_cluster.cu): conv_in -> ONE launch for the 26 width-8 layers -> conv_out
    if ((precision & GC_PREC_CLUSTER) && rec_dev != nullptr && (precision & GC_PREC_BF16_TC) == GC_PREC_BF16_TC &&
        unet_cluster_eligible(C, H, W) && conv_in_tc_eligible(C, H, W) && conv_out_tc_eligible(C, H, W)) {
        Bias8 bi;
        for (int i = 0; i < 8; ++i) bi.b[i] = tail.conv_in_bias[i];
        if (conv_in_tc2_eligible(C, H, W) && !getenv("GC_CONV_IN_V1")) {
            p[0].tiles = conv_in_tc2_tiles(H);
            if (int rc = conv_in_tc2(st, A, cond, ws.x, ws.tc_packed, bi, C, H, W, p[0].data, p[0].stats)) return rc;
        } else {
            p[0].tiles = conv_in_tc_tiles(H, W);
            if (int rc = conv_in_tc(st, A, cond, ws.x, ws.tc_packed, bi, C, H, W, p[0].data, p[0].stats)) return rc;
        }
        if (int rc = unet_middle_cluster(st, A, p[0].data, rec_dev, p[11].data, p[11].stats, trace)) return rc;
        p[11].tiles = kCl;
        Affine8 aff;
        for (int i = 0; i < 8; ++i) { aff.gamma[i] = tail.norm_out_gamma[i]; aff.beta[i] = tail.norm_out_beta[i]; }
        if (trace) {   // hs0 and the last layer's output are in p[0] / p[11]; the kernel wrote the others
            trace_copy(st, p[0], 0, A, H, W, trace);
            trace_copy(st, p[11], kC8Layers, A, H, W, trace);
        }
        return conv_out_tc(st, A, p[11].data, p[11].stats, p[11].tiles, ws.tc_packed, b_out, aff, C, H, W, mode, c1, c2, sigma,
                           noise, ws.x, pred, 0);
    }
    Bias8 bi;
    for (int i = 0; i < 8; ++i) bi.b[i] = tail.conv_in_bias[i];
    const dim3 gridP((W + kTW - 1) / kTW, (H + kTH - 1) / kTH, A);
    if ((precision & GC_PREC_TC_CONV_IN) && conv_in_tc2_eligible(C, H, W) && !getenv("GC_CONV_IN_V1")) {   // hs[0], tcgen05
        p[0].tiles = conv_in_tc2_tiles(H);
        if (int rc = conv_in_tc2(st, A, cond, ws.x, ws.tc_packed, bi, C, H, W, p[0].data, p[0].stats)) return rc;
    } else if ((precision & GC_PREC_TC_CONV_IN) && conv_in_tc_eligible(C, H, W)) {
        p[0].tiles = conv_in_tc_tiles(H, W);
        if (int rc = conv_in_tc(st, A, cond, ws.x, ws.tc_packed, bi, C, H, W, p[0].data, p[0].stats)) return rc;
    } else {
        k_conv_in<<<gridP, 256, 0, st>>>(cond, ws.x, w_in, bi, C, H, W, p[0].data, p[0].stats);     // hs[0]
    }
    resblock8(st, A, p[0], p[1], p[2], prm + 0);                                                   // down.0.block.0 -> hs[1]
    resblock8(st, A, p[2], p[3], p[4], prm + 2);                                                   // down.0.block.1 -> hs[2]
    launch_c8<8, false, kDown, kNone>(st, A, p[4], nullptr, nullptr, nullptr, q[0], prm[4]);       // downsample -> hs[3]
    resblock8(st, A, q[0], q[1], q[2], prm + 5);                                                   // down.1.block.0 -> hs[4]
    resblock8(st, A, q[2], q[3], q[4], prm + 7);                                                   // down.1.block.1 -> hs[5]
    resblock8(st, A, q[4], q[5], q[6], prm + 9);                                                   // mid.block_1
    resblock8(st, A, q[6], q[7], q[8], prm + 11);                                                  // mid.block_2
    resblock16(st, A, q[8], q[4], q[9], q[10], prm + 13);                                          // up.1.block.0  (pops hs[5])
    resblock16(st, A, q[10], q[2], q[11], q[12], prm + 15);                                        // up.1.block.1  (pops hs[4])
    resblock16(st, A, q[12], q[0], q[13], q[14], prm + 17);                                        // up.1.block.2  (pops hs[3])
    launch_c8<8, false, kUp, kNone>(st, A, q[14], nullptr, nullptr, nullptr, p[5], prm[19]);       // up.1.upsample
    resblock16(st, A, p[5], p[4], p[6], p[7], prm + 20);                                           // up.0.block.0  (pops hs[2])
    resblock16(st, A, p[7], p[2], p[8], p[9], prm + 22);                                           // up.0.block.1  (pops hs[1])
    resblock16(st, A, p[9], p[0], p[10], p[11], prm + 24);                                         // up.0.block.2  (pops hs[0])
    if (trace) {   // tensor k: p[0 .. 4] = hs0, layers 0 .. 3; q[0 .. 14] = layers 4 .. 18; p[5 .. 11] = layers 19 .. 25
        for (int k = 0; k <= kC8Layers; ++k) trace_copy(st, k < 5 ? p[k] : (k < 20 ? q[k - 5] : p[k - 15]), k, A, H, W, trace);
    }
    Affine8 aff;
    for (int i = 0; i < 8; ++i) { aff.gamma[i] = tail.norm_out_gamma[i]; aff.beta[i] = tail.norm_out_beta[i]; }
    if ((precision & GC_PREC_TC_CONV_OUT) && conv_out_tc_eligible(C, H, W)) {
        if (int rc = conv_out_tc(st, A, p[11].data, p[11].stats, p[11].tiles, ws.tc_packed, b_out, aff, C, H, W, mode, c1, c2,
                                 sigma, noise, ws.x, pred, (precision & GC_PREC_TC_MATERIALIZE) ? 1 : 0))
            return rc;
    } else {
        const int splits = (C + 63) / 64;
        const dim3 gridO(gridP.x, gridP.y, A * splits);
        k_conv_out<<<gridO, 256, 0, st>>>(p[11].data, p[11].stats, p[11].tiles, w_out, b_out, aff, C, H, W, mode, c1, c2,
                                          sigma, noise, ws.x, pred);
    }
    GC_LAUNCH_CHECK("unet_eval");
    return GC_OK;
}

}  // namespace gc

using namespace gc;

extern "C" size_t gc_gencomm_host_weight_floats(int T) {
    return (size_t)T * kC8Layers * (sizeof(C8Params) / 4) + sizeof(HostTail) / 4;
}

extern "C" size_t gc_gencomm_cluster_weight_floats(int T) { return (size_t)T * kClLayers * kClRecFloats; }

extern "C" size_t gc_gencomm_device_weight_floats(int C) {
    return (size_t)(C + 2) * 72 + (size_t)C * 72 + (size_t)C;
}

extern "C" size_t gc_gencomm_workspace_bytes(int total_agents, int C, int H, int W) {
    if (total_agents <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
    return carve_unet(nullptr, total_agents, C, H, W).bytes;
}

static int check_unet_args(int A, int C, int H, int W, int T) {
    GC_REQUIRE(A > 0 && C > 0 && H > 0 && W > 0 && T > 0, GC_EINVAL, "gencomm: bad sizes");
    GC_REQUIRE(H % 2 == 0 && W % 2 == 0, GC_EUNSUPPORTED, "gencomm: H and W must be even (one down/up-sampling level)");
    GC_REQUIRE((size_t)C * H * W % 4 == 0, GC_EUNSUPPORTED, "gencomm: C*H*W must be a multiple of 4");
    GC_REQUIRE(A * ((C + 63) / 64) <= 65535 && (H + kTH - 1) / kTH <= 65535, GC_EUNSUPPORTED, "gencomm: grid too large");
    return GC_OK;
}

extern "C" size_t gc_unet_trace_floats(int total_agents, int H, int W) {
    if (total_agents <= 0 || H <= 0 || W <= 0) return 0;
    return trace_offset(kC8Layers + 1, total_agents, H, W);
}

static int unet_forward(const char *name, const float *cond, const float *x, int total_agents, int t_index,
                        const float *w_host, const float *w_dev, const float *w_cluster_dev, int C, int H, int W, int T,
                        int precision, void *workspace, float *pred, float *trace, void *stream) {
    if (int rc = check_unet_args(total_agents, C, H, W, T)) return rc;
    GC_REQUIRE(cond && x && w_host && w_dev && workspace && pred, GC_EINVAL, "%s: null pointer", name);
    GC_REQUIRE(t_index >= 0 && t_index < T, GC_EINVAL, "%s: bad timestep", name);
    cudaStream_t st = (cudaStream_t)stream;
    UnetWorkspace ws = carve_unet(workspace, total_agents, C, H, W);
    cudaMemcpyAsync(ws.x, x, (size_t)total_agents * C * H * W * 4, cudaMemcpyDeviceToDevice, st);
    const C8Params *prm = reinterpret_cast<const C8Params *>(w_host) + (size_t)t_index * kC8Layers;
    const HostTail &tail = *reinterpret_cast<const HostTail *>(reinterpret_cast<const C8Params *>(w_host) + (size_t)T * kC8Layers);
    const float *w_in = w_dev, *w_out = w_dev + (size_t)(C + 2) * 72, *b_out = w_out + (size_t)C * 72;
    if (precision & GC_PREC_BF16_TC)
        if (int rc = conv_tc_pack_weights(st, w_in, w_out, C, ws.tc_packed)) return rc;
    return unet_eval(st, total_agents, C, H, W, cond, ws, prm, tail, w_in, w_out, b_out, 0, 0.f, 0.f, 0.f, nullptr, pred,
                     precision, w_cluster_dev ? w_cluster_dev + (size_t)t_index * kClLayers * kClRecFloats : nullptr, trace);
}

// One denoiser evaluation x0 = UNet(cat[cond, x], t) for tests/diagnostics: writes pred [A][C][H][W].
extern "C" int gc_unet_forward(const float *cond, const float *x, int total_agents, int t_index, const float *w_host,
                               const float *w_dev, const float *w_cluster_dev, int C, int H, int W, int T, int precision,
                               void *workspace, float *pred, void *stream) {
    return unet_forward("gc_unet_forward", cond, x, total_agents, t_index, w_host, w_dev, w_cluster_dev, C, H, W, T, precision,
                        workspace, pred, nullptr, stream);
}

// gc_unet_forward that also writes hs0 and every middle layer's output to trace (include/gencomm_b200.h).
extern "C" int gc_unet_trace(const float *cond, const float *x, int total_agents, int t_index, const float *w_host,
                             const float *w_dev, const float *w_cluster_dev, int C, int H, int W, int T, int precision,
                             void *workspace, float *pred, float *trace, void *stream) {
    GC_REQUIRE(trace, GC_EINVAL, "gc_unet_trace: null pointer");
    return unet_forward("gc_unet_trace", cond, x, total_agents, t_index, w_host, w_dev, w_cluster_dev, C, H, W, T, precision,
                        workspace, pred, trace, stream);
}

extern "C" int gc_gencomm_sample(const float *feat, const float *cond, const int32_t *agent_offsets, int n_frames,
                                 int total_agents, const float *noise0, const float *step_noise,
                                 const float *w_host, const float *w_dev, const float *w_cluster_dev,
                                 const float *schedule_host, int C, int H, int W, int T, int precision, void *workspace,
                                 float *pred, void *stream) {
    if (int rc = check_unet_args(total_agents, C, H, W, T)) return rc;
    GC_REQUIRE(feat && cond && agent_offsets && noise0 && w_host && w_dev && schedule_host && workspace && pred,
               GC_EINVAL, "gc_gencomm_sample: null pointer");
    GC_REQUIRE(T == 1 || step_noise, GC_EINVAL, "gc_gencomm_sample: step_noise required for T > 1");
    GC_REQUIRE(n_frames > 0 && n_frames <= total_agents, GC_EINVAL, "gc_gencomm_sample: bad frame count");
    cudaStream_t st = (cudaStream_t)stream;
    UnetWorkspace ws = carve_unet(workspace, total_agents, C, H, W);
    const size_t per_agent = (size_t)C * H * W;
    const HostTail &tail = *reinterpret_cast<const HostTail *>(reinterpret_cast<const C8Params *>(w_host) + (size_t)T * kC8Layers);
    const float *w_in = w_dev, *w_out = w_dev + (size_t)(C + 2) * 72, *b_out = w_out + (size_t)C * 72;
    // schedule_host: [T][5] = sqrt_alphas_cumprod, sqrt_one_minus_alphas_cumprod, posterior_mean_coef1,
    //                         posterior_mean_coef2, exp(0.5 * posterior_log_variance_clipped)
    if (precision & GC_PREC_BF16_TC)
        if (int rc = conv_tc_pack_weights(st, w_in, w_out, C, ws.tc_packed)) return rc;
    const float *sT = schedule_host + (size_t)(T - 1) * 5;
    int gx = (int)((per_agent / 4 + 255) / 256);
    gx = gx > 1024 ? 1024 : gx;
    k_q_sample<<<dim3(gx, total_agents), 256, 0, st>>>(feat, agent_offsets, n_frames, noise0, sT[0], sT[1], per_agent, ws.x);
    GC_LAUNCH_CHECK("k_q_sample");
    for (int t = T - 1; t >= 0; --t) {
        const C8Params *prm = reinterpret_cast<const C8Params *>(w_host) + (size_t)t * kC8Layers;
        const float *s = schedule_host + (size_t)t * 5;
        const float *nz = t > 0 ? step_noise + (size_t)(T - 1 - t) * total_agents * per_agent : nullptr;
        int rc = unet_eval(st, total_agents, C, H, W, cond, ws, prm, tail, w_in, w_out, b_out, t > 0 ? 1 : 0, s[2], s[3],
                           s[4], nz, pred, precision,
                           w_cluster_dev ? w_cluster_dev + (size_t)t * kClLayers * kClRecFloats : nullptr);
        if (rc) return rc;
    }
    return GC_OK;
}
