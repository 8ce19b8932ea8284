// Enhancer for sm_100a (SURVEY.md section 8f, rank 1): the feature-refinement block GenComm applies to the received /
// generated BEV features before fusion.
//
// Replaces (paths relative to /root/reference/opencood):
//   models/gencomm_modules/enhancer.py:335-383  Enhancer.forward       (only block_1 + split_attn are evaluated, :369-374)
//   :316-333  Enhancer_block.forward   x1 = x + LN1(x)  (the attention call is commented out, :326);  x2 = x1 + FRFN(LN2(x1))
//   :205-250  FRFN.forward             partial 3x3 conv on C/4 channels, Linear C -> 4C + GELU, depth-wise 3x3 + GELU on one
//                                      half gated by the other, Linear 2C -> C
//   :286-314  SplitAttn.forward        global average pool -> fc1 -> LayerNorm -> ReLU -> fc2 -> sigmoid -> scale
// Everything is per agent, so all agents of all frames run in one pass (regroup / record_len only split and re-join).
//
// The three dense contractions (98 % of the 1.8 GFLOP per agent at C = 128) run on tcgen05 as plane-convolution layers
// (conv_layer.cuh) in "bf16x3" (value + residual bf16 planes of both operands, three MMAs per K = 16 step,
// fp32 accumulation in TMEM -- fp32-grade results):
//   partial_conv3 : N = C/4, plain 3x3           K = 9 C/4
//   linear1+GELU  : N = 256, 1x1, GELU  x C/64   K = C,   N = 4C in chunks of 256 TMEM columns
//   linear2       : N = 128, 1x1        x C/128  K = 2C,  N = C
// fed by k_me_to_nhwc (NCHW fp32 -> channel-last bf16 planes).  LayerNorms, the depth-wise convolution + gate, the
// pool / excite and the final scale are fp32 CUDA-core kernels (thread = pixel, plane-coalesced).
// linear1 writes its GELU'd output channel-last (fp32) and the depth-wise + gate kernel turns it directly into linear2's
// bf16 operand planes; the other intermediates are still NCHW fp32 tensors between the kernels (DESIGN.md section 5c).
#include <stdlib.h>

#include "common.cuh"
#include "conv_layer.cuh"
#include "implicit_gemm.cuh"

namespace gc {
namespace enh {

using namespace me;

// small fp32 parameters, one device blob (floats); C = channels
struct Prm {
    int n1w, n1b, n2w, n2b, l1b, dww, dwb, l2b, fc1, bnw, bnb, fc2, total;
};
__host__ __device__ inline Prm prm_layout(int C) {
    Prm p;
    int o = 0;
    p.n1w = o; o += C;          // block_1.norm1.weight
    p.n1b = o; o += C;          // block_1.norm1.bias
    p.n2w = o; o += C;          // block_1.norm2.weight
    p.n2b = o; o += C;          // block_1.norm2.bias
    p.l1b = o; o += 4 * C;      // block_1.mlp.linear1.0.bias
    p.dww = o; o += 2 * C * 9;  // block_1.mlp.dwconv.0.weight [2C][1][3][3]
    p.dwb = o; o += 2 * C;      // block_1.mlp.dwconv.0.bias
    p.l2b = o; o += C;          // block_1.mlp.linear2.0.bias
    p.fc1 = o; o += C * C;      // split_attn.fc1.weight [C][C]
    p.bnw = o; o += C;          // split_attn.bn1.weight
    p.bnb = o; o += C;          // split_attn.bn1.bias
    p.fc2 = o; o += C * C;      // split_attn.fc2.weight [C][C]
    p.total = o;
    return p;
}

// x1 = x + LN1(x);  y = LN2(x1)   (nn.LayerNorm over C, eps 1e-5, biased variance).  thread = pixel; the channel loops
// re-read the thread's own column of planes (L1 / L2 resident: 128 pixels x C x 4 B per CTA).  grid = (HW/128, A), 128 thr.
__global__ void __launch_bounds__(128)
k_enh_ln(const float *__restrict__ x, const float *__restrict__ prm, Prm L, int C, int HW, float *__restrict__ x1,
         float *__restrict__ y) {
    const int a = blockIdx.y, p = blockIdx.x * 128 + threadIdx.x;
    if (p >= HW) return;
    const float *xs = x + (size_t)a * C * HW + p;
    float *x1s = x1 + (size_t)a * C * HW + p, *ys = y + (size_t)a * C * HW + p;
    const float inv_c = 1.0f / (float)C;
    // three passes over the thread's column of planes instead of five: the variances come from sum / sum of squares
    // (C values of O(1) magnitude: the cancellation error is ~1e-6 of the variance)
    float s = 0.0f, q = 0.0f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) { const float v = __ldg(xs + (size_t)c * HW); s += v; q = fmaf(v, v, q); }
    const float m0 = s * inv_c;
    const float r0 = rsqrtf(fmaxf(q * inv_c - m0 * m0, 0.0f) + 1e-5f);
    s = 0.0f; q = 0.0f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) {
        const float v = __ldg(xs + (size_t)c * HW);
        const float t = v + ((v - m0) * r0 * __ldg(prm + L.n1w + c) + __ldg(prm + L.n1b + c));
        x1s[(size_t)c * HW] = t;
        s += t;
        q = fmaf(t, t, q);
    }
    const float m1 = s * inv_c;
    const float r1 = rsqrtf(fmaxf(q * inv_c - m1 * m1, 0.0f) + 1e-5f);
#pragma unroll 8
    for (int c = 0; c < C; ++c)
        ys[(size_t)c * HW] = (x1s[(size_t)c * HW] - m1) * r1 * __ldg(prm + L.n2w + c) + __ldg(prm + L.n2b + c);
}

// v[c] = GELU(dwconv3x3(u[c]) + b[c]) * u[2C + c]   for c < 2C (FRFN gate, enhancer.py:241-246), channel-last:
// u [A][HW][4C] f32 (linear1 epilogue EPI = 2)  ->  v as bf16 value + residual planes [A][HW][2C], i.e. directly the A
// operand of linear2.  (The first version kept u and v as NCHW fp32 tensors: thread = pixel, 535 us, then 310 us with a
// sliding 3x3 register window over 8 rows, plus an NCHW -> channel-last conversion of v.)
// Any W.
// CTA = 8 pixels of a row x kDwRows rows x 128 channels; thread = (x, channel quad) walks the rows with a sliding 3x3 window
// of float4 in registers, so every u element is fetched once per CTA (+ halo: 1.56x) instead of by nine pixel threads
// of different CTAs through L2 (first channel-last version, one thread per (pixel, quad): 422 us).
// grid = (ceil(W/8) * ceil(H/kDwRows), 2C/128, A), 256 threads.
constexpr int kDwRows = 8;
__global__ void __launch_bounds__(256)
k_enh_dw_cl(const float *__restrict__ u, const float *__restrict__ prm, Prm L, int C, int H, int W,
            uint2 *__restrict__ vh, uint2 *__restrict__ vl) {
    __shared__ __align__(16) float s_dw[10][128];   // [9 taps + bias][128 channels of this CTA]
    const int C2 = 2 * C, c0 = blockIdx.y * 128, a = blockIdx.z, HW = H * W;
    for (int i = threadIdx.x; i < 128 * 9; i += 256) s_dw[i % 9][i / 9] = prm[L.dww + (c0 + i / 9) * 9 + i % 9];
    if (threadIdx.x < 128) s_dw[9][threadIdx.x] = prm[L.dwb + c0 + threadIdx.x];
    __syncthreads();
    const int xb = (W + 7) / 8;
    const int x = (blockIdx.x % xb) * 8 + (threadIdx.x >> 5), r0 = (blockIdx.x / xb) * kDwRows;
    const int q = threadIdx.x & 31;             // channel quad within the CTA's 128 channels
    if (x >= W) return;
    const float4 *ub = reinterpret_cast<const float4 *>(u + (size_t)a * HW * 4 * C) + (c0 >> 2) + q;   // + pixel * C (float4)
    const bool lok = x > 0, rok = x + 1 < W;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    auto row3 = [&](int r, float4 (&o)[3]) {
        if (r < 0 || r >= H) { o[0] = o[1] = o[2] = z; return; }
        const float4 *p = ub + (size_t)(r * W + x) * C;
        o[0] = lok ? __ldg(p - C) : z;
        o[1] = __ldg(p);
        o[2] = rok ? __ldg(p + C) : z;
    };
    float4 w[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) w[k] = *reinterpret_cast<const float4 *>(&s_dw[k][4 * q]);
    const float4 bias = *reinterpret_cast<const float4 *>(&s_dw[9][4 * q]);
    // software pipeline: the three pixels of row r + 2 and the gate of row r + 1 are in flight while row r is computed (the
    // first version issued the row loads at the top of the iteration and the gate load right before its use: two exposed
    // memory latencies per row at 16 warps per SM -- FMUL / FFMA on just-loaded data took 57 % of the stall samples, 361 us)
    auto gate = [&](int r) { return r < H ? __ldg(ub + (size_t)(r * W + x) * C + (C2 >> 2)) : z; };
    float4 top[3], mid[3], bot[3], nxt[3];
    row3(r0 - 1, top);
    row3(r0, mid);
    row3(r0 + 1, bot);
    float4 g = gate(r0);
#pragma unroll 1
    for (int i = 0; i < kDwRows; ++i) {
        const int r = r0 + i;
        if (r >= H) break;
        row3(r + 2, nxt);
        const float4 g_nxt = gate(r + 1);
        float4 acc = bias;   // tap order ky*3+kx like the reference weight layout
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            acc.x = fmaf(w[k].x, top[k].x, acc.x); acc.y = fmaf(w[k].y, top[k].y, acc.y);
            acc.z = fmaf(w[k].z, top[k].z, acc.z); acc.w = fmaf(w[k].w, top[k].w, acc.w);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            acc.x = fmaf(w[3 + k].x, mid[k].x, acc.x); acc.y = fmaf(w[3 + k].y, mid[k].y, acc.y);
            acc.z = fmaf(w[3 + k].z, mid[k].z, acc.z); acc.w = fmaf(w[3 + k].w, mid[k].w, acc.w);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            acc.x = fmaf(w[6 + k].x, bot[k].x, acc.x); acc.y = fmaf(w[6 + k].y, bot[k].y, acc.y);
            acc.z = fmaf(w[6 + k].z, bot[k].z, acc.z); acc.w = fmaf(w[6 + k].w, bot[k].w, acc.w);
        }
        const size_t pa = (size_t)a * HW + (size_t)r * W + x;
        const float r0v = gelu_erf(acc.x) * g.x, r1v = gelu_erf(acc.y) * g.y, r2v = gelu_erf(acc.z) * g.z,
                    r3v = gelu_erf(acc.w) * g.w;
        const size_t o = pa * (C2 >> 2) + (c0 >> 2) + q;
        vh[o] = make_uint2(pack_bf16(r0v, r1v), pack_bf16(r2v, r3v));
        vl[o] = make_uint2(pack_bf16(bf16_residual(r0v), bf16_residual(r1v)), pack_bf16(bf16_residual(r2v), bf16_residual(r3v)));
#pragma unroll
        for (int k = 0; k < 3; ++k) { top[k] = mid[k]; mid[k] = bot[k]; bot[k] = nxt[k]; }
        g = g_nxt;
    }
}

// s += x1 (residual, enhancer.py:328) and gap[a][c] = mean over the plane (SplitAttn :300-302).  One CTA per plane,
// fixed-order reduction.  grid = (C, A), 256 threads.
__global__ void __launch_bounds__(256)
k_enh_res_gap(const float *__restrict__ x1, float *__restrict__ s, int HW, float *__restrict__ gap) {
    __shared__ float red[8];
    const size_t base = ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * HW;
    float t = 0.0f;
    for (int p = threadIdx.x; p < HW; p += 256) {
        const float v = s[base + p] + __ldg(x1 + base + p);
        s[base + p] = v;
        t += v;
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) t += __shfl_xor_sync(0xffffffffu, t, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        float r = 0.0f;
        for (int i = 0; i < 8; ++i) r += red[i];
        gap[blockIdx.y * gridDim.x + blockIdx.x] = r / (float)HW;
    }
}

// attn = sigmoid(fc2(relu(LN(fc1(gap)))))   (SplitAttn :303-309, RadixSoftmax(1,1) = sigmoid).  grid = A, C threads.
__global__ void k_enh_attn(const float *__restrict__ gap, const float *__restrict__ prm, Prm L, int C, float *__restrict__ attn) {
    extern __shared__ float sh[];   // [C] gap, [C] hidden, [2] stats
    float *s_g = sh, *s_h = sh + C, *s_st = sh + 2 * C;
    const int a = blockIdx.x, c = threadIdx.x;
    s_g[c] = gap[a * C + c];
    __syncthreads();
    float h = 0.0f;
    for (int k = 0; k < C; ++k) h = fmaf(prm[L.fc1 + c * C + k], s_g[k], h);
    s_h[c] = h;
    __syncthreads();
    if (c == 0) {
        float m = 0.0f;
        for (int k = 0; k < C; ++k) m += s_h[k];
        m /= (float)C;
        float q = 0.0f;
        for (int k = 0; k < C; ++k) { const float d = s_h[k] - m; q = fmaf(d, d, q); }
        s_st[0] = m;
        s_st[1] = rsqrtf(q / (float)C + 1e-5f);
    }
    __syncthreads();
    const float hn = fmaxf((h - s_st[0]) * s_st[1] * prm[L.bnw + c] + prm[L.bnb + c], 0.0f);
    __syncthreads();
    s_h[c] = hn;
    __syncthreads();
    float z = 0.0f;
    for (int k = 0; k < C; ++k) z = fmaf(prm[L.fc2 + c * C + k], s_h[k], z);
    attn[a * C + c] = 1.0f / (1.0f + expf(-z));
}

// out = s * attn[a][c]   (SplitAttn :311).  grid = (ceil(HW/1024), C, A), 256 threads x float4.
__global__ void __launch_bounds__(256)
k_enh_scale(const float *__restrict__ s, const float *__restrict__ attn, int HW, float *__restrict__ out) {
    const size_t plane = (size_t)blockIdx.z * gridDim.y + blockIdx.y;
    const float w = __ldg(attn + plane);
    const int i = (blockIdx.x * 256 + threadIdx.x) * 4;
    if (i + 3 < HW) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(s + plane * HW + i));
        *reinterpret_cast<float4 *>(out + plane * HW + i) = make_float4(v.x * w, v.y * w, v.z * w, v.w * w);
    } else {
        for (int k = i; k < HW; ++k) out[plane * HW + k] = __ldg(s + plane * HW + k) * w;
    }
}

struct Workspace {
    float *x1, *y, *u, *s, *gap, *attn;
    uint4 *yh, *yl, *vh, *vl;
    size_t bytes;
};
static Workspace carve(void *base, int A, int C, int HW) {
    Workspace w;
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    const size_t plane = (size_t)A * HW * 4;
    w.x1 = (float *)take(plane * C);
    w.y = (float *)take(plane * C);
    w.u = (float *)take(plane * 4 * C);
    w.s = (float *)take(plane * C);
    w.gap = (float *)take((size_t)A * C * 4);
    w.attn = (float *)take((size_t)A * C * 4);
    w.yh = (uint4 *)take((size_t)A * HW * C * 2);
    w.yl = (uint4 *)take((size_t)A * HW * C * 2);
    w.vh = (uint4 *)take((size_t)A * HW * 2 * C * 2);
    w.vl = (uint4 *)take((size_t)A * HW * 2 * C * 2);
    w.bytes = off;
    return w;
}

// packed bf16x3 B operands: [partial_conv3][linear1: C/64 chunks of 256 rows][linear2: C/128 chunks of 128 rows]
static inline size_t pk_pconv_bytes(int C) { return conv_packed_bytes(9, C / 4, C / 4); }     // N = C/4 rows
static inline size_t pk_lin1_chunk_bytes(int C) { return conv_packed_bytes(1, C, 256); }   // 256 rows per launch
static inline size_t pk_lin2_chunk_bytes(int C) { return conv_packed_bytes(1, 2 * C, 128); }
static inline size_t pk_lin1_off(int C) { return align_up(pk_pconv_bytes(C), 256); }
static inline size_t pk_lin2_off(int C) { return pk_lin1_off(C) + (size_t)(C / 64) * pk_lin1_chunk_bytes(C); }
static inline size_t pk_total(int C) { return pk_lin2_off(C) + (size_t)(C / 128) * pk_lin2_chunk_bytes(C); }

}  // namespace enh
}  // namespace gc

using namespace gc;

extern "C" size_t gc_enhancer_param_floats(int C) { return C > 0 ? (size_t)enh::prm_layout(C).total : 0; }
extern "C" size_t gc_enhancer_packed_bytes(int C) { return C > 0 && C % 128 == 0 ? enh::pk_total(C) : 0; }
extern "C" size_t gc_enhancer_workspace_bytes(int total_agents, int C, int H, int W) {
    if (total_agents <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
    return enh::carve(nullptr, total_agents, C, H * W).bytes;
}

extern "C" int gc_enhancer_pack_weights(const float *w_pconv, const float *w_lin1, const float *w_lin2, int C, void *packed,
                                        void *stream) {
    GC_REQUIRE(w_pconv && w_lin1 && w_lin2 && packed, GC_EINVAL, "gc_enhancer_pack_weights: null pointer");
    GC_REQUIRE(C == 128 || C == 256, GC_EUNSUPPORTED, "gc_enhancer_pack_weights: C must be 128 or 256 (got %d)", C);
    cudaStream_t st = (cudaStream_t)stream;
    char *pk = (char *)packed;
    const int c4 = C / 4;
    // partial_conv3.weight [C/4][C/4][3][3]
    int rc = conv_pack(st, w_pconv, 9, c4, c4, 32, pk);
    for (int j = 0; j < C / 64 && !rc; ++j)   // linear1.weight [4C][C], rows 256 j ..
        rc = conv_pack(st, w_lin1 + (size_t)j * 256 * C, 1, C, 256, 32, pk + enh::pk_lin1_off(C) + j * enh::pk_lin1_chunk_bytes(C));
    for (int j = 0; j < C / 128 && !rc; ++j)   // linear2.weight [C][2C], rows 128 j ..
        rc = conv_pack(st, w_lin2 + (size_t)j * 128 * 2 * C, 1, 2 * C, 128, 32, pk + enh::pk_lin2_off(C) + j * enh::pk_lin2_chunk_bytes(C));
    return rc;
}

extern "C" int gc_enhancer(const float *x, int total_agents, int C, int H, int W, const void *packed, const float *params,
                           void *workspace, float *out, void *stream) {
    GC_REQUIRE(total_agents >= 0 && total_agents <= 65535, GC_EINVAL, "gc_enhancer: bad agent count");
    if (total_agents == 0) return GC_OK;
    GC_REQUIRE(x && packed && params && workspace && out, GC_EINVAL, "gc_enhancer: null pointer");
    GC_REQUIRE(C == 128 || C == 256, GC_EUNSUPPORTED, "gc_enhancer: C must be 128 or 256 (got %d)", C);
    GC_REQUIRE(H > 0 && W > 0 && (H * W) % me::kPix == 0, GC_EUNSUPPORTED,
               "gc_enhancer: H*W must be a multiple of 128 (got %dx%d)", H, W);
    cudaStream_t st = (cudaStream_t)stream;
    const int A = total_agents, HW = H * W, tiles = HW / me::kPix, c4 = C / 4;
    const enh::Workspace ws = enh::carve(workspace, A, C, HW);
    const enh::Prm L = enh::prm_layout(C);
    const char *pk = (const char *)packed;
    const dim3 grid(tiles, A);
    int rc;

    enh::k_enh_ln<<<grid, 128, 0, st>>>(x, params, L, C, HW, ws.x1, ws.y);
    GC_LAUNCH_CHECK("k_enh_ln");
    if ((rc = to_planes(st, ws.y, A, C, HW, ws.yh, ws.yl))) return rc;
    // partial_conv3 on the first C/4 channels, written over planes 0 .. C/4-1 of y (it reads the bf16 planes, not y)
    ConvLayer cv;
    cv.xh = ws.yh; cv.xl = ws.yl; cv.A = A; cv.C = C; cv.c_in = c4; cv.H_in = H; cv.W_in = W; cv.taps = 9;
    cv.w = (const uint4 *)pk; cv.n_pad = conv_n_pad(c4, 32); cv.n_out = c4; cv.epi = 0; cv.out = ws.y; cv.out_ch_total = C;
    if ((rc = conv_layer(st, cv))) return rc;
    if ((rc = to_planes(st, ws.y, A, C, HW, ws.yh, ws.yl))) return rc;
    // linear1 + GELU, 256 output channels (= 256 TMEM columns) per launch: the A operand is staged once per 256 columns
    // (128 per launch was measured first: 4 x 125 us at C = 128)
    cv.c_in = C; cv.taps = 1; cv.n_pad = cv.n_out = 256;
    cv.epi = 2; cv.out = ws.u; cv.out_ch_total = 4 * C;
    for (int j = 0; j < C / 64; ++j) {
        cv.w = (const uint4 *)(pk + enh::pk_lin1_off(C) + j * enh::pk_lin1_chunk_bytes(C));
        cv.bias = params + L.l1b + 256 * j; cv.out_ch_off = 256 * j;
        if ((rc = conv_layer(st, cv))) return rc;
    }
    {   // depth-wise 3x3 + GELU + gate on the channel-last u, straight into linear2's bf16 operand planes
        const dim3 g3(((W + 7) / 8) * ((H + enh::kDwRows - 1) / enh::kDwRows), 2 * C / 128, A);
        enh::k_enh_dw_cl<<<g3, 256, 0, st>>>(ws.u, params, L, C, H, W, (uint2 *)ws.vh, (uint2 *)ws.vl);
        GC_LAUNCH_CHECK("k_enh_dw_cl");
    }
    // linear2
    cv.xh = ws.vh; cv.xl = ws.vl; cv.C = cv.c_in = 2 * C; cv.n_pad = cv.n_out = 128;
    cv.epi = 0; cv.out = ws.s; cv.out_ch_total = C;
    for (int j = 0; j < C / 128; ++j) {
        cv.w = (const uint4 *)(pk + enh::pk_lin2_off(C) + j * enh::pk_lin2_chunk_bytes(C));
        cv.bias = params + L.l2b + 128 * j; cv.out_ch_off = 128 * j;
        if ((rc = conv_layer(st, cv))) return rc;
    }
    enh::k_enh_res_gap<<<dim3(C, A), 256, 0, st>>>(ws.x1, ws.s, HW, ws.gap);
    GC_LAUNCH_CHECK("k_enh_res_gap");
    enh::k_enh_attn<<<A, C, (2 * C + 2) * sizeof(float), st>>>(ws.gap, params, L, C, ws.attn);
    GC_LAUNCH_CHECK("k_enh_attn");
    enh::k_enh_scale<<<dim3((HW + 1023) / 1024, C, A), 256, 0, st>>>(ws.s, ws.attn, HW, out);
    GC_LAUNCH_CHECK("k_enh_scale");
    return GC_OK;
}
