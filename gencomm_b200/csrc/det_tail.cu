// DownsampleConv (shrink header) and the shared detection heads for sm_100a -- the first slice of SURVEY.md section 8f
// rank 2 (the cuDNN layers either side of the fusion).
//
// Replaces (paths relative to /root/reference/opencood):
//   models/sub_modules/downsample_conv.py:7-50   DoubleConv = Conv2d(k, stride s, pad) + ReLU + Conv2d(3x3, pad 1) + ReLU,
//                                                DownsampleConv = a list of them (shipped configs: one 3x3 layer, stride 1 or 2)
//   models/heter_model_baseline.py:130-135        cls_head / reg_head / dir_head: three 1x1 Conv2d on the fused feature
// All of it runs as plane-convolution layers (conv_layer.cuh) in bf16x3 (value + residual bf16 planes of both operands, fp32
// accumulation in TMEM: fp32-grade results): strided / plain 3x3 with a bias + ReLU epilogue, and ONE 1x1 GEMM for the three
// heads (their weight matrices concatenated, N <= 64).
#include "common.cuh"

#include "conv_layer.cuh"

namespace gc {
namespace dt {

// both convolutions of a DoubleConv are packed for N = conv_n_pad(c_out, 32), the second at a 256-byte boundary
static inline size_t second_conv_off(int c_in, int c_out) { return align_up(conv_packed_bytes(9, c_in, conv_n_pad(c_out, 32)), 256); }

struct Ws {
    uint4 *xh, *xl;   // channel-last planes of the current layer's input (sized for the larger of the two layers)
    float *mid;       // [A][N1][Ho*Wo] output of the first convolution
    size_t bytes;
};
static Ws carve(void *base, int A, int cin, int hw_in, int n1, int hw_out) {
    Ws w;
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    const size_t plane = (size_t)A * 2 * ((size_t)cin * hw_in > (size_t)n1 * hw_out ? (size_t)cin * hw_in : (size_t)n1 * hw_out);
    w.xh = (uint4 *)take(plane);
    w.xl = (uint4 *)take(plane);
    w.mid = (float *)take((size_t)A * n1 * hw_out * 4);
    w.bytes = off;
    return w;
}

// DoubleConv on channel-last planes: conv3x3(stride) + ReLU written as planes into `mid` (two planes of A*c_out*Ho*Wo*2 bytes
// = the bytes of one fp32 tensor), conv3x3 + ReLU -> fp32 NCHW.  No fp32 intermediate, no second layout conversion.
static int double_conv_from_planes(cudaStream_t st, int A, const uint4 *xh, const uint4 *xl, int c_in, int H, int W, int stride,
                                   int c_out, const void *packed, const float *bias, float *mid, float *out) {
    ConvLayer L;
    L.xh = xh; L.xl = xl; L.A = A; L.C = L.c_in = c_in; L.H_in = H; L.W_in = W; L.taps = 9; L.stride = stride;
    L.w = (const uint4 *)packed; L.n_pad = conv_n_pad(c_out, 32); L.bias = bias; L.n_out = L.out_ch_total = c_out;
    L.epi = 5; L.oh = (uint4 *)mid; L.ol = (uint4 *)((char *)mid + (size_t)A * c_out * L.Ho() * L.Wo() * 2);
    if (int rc = conv_layer(st, L)) return rc;
    ConvLayer L2 = L;   // the second convolution: stride 1 over the planes the first wrote
    L2.xh = L.oh; L2.xl = L.ol; L2.C = L2.c_in = c_out; L2.H_in = L.Ho(); L2.W_in = L.Wo(); L2.stride = 1;
    L2.w = (const uint4 *)((const char *)packed + second_conv_off(c_in, c_out)); L2.bias = bias + c_out;
    L2.epi = 3; L2.out = out; L2.oh = L2.ol = nullptr;
    return conv_layer(st, L2);
}

}  // namespace dt
}  // namespace gc

using namespace gc;

extern "C" size_t gc_double_conv_packed_bytes(int c_in, int c_out) {
    if (c_in <= 0 || c_out <= 0) return 0;
    return dt::second_conv_off(c_in, c_out) + conv_packed_bytes(9, c_out, conv_n_pad(c_out, 32));
}
extern "C" size_t gc_double_conv_workspace_bytes(int total_agents, int c_in, int H, int W, int stride, int c_out) {
    if (total_agents <= 0 || c_in <= 0 || c_out <= 0 || H <= 0 || W <= 0 || stride <= 0) return 0;
    return dt::carve(nullptr, total_agents, c_in, H * W, c_out, conv_out_size(H, stride) * conv_out_size(W, stride)).bytes;
}
extern "C" int gc_double_conv_pack(const float *w1, const float *w2, int c_in, int c_out, void *packed, void *stream) {
    GC_REQUIRE(w1 && w2 && packed, GC_EINVAL, "gc_double_conv_pack: null pointer");
    GC_REQUIRE(c_in > 0 && c_in % 64 == 0 && c_out > 0 && c_out % 64 == 0 && c_out <= 256, GC_EUNSUPPORTED,
               "gc_double_conv_pack: channels must be multiples of 64, c_out <= 256 (got %d -> %d)", c_in, c_out);
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = conv_pack(st, w1, 9, c_in, c_out, 32, packed)) return rc;
    return conv_pack(st, w2, 9, c_out, c_out, 32, (char *)packed + dt::second_conv_off(c_in, c_out));
}

extern "C" int gc_double_conv(const float *x, int total_agents, int c_in, int H, int W, int stride, int c_out,
                              const void *packed, const float *bias /* [2][c_out] */, void *workspace, float *out,
                              void *stream) {
    GC_REQUIRE(total_agents >= 0 && total_agents <= 65535, GC_EINVAL, "gc_double_conv: bad agent count");
    if (total_agents == 0) return GC_OK;
    GC_REQUIRE(x && packed && bias && workspace && out, GC_EINVAL, "gc_double_conv: null pointer");
    GC_REQUIRE(c_in > 0 && c_in % 64 == 0 && c_out > 0 && c_out % 64 == 0 && c_out <= 256, GC_EUNSUPPORTED,
               "gc_double_conv: channels must be multiples of 64, c_out <= 256 (got %d -> %d)", c_in, c_out);
    GC_REQUIRE(stride == 1 || stride == 2, GC_EUNSUPPORTED, "gc_double_conv: stride must be 1 or 2 (got %d)", stride);
    const int Ho = conv_out_size(H, stride), Wo = conv_out_size(W, stride);
    GC_REQUIRE(H > 0 && W > 0 && (Ho * Wo) % 128 == 0, GC_EUNSUPPORTED,
               "gc_double_conv: output H*W must be a multiple of 128 (got %dx%d)", Ho, Wo);
    cudaStream_t st = (cudaStream_t)stream;
    const int A = total_agents;
    const dt::Ws ws = dt::carve(workspace, A, c_in, H * W, c_out, Ho * Wo);
    if (int rc = to_planes(st, x, A, c_in, H * W, ws.xh, ws.xl)) return rc;
    return dt::double_conv_from_planes(st, A, ws.xh, ws.xl, c_in, H, W, stride, c_out, packed, bias, ws.mid, out);
}
extern "C" size_t gc_double_conv_planes_workspace_bytes(int total_agents, int H, int W, int stride, int c_out) {
    if (total_agents <= 0 || c_out <= 0 || H <= 0 || W <= 0 || stride <= 0) return 0;
    return align_up((size_t)total_agents * c_out * conv_out_size(H, stride) * conv_out_size(W, stride) * 4, 256);
}
extern "C" int gc_double_conv_planes(const void *xh, const void *xl, int total_agents, int c_in, int H, int W, int stride, int c_out,
                                     const void *packed, const float *bias /* [2][c_out] */, void *workspace, float *out,
                                     void *stream) {
    GC_REQUIRE(total_agents >= 0 && total_agents <= 65535, GC_EINVAL, "gc_double_conv_planes: bad agent count");
    if (total_agents == 0) return GC_OK;
    GC_REQUIRE(xh && xl && packed && bias && workspace && out, GC_EINVAL, "gc_double_conv_planes: null pointer");
    GC_REQUIRE(c_in > 0 && c_in % 64 == 0 && c_out > 0 && c_out % 64 == 0 && c_out <= 256, GC_EUNSUPPORTED,
               "gc_double_conv_planes: channels must be multiples of 64, c_out <= 256 (got %d -> %d)", c_in, c_out);
    GC_REQUIRE(stride == 1 || stride == 2, GC_EUNSUPPORTED, "gc_double_conv_planes: stride must be 1 or 2 (got %d)", stride);
    const int Ho = conv_out_size(H, stride), Wo = conv_out_size(W, stride);
    GC_REQUIRE(H > 0 && W > 0 && (Ho * Wo) % 128 == 0, GC_EUNSUPPORTED,
               "gc_double_conv_planes: output H*W must be a multiple of 128 (got %dx%d)", Ho, Wo);
    return dt::double_conv_from_planes((cudaStream_t)stream, total_agents, (const uint4 *)xh, (const uint4 *)xl, c_in, H, W, stride,
                                       c_out, packed, bias, (float *)workspace, out);
}

extern "C" size_t gc_det_heads_packed_bytes(int C, int n_out) {
    return C > 0 && n_out > 0 ? conv_packed_bytes(1, C, conv_n_pad(n_out, 32)) : 0;
}
extern "C" size_t gc_det_heads_workspace_bytes(int n_frames, int C, int H, int W) {
    if (n_frames <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
    return 2 * align_up((size_t)n_frames * H * W * C * 2, 256);
}
extern "C" int gc_det_heads_pack(const float *w /* [n_out][C] */, int C, int n_out, void *packed, void *stream) {
    GC_REQUIRE(w && packed, GC_EINVAL, "gc_det_heads_pack: null pointer");
    GC_REQUIRE(C > 0 && C % 64 == 0 && n_out > 0 && n_out <= 64, GC_EUNSUPPORTED,
               "gc_det_heads_pack: C must be a multiple of 64 and n_out <= 64 (got %d, %d)", C, n_out);
    return conv_pack((cudaStream_t)stream, w, 1, C, n_out, 32, packed);
}
extern "C" int gc_det_heads(const float *x, int n_frames, int C, int H, int W, int n_out, const void *packed,
                            const float *bias /* [n_out] */, void *workspace, float *out /* [B][n_out][H][W] */,
                            void *stream) {
    GC_REQUIRE(n_frames >= 0 && n_frames <= 65535, GC_EINVAL, "gc_det_heads: bad frame count");
    if (n_frames == 0) return GC_OK;
    GC_REQUIRE(x && packed && bias && workspace && out, GC_EINVAL, "gc_det_heads: null pointer");
    GC_REQUIRE(C > 0 && C % 64 == 0 && n_out > 0 && n_out <= 64, GC_EUNSUPPORTED,
               "gc_det_heads: C must be a multiple of 64 and n_out <= 64 (got %d, %d)", C, n_out);
    GC_REQUIRE(H > 0 && W > 0 && (H * W) % 128 == 0, GC_EUNSUPPORTED,
               "gc_det_heads: H*W must be a multiple of 128 (got %dx%d)", H, W);
    cudaStream_t st = (cudaStream_t)stream;
    ConvLayer L;
    L.xh = (const uint4 *)workspace;
    L.xl = (const uint4 *)((char *)workspace + align_up((size_t)n_frames * H * W * C * 2, 256));
    if (int rc = to_planes(st, x, n_frames, C, H * W, (void *)L.xh, (void *)L.xl)) return rc;
    L.A = n_frames; L.C = L.c_in = C; L.H_in = H; L.W_in = W; L.taps = 1;
    L.w = (const uint4 *)packed; L.n_pad = conv_n_pad(n_out, 32); L.bias = bias; L.n_out = L.out_ch_total = n_out;
    L.epi = 0; L.out = out;
    return conv_layer(st, L);
}
