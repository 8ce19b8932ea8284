// Kernel selection for the plane-convolution layers (conv_layer.cuh), and the generic layer entry points over the
// channel-last bf16 planes used by the host mirror of BaseBEVBackbone (models/sub_modules/base_bev_backbone.py:96-124):
// conv3x3 (stride 1/2, pad 1) or 1x1, folded-BN bias, ReLU, written either as the next layer's planes or as NCHW fp32
// (optionally pixel-shuffled = one phase of a ConvTranspose2d whose kernel equals its stride).
#include "common.cuh"
#include <stdlib.h>

#include "conv_layer.cuh"
#include "conv_rows.cuh"
#include "conv_tma.cuh"
#include "implicit_gemm.cuh"

namespace gc {
namespace {

using namespace me;
constexpr int kSc = 32;   // channels per weight stage of the packed layout

// k_me_conv, MT 128-pixel tiles per CTA sharing one weight stage
template <int NOUT, int TAPS, int EPI, int MT>
int launch_me_conv(cudaStream_t st, const ConvLayer &L) {
    constexpr int kSmem = conv_smem_bytes(NOUT, true, kSc, MT);
    static const cudaError_t setup = cudaFuncSetAttribute(k_me_conv<NOUT, false, kSc, TAPS, EPI, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (setup != cudaSuccess) {
        (void)cudaGetLastError();
        set_error("k_me_conv: launch set-up failed (%d)", (int)setup);
        return (int)setup;
    }
    const int Ho = L.Ho(), Wo = L.Wo();
    const dim3 grid(Ho * Wo / kPix / MT, L.A);
    k_me_conv<NOUT, false, kSc, TAPS, EPI, MT><<<grid, conv_block_threads(false), kSmem, st>>>(
        L.xh, L.xl, nullptr, L.w, L.bias, L.C, L.c_in, Ho, Wo, L.n_out, L.out_ch_total, L.out_ch_off, L.out, nullptr, L.H_in, L.W_in,
        L.stride, L.oh, L.ol, L.up, L.up_dy, L.up_dx);
    GC_LAUNCH_CHECK("k_me_conv");
    return GC_OK;
}

template <int NOUT, int TAPS, int EPI>
int launch(cudaStream_t st, const ConvLayer &L) {
    const int Ho = L.Ho(), Wo = L.Wo();
    // 3x3 plane-to-plane layers (the backbone's bulk) can run two 128-pixel tiles per CTA on one weight stage (half the weight
    // traffic from L2).  Measured on the B200: backbone 7.89 ms vs 7.66 ms with one tile -- no gain (DESIGN.md 5e), opt-in for A/B.
    static const bool two = getenv("GC_CONV_MT2") != nullptr;
    if constexpr (TAPS == 9 && EPI == 5) {
        const int tiles = Ho * Wo / kPix;   // per agent
        if (two && tiles % 2 == 0 && (long long)tiles * L.A >= 2 * 148) return launch_me_conv<NOUT, TAPS, EPI, 2>(st, L);
    }
    if (ct::conv_tma_eligible(L.stride, L.C, L.c_in, Ho, Wo, L.up))
        return ct::launch_conv_tma<NOUT, TAPS, EPI>(st, L.A, L.xh, L.xl, L.w, L.bias, L.C, L.c_in, Ho, Wo, L.H_in, L.W_in, L.stride,
                                                    L.n_out, L.out_ch_total, L.out_ch_off, L.out, L.oh, L.ol, L.up, L.up_dy, L.up_dx);
    return launch_me_conv<NOUT, TAPS, EPI, 1>(st, L);
}

// Every (N, taps, epilogue) a caller builds, and nothing else: the heads' 1x1 GEMM; the Enhancer's partial 3x3, linear1 + GELU
// and linear2; the backbone, deblock and DoubleConv layers.
struct Kernel {
    int n, taps, epi;
    int (*run)(cudaStream_t, const ConvLayer &);
};
constexpr Kernel kKernels[] = {
    {32, 1, 0, launch<32, 1, 0>},    {64, 1, 0, launch<64, 1, 0>},                                        // detection heads
    {32, 9, 0, launch<32, 9, 0>},    {64, 9, 0, launch<64, 9, 0>},                                        // Enhancer
    {256, 1, 2, launch<256, 1, 2>},  {128, 1, 0, launch<128, 1, 0>},
    {64, 1, 3, launch<64, 1, 3>},    {64, 1, 5, launch<64, 1, 5>},    {64, 9, 3, launch<64, 9, 3>},       // layers
    {64, 9, 5, launch<64, 9, 5>},    {128, 1, 3, launch<128, 1, 3>},  {128, 1, 5, launch<128, 1, 5>},
    {128, 9, 3, launch<128, 9, 3>},  {128, 9, 5, launch<128, 9, 5>},  {256, 1, 3, launch<256, 1, 3>},
    {256, 1, 5, launch<256, 1, 5>},  {256, 9, 3, launch<256, 9, 3>},  {256, 9, 5, launch<256, 9, 5>},
};

}  // namespace

int conv_layer(cudaStream_t st, const ConvLayer &L) {
    if (L.up_dy == -1 && !(ct::conv_tma_eligible(L.stride, L.C, L.c_in, L.H_in, L.W_in, L.up) && L.n_out % 16 == 0 && L.n_out >= 64)) {
        // all phases requested but the fused launch does not apply: one launch per phase
        ConvLayer p = L;
        for (int ph = 0; ph < L.up * L.up; ++ph) {
            p.up_dy = ph / L.up;
            p.up_dx = ph % L.up;
            p.w = (const uint4 *)((const char *)L.w + ph * conv_packed_bytes(L.taps, L.c_in, L.n_pad));
            if (int rc = conv_layer(st, p)) return rc;
        }
        return GC_OK;
    }
    // wide stride-1 layers: the row-staged kernel (conv_rows.cu) reads every input row once per channel chunk instead of nine times
    if (conv_rows_eligible(L)) return conv_rows(st, L);
    for (const Kernel &k : kKernels)
        if (k.n == L.n_pad && k.taps == L.taps && k.epi == L.epi) return k.run(st, L);
    set_error("conv_layer: no kernel for N = %d, taps = %d, epilogue %d", L.n_pad, L.taps, L.epi);
    return GC_EUNSUPPORTED;
}

int conv_pack(cudaStream_t st, const float *w, int taps, int c_in, int n_out, int n_min, void *packed) {
    const int n = conv_n_pad(n_out, n_min), t = taps * (c_in / 8) * n;
    k_me_pack<<<(t + 255) / 256, 256, 0, st>>>(w, n_out, n, c_in, kSc, taps, 1, (uint4 *)packed);
    GC_LAUNCH_CHECK("k_me_pack");
    return GC_OK;
}

int to_planes(cudaStream_t st, const float *x, int A, int C, int HW, void *xh, void *xl) {
    k_me_to_nhwc<<<dim3((HW + 63) / 64, C / 64, A), 256, 0, st>>>(x, C, HW, (uint4 *)xh, (uint4 *)xl);
    GC_LAUNCH_CHECK("k_me_to_nhwc");
    return GC_OK;
}

}  // namespace gc

using namespace gc;

extern "C" size_t gc_conv_packed_bytes(int taps, int c_in, int n_out) {
    return (taps == 1 || taps == 9) && c_in > 0 && n_out > 0 ? conv_packed_bytes(taps, c_in, conv_n_pad(n_out, 64)) : 0;
}
extern "C" int gc_conv_pack(const float *w /* [n_out][c_in][taps] */, int taps, int c_in, int n_out, void *packed, void *stream) {
    GC_REQUIRE(w && packed, GC_EINVAL, "gc_conv_pack: null pointer");
    GC_REQUIRE((taps == 1 || taps == 9) && c_in > 0 && c_in % 32 == 0 && n_out > 0 && n_out <= 256, GC_EUNSUPPORTED,
               "gc_conv_pack: taps in {1,9}, c_in %% 32 == 0, n_out <= 256 (got %d, %d, %d)", taps, c_in, n_out);
    return conv_pack((cudaStream_t)stream, w, taps, c_in, n_out, 64, packed);
}
extern "C" int gc_to_planes(const float *x, int total_agents, int C, int HW, void *xh, void *xl, void *stream) {
    GC_REQUIRE(total_agents >= 0 && C > 0 && C % 64 == 0 && HW > 0, GC_EUNSUPPORTED, "gc_to_planes: C must be a multiple of 64");
    if (total_agents == 0) return GC_OK;
    GC_REQUIRE(x && xh && xl, GC_EINVAL, "gc_to_planes: null pointer");
    return to_planes((cudaStream_t)stream, x, total_agents, C, HW, xh, xl);
}
extern "C" int gc_conv_planes(const void *xh, const void *xl, int total_agents, int c_in, int H_in, int W_in, int stride, int taps,
                              int n_out, const void *packed, const float *bias, void *oh, void *ol, float *out_nchw,
                              int out_ch_total, int out_ch_off, int up, int up_dy, int up_dx, void *stream) {
    GC_REQUIRE(total_agents >= 0 && total_agents <= 65535, GC_EINVAL, "gc_conv_planes: bad agent count");
    if (total_agents == 0) return GC_OK;
    GC_REQUIRE(xh && xl && packed && ((oh && ol) || out_nchw), GC_EINVAL, "gc_conv_planes: null pointer");
    GC_REQUIRE((taps == 1 || taps == 9) && c_in > 0 && c_in % 32 == 0 && n_out >= 8 && n_out <= 256 && n_out % 8 == 0,
               GC_EUNSUPPORTED, "gc_conv_planes: taps in {1,9}, c_in %% 32 == 0, n_out %% 8 == 0, n_out <= 256");
    GC_REQUIRE((stride == 1 || stride == 2) && (taps == 9 || stride == 1) && up >= 1 &&
                   ((up_dy >= 0 && up_dy < up && up_dx >= 0 && up_dx < up) || (up_dy == -1 && taps == 1)),
               GC_EUNSUPPORTED, "gc_conv_planes: bad stride / up-sampling phase");
    ConvLayer L;
    L.xh = (const uint4 *)xh; L.xl = (const uint4 *)xl; L.A = total_agents; L.C = L.c_in = c_in; L.H_in = H_in; L.W_in = W_in;
    L.taps = taps; L.stride = stride; L.w = (const uint4 *)packed; L.n_pad = conv_n_pad(n_out, 64); L.bias = bias; L.n_out = n_out;
    if (oh) { L.epi = 5; L.oh = (uint4 *)oh; L.ol = (uint4 *)ol; }
    else { L.epi = 3; L.out = out_nchw; }
    L.out_ch_total = out_ch_total; L.out_ch_off = out_ch_off; L.up = up; L.up_dy = up_dy; L.up_dx = up_dx;
    const int Ho = L.Ho(), Wo = L.Wo();
    GC_REQUIRE(Ho > 0 && Wo > 0 && (Ho * Wo) % me::kPix == 0, GC_EUNSUPPORTED,
               "gc_conv_planes: output H*W must be a multiple of 128 (got %dx%d)", Ho, Wo);
    GC_REQUIRE(out_ch_total >= out_ch_off + n_out && out_ch_total % 8 == 0 && out_ch_off % 8 == 0, GC_EINVAL,
               "gc_conv_planes: bad output channel window");
    GC_REQUIRE(!oh || n_out % 16 == 0, GC_EUNSUPPORTED, "gc_conv_planes: plane outputs need n_out %% 16 == 0");
    return conv_layer((cudaStream_t)stream, L);
}
