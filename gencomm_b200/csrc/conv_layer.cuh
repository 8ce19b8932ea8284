// The plane-convolution layer: one descriptor for every tcgen05 convolution over channel-last bf16 value + residual planes
// (backbone, deblocks, shrink header, detection heads, Enhancer GEMMs) and the one function that picks its kernel.
#pragma once
#include <cuda_runtime.h>

namespace gc {

// Output extent of a 3x3 / padding 1 or a 1x1 (stride 1) convolution over n_in pixels.
inline int conv_out_size(int n_in, int stride) { return (n_in - 1) / stride + 1; }

// The kernel N for n_out output channels: weights are packed for this N, and the kernel instantiated for it, so every packer
// and every launcher takes it from here.  n_min is 32 for the detection heads, DoubleConv and the Enhancer, 64 for
// gc_conv_pack / gc_conv_planes.
inline int conv_n_pad(int n_out, int n_min) {
    const int n = n_out < n_min ? n_min : n_out;
    return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : 256;
}
// Bytes of weights conv_pack writes for taps x c_in x n_pad (value + residual bf16).
inline size_t conv_packed_bytes(int taps, int c_in, int n_pad) { return (size_t)taps * c_in * n_pad * 2 * 2; }

struct ConvLayer {
    const uint4 *xh = nullptr, *xl = nullptr;   // input planes [A][H_in][W_in][C]
    int A = 0, C = 0, c_in = 0;                  // agents, plane channels, channels contracted (<= C)
    int H_in = 0, W_in = 0, taps = 9, stride = 1;   // taps 9: 3x3 with padding 1 (stride 1 or 2); 1: 1x1 (stride 1)
    const uint4 *w = nullptr;                    // weights packed by conv_pack for N = n_pad
    int n_pad = 0;
    const float *bias = nullptr;                 // [n_out] (or null: no bias, epilogue 0)
    int n_out = 0;                               // channels stored
    // 0: bias -> NCHW fp32; 2: bias + GELU -> channel-last fp32; 3: bias + ReLU -> NCHW fp32; 5: bias + ReLU -> bf16 planes
    int epi = 0;
    float *out = nullptr;                        // epilogues 0, 2, 3
    uint4 *oh = nullptr, *ol = nullptr;          // epilogue 5
    int out_ch_total = 0, out_ch_off = 0;        // the n_out channels go to out_ch_off .. of out_ch_total
    // up > 1: the output is up-sampled by a pixel shuffle, this launch stores phase (up_dy, up_dx); up_dy = -1: all phases,
    // with the weights of phase ph = dy * up + dx at ph * conv_packed_bytes(taps, c_in, n_pad)
    int up = 1, up_dy = 0, up_dx = 0;

    int Ho() const { return conv_out_size(H_in, stride); }
    int Wo() const { return conv_out_size(W_in, stride); }
};

// Runs the layer on the kernel that fits it (k_conv_rows, k_me_conv with two tiles per CTA, k_conv_tma or k_me_conv).
// The caller has validated the shapes.  Returns GC_OK, or an error code with the message set.
int conv_layer(cudaStream_t st, const ConvLayer &L);

// weights [n_out][c_in][taps] fp32 -> the packed B operand for N = conv_n_pad(n_out, n_min) (k_me_pack, split, 32-channel stages)
int conv_pack(cudaStream_t st, const float *w, int taps, int c_in, int n_out, int n_min, void *packed);
// x [A][C][HW] fp32 -> channel-last bf16 value + residual planes [A][HW][C] (k_me_to_nhwc); C % 64 == 0
int to_planes(cudaStream_t st, const float *x, int A, int C, int HW, void *xh, void *xl);

}  // namespace gc
