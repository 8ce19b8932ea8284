// Row-staged 3x3 stride-1 convolution on tcgen05 (conv_rows.cu), chosen by conv_layer for wide maps when GC_CONV_ROWS=1.
#pragma once
#include <cuda_runtime.h>

#include "conv_layer.cuh"

namespace gc {

// GC_CONV_ROWS=1 (read per call; k_conv_tma is the default for these layers) and a 3x3 stride-1 layer without up-sampling
// with a ReLU epilogue (3 or 5) over every channel of the planes (c_in == C, c_in % 32 == 0), Wo % 128 == 0 and
// n_out in {64 (Ho % 4 == 0), 128 (Ho % 2 == 0)}
bool conv_rows_eligible(const ConvLayer &L);

// ReLU(conv3x3(planes) + bias): epilogue 5 writes channel-last bf16 value + residual planes (oh, ol), epilogue 3 fp32 NCHW (out),
// at channel offset out_ch_off of out_ch_total channels.  All n_out = N channels are stored.
int conv_rows(cudaStream_t st, const ConvLayer &L);

}  // namespace gc
