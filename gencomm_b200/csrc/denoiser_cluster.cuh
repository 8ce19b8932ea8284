// Interface of the cluster-resident DiffusionUNet kernels (denoiser_cluster.cu) used by denoiser.cu.
#pragma once
#include <cuda_runtime.h>

namespace gc {

constexpr int kCl = 8;               // CTAs per cluster = row bands per agent
constexpr int kClLayers = 26;        // width-8 layers per UNet evaluation (execution order of denoiser.cu)

// Per-layer weight record in device memory (floats), packed by gencomm_b200/gencomm.py::pack_unet_cluster:
//   [0, 1536)     tensor-core layers: B operand [kx 3][cin group 2][k half 2][block j 4][cout 8][4 cin] with block j
//                 = tap row ky = 2 - j (block 3 = 0); down.0.downsample (CUDA cores): w [tap 9][cin 8][cout 8]
//   [1536, 1544)  bias (+ the step's timestep-embedding projection for conv1 of a ResnetBlock)
//   [1544, 1560)  GroupNorm gamma of the (concatenated) input, [1560, 1576) beta
//   [1576, 1704)  nin_shortcut w [cin 16][cout 8], [1704, 1712) nin_shortcut bias
constexpr int kClRecBias = 1536, kClRecGamma = 1544, kClRecBeta = 1560, kClRecNinW = 1576, kClRecNinB = 1704;
constexpr int kClRecFloats = 1712, kClRecBytes = kClRecFloats * 4;

bool unet_cluster_eligible(int C, int H, int W);

// 26 middle layers: h0 [A][64][128][8] (conv_in output, NHWC8) -> out [A][64][128][8] (input of norm_out) +
// stats_out [A][8][8] (GroupNorm partial sums per row band, the format k_conv_out_tc consumes with tiles = 8).
// rec_dev: kClLayers records of the step being evaluated.  layer_dump (gc_unet_trace, else NULL): the outputs of layers
// 0 .. 24 are also written there, in the layout of the trace of include/gencomm_b200.h (tensor 1 + l at its offset).
int unet_middle_cluster(cudaStream_t st, int A, const float *h0, const float *rec_dev, float *out, float *stats_out,
                        float *layer_dump);

}  // namespace gc
