/*
 * gencomm_b200 -- C ABI of the B200-native (sm_100a) GenComm per-frame hot path.
 *
 * The reference (jeffreychou777/GenComm, an OpenCOOD fork) is pure Python/PyTorch and has no FFI
 * for this path (SURVEY.md section 8b); its "plugin API" is the set of Python operators listed
 * below.  Each entry point here replaces the body of one of them and is what a ctypes binding in
 * the reference would call (see INTEGRATION.md).  Conventions:
 *
 *   - plain C: pointers + sizes, no torch types.  Unless a parameter is marked [host], every
 *     pointer is a DEVICE pointer to contiguous memory; nothing is allocated inside;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), never synchronises,
 *     and is re-entrant (all state lives in caller-provided buffers);
 *   - return value: 0 on success, a negative GC_E* code for an argument error (nothing launched),
 *     or a positive cudaError_t from the launch.  gc_last_error() returns a static description of
 *     the most recent failure on the calling thread.
 *
 * Paths are relative to /root/reference/opencood.
 */
#ifndef GENCOMM_B200_H_
#define GENCOMM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GC_OK 0
#define GC_EINVAL (-1)      /* bad shape / size / null pointer */
#define GC_EUNSUPPORTED (-2) /* configuration outside what the kernels implement */

#define GC_MAX_POINTS_PER_PILLAR 32 /* max_points_per_voxel of every shipped yaml */
#define GC_PFN_OUT 64               /* pillar_vfe.num_filters = [64] */
#define GC_MAX_AGENTS_PER_FRAME 8   /* max_cav is 5 in every shipped yaml; microbench goes to 8 */

#define GC_FUSE_WARP_ONLY 0 /* warp_affine_simple / warp_feature: no reduction */
#define GC_FUSE_MAX 1       /* MaxFusion */
#define GC_FUSE_ATT 2       /* AttFusion (ego row of the per-pixel attention) */

/* Denoiser arithmetic (bit mask).  0 = every layer in fp32 on CUDA cores (parity path, <= 1e-4 of the
 * fp32 reference).  The TC bits run the GEMM-shaped layers as bf16 tcgen05 implicit GEMMs with fp32
 * accumulation in TMEM where the shape is eligible (W % 128 == 0, C % 64 == 0), fp32 otherwise. */
#define GC_PREC_F32 0
#define GC_PREC_TC_CONV_IN 1   /* conv_in  ((C+2) -> 8, K = 9(C+2)) */
#define GC_PREC_TC_CONV_OUT 2  /* norm_out + swish + conv_out (8 -> C, K = 72) */
#define GC_PREC_BF16_TC 3      /* both */
#define GC_PREC_TC_MATERIALIZE 4 /* validation: explicit im2col operand instead of overlapping windows */
#define GC_PREC_TC_MIDDLE 8    /* full-resolution width-8 middle layers as tf32 tcgen05 implicit GEMMs */
#define GC_PREC_TC_ALL 11      /* conv_in/conv_out bf16 + middle layers tf32 */
#define GC_PREC_CLUSTER 16     /* with GC_PREC_BF16_TC, H x W = 64 x 128 and w_cluster_dev != NULL: the 26 width-8 layers of
                                  an evaluation run in ONE launch, one thread-block cluster of 8 CTAs per agent, activations
                                  resident in (distributed) shared memory, tf32 tcgen05 (csrc/denoiser_cluster.cu) */
#define GC_PREC_CLUSTER_ALL 27 /* GC_PREC_TC_ALL | GC_PREC_CLUSTER: the module default; ineligible shapes fall back to TC_ALL */

int gc_version(void);
const char *gc_last_error(void);

/* Voxelizer geometry: data_utils/pre_processor/sp_voxel_preprocessor.py:32-60. */
typedef struct gcVoxelGeom {
    float range_min[3]; /* cav_lidar_range[0:3]  x,y,z */
    float voxel[3];     /* args.voxel_size       x,y,z */
    int32_t grid[3];    /* round((max-min)/voxel) = nx,ny,nz (:41-43) */
    int32_t max_points; /* max_points_per_voxel (must be 32) */
    int32_t max_voxels; /* max_voxel_test / max_voxel_train */
} gcVoxelGeom;

/* ---------------------------------------------------------------------------------------------
 * (a1) SpVoxelPreprocessor.preprocess -> spconv Point2VoxelCPU3d.point_to_voxel
 *      (sp_voxel_preprocessor.py:62-85), for all agents of a batch at once.
 *
 * Device workspace layout is private; size it with gc_voxelize_workspace_bytes().
 *   points        [total_points][4] f32, agents concatenated
 *   point_offsets [n_agents+1] i32, exclusive prefix of points per agent (device)
 *   n_pillars     [n_agents] i32 out: M_a = min(#occupied cells in first-come order, max_voxels)
 * After the call the workspace holds, per agent, the cell->pillar map and the per-pillar list of
 * the first 32 point indices in input order; gc_voxel_gather / gc_pillar_canvas consume it.
 * ------------------------------------------------------------------------------------------- */
size_t gc_voxelize_workspace_bytes(const gcVoxelGeom *geom /*[host]*/, int n_agents, int total_points);

int gc_voxelize(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                int max_agent_points /* upper bound on any one agent's point count; <=0: total_points */,
                const gcVoxelGeom *geom /*[host]*/, void *workspace, int32_t *n_pillars, void *stream);

/* Materialise the reference-shaped voxel tensors (the dict `preprocess` returns, then
 * collate_batch_list :109-142) from the workspace:
 *   pillar_offsets [n_agents+1] i32: exclusive prefix of n_pillars (device; caller computes it),
 *   total_pillars = pillar_offsets[n_agents] (host copy; sizes the launch and the outputs)
 *   voxels [sum M][32][4] f32 zero padded, coords [sum M][4] i32 (agent,z,y,x), num_points [sum M] i32
 */
int gc_voxel_gather(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                    const gcVoxelGeom *geom /*[host]*/, const void *workspace,
                    const int32_t *pillar_offsets, int total_pillars, float *voxels, int32_t *coords,
                    int32_t *num_points, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a3) PillarVFE.forward + PFNLayer.forward (models/sub_modules/pillar_vfe.py:105-155, :31-53)
 *      for use_norm=True, use_absolute_xyz=True, with_distance=False, num_filters=[64], eval BN.
 *
 *   pfn  [64][16] f32 per output channel k, packed by the host (gencomm_b200/ops.py::pack_pfn) with the
 *        eval BatchNorm (scale, shift) folded in:
 *        [0..2] A = ((W[k][j]+W[k][4+j])+W[k][7+j])*scale, [3] W[k][3]*scale, [4..6] W[k][0..2]*scale,
 *        [7..9] (-W[k][4..6])*scale, [10] shift, [11] max(shift,0), [12..15] 0
 *   centre_offset[3] = voxel/2 + range_min (pillar_vfe.py:87-89), voxel[3]  -- in geom/arguments
 *   voxels [M][32][4], num_points [M], coords [M][4] (b,z,y,x)  ->  pillar_features [M][64]
 * ------------------------------------------------------------------------------------------- */
int gc_pillar_vfe(const float *voxels, const int32_t *num_points, const int32_t *coords, int n_pillars,
                  const float *pfn, const float voxel[3] /*[host]*/, const float centre_offset[3] /*[host]*/,
                  float *pillar_features, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a4) PointPillarScatter.forward (models/sub_modules/point_pillar_scatter.py:19-76).
 *      canvas[b][c][y][x] = pillar_features[m][c] for coords[m] = (b,z,y,x), zero elsewhere;
 *      idx = z + y*nx + x (:58), nz == 1 (:17).  Written canvas-stationary: every canvas byte is
 *      stored exactly once (no separate memset), through a dense cell->pillar map.
 *   cell_map [n_batch][ny*nx] i32 scratch (device), fully rewritten by the call
 *   canvas   [n_batch][C][ny][nx] f32
 * ------------------------------------------------------------------------------------------- */
int gc_scatter_canvas(const float *pillar_features, const int32_t *coords, int n_pillars, int C,
                      int nx, int ny, int n_batch, int32_t *cell_map, float *canvas, void *stream);

/* Fused (a1 workspace) -> (a3) -> (a4): voxel workspace straight to the BEV canvas, never
 * materialising voxels[M,32,4] or pillar_features[M,64].  canvas [n_agents][64][ny][nx]. */
int gc_pillar_canvas(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                     const gcVoxelGeom *geom /*[host]*/, const void *workspace, const float *pfn,
                     const float centre_offset[3] /*[host]*/, float *canvas, void *stream);
/* The same canvas as channel-last bf16 value + residual planes xh, xl [n_agents][ny*nx][64] (the operand layout of
 * gc_conv_planes): what PointPillar hands to this package's BaseBEVBackbone -- no fp32 canvas, no gc_to_planes pass. */
int gc_pillar_canvas_planes(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                            const gcVoxelGeom *geom /*[host]*/, const void *workspace, const float *pfn,
                            const float centre_offset[3] /*[host]*/, void *xh, void *xl, void *stream);
/* Sparse maintenance of the same planes (a persistent buffer of the caller that is all-zero between frames): only the
 * occupied cells are written -- 16 % of a 512 x 256 grid at 100 k points -- and gc_planes_clear_occupied, called with the
 * same workspace once the planes have been consumed (before the next gc_voxelize on that workspace), zeroes exactly those
 * cells again.  Same plane contents as gc_pillar_canvas_planes, bit for bit. */
int gc_pillar_canvas_planes_sparse(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                                   const gcVoxelGeom *geom /*[host]*/, const void *workspace, const float *pfn,
                                   const float centre_offset[3] /*[host]*/, void *xh, void *xl, void *stream);
int gc_planes_clear_occupied(const gcVoxelGeom *geom /*[host]*/, int n_agents, int total_points, const void *workspace,
                             void *xh, void *xl, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a6)+(a7)+(a8)/(a9) regroup + warp_affine_simple + MaxFusion / AttFusion
 *      (models/fuse_modules/fusion_in_one.py:48-51, :91-124, :131-151;
 *       models/sub_modules/torch_transformation_utils.py:323-332).
 *
 *   feat          [sum N][C][H][W] f32 (NCHW), agents of frame b at agent_offsets[b]..[b+1]
 *   agent_offsets [n_frames+1] i32 exclusive prefix of record_len (device)
 *   theta         [n_frames][L][L][2][3] f64 = normalize_pairwise_tfm output (float64 on the real
 *                 path, transformation_utils.py:40); only row [b][0][j] (ego <- agent j) is read
 *   mode          GC_FUSE_MAX / GC_FUSE_ATT: out [n_frames][C][H][W]
 *                 GC_FUSE_WARP_ONLY:        out [sum N][C][H][W] (total_agents must be given)
 *   affine_grid is evaluated in float64 and only the grid is rounded to float32, exactly like
 *   F.affine_grid(theta_f64).to(src); sampling follows ATen's grid_sampler_2d (bilinear, zeros
 *   padding, align_corners=False).
 *   max_agents_per_frame is a HOST-side promise used to pick a kernel specialisation (no device -> host sync to read
 *   record_len): it must be >= every record_len entry.  A smaller value is a contract violation -- the tiled kernels then
 *   fuse only the first max_agents_per_frame agents of a frame and ignore the rest; pass <= 0 when unknown (L is used).
 * ------------------------------------------------------------------------------------------- */
int gc_warp_fuse(const float *feat, const int32_t *agent_offsets, int n_frames, int total_agents,
                 int max_agents_per_frame /* host-side upper bound on any record_len entry; <= 0: unknown (L is used) */,
                 const double *theta, int L, int C, int H, int W, int mode, float *out, void *stream);

/* (a5) normalize_pairwise_tfm (utils/transformation_utils.py:68-92):
 *   pairwise [n][4][4] f64 -> theta [n][2][3] f64, n = B*L*L matrices. */
int gc_normalize_pairwise_tfm(const double *pairwise, int n, double H, double W, double discrete_ratio,
                              double downsample_rate, double *theta, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a10)+(a11) GenComm.forward (eval branch) + DiffusionUNet.forward
 *      (models/gencomm_modules/cond_diff.py:331-383, :262-329; models/gencomm_modules/unet.py:307-344)
 *      for ch=8, ch_mult=[1,1], num_res_blocks=2, resamp_with_conv=True (no attention block is ever
 *      instantiated by the shipped configs).  x0-parameterised ancestral sampling, T steps:
 *        x_T = sqrt(ac_T) * ego(frame of agent) + sqrt(1-ac_T) * noise0            (:333-337, :372)
 *        t = T-1..1: x0 = UNet(cat[cond, x_t], t); x_{t-1} = c1_t x0 + c2_t x_t + sigma_t noise_t  (:272-279, :310)
 *        t = 0:      pred = UNet(cat[cond, x_0'], 0)                                  (:292-294, :313)
 *      Noise is an INPUT (the reference draws it with torch.randn; bit-parity with that stream is
 *      not a goal, SURVEY.md App. A.6): noise0 [sumN][C][H][W]; step_noise [T-1][sumN][C][H][W] for
 *      t = T-1, ..., 1.
 *
 *   feat  [sumN][C][H][W] f32, cond [sumN][2][H][W] f32 (the 2-channel messages), pred like feat
 *   agent_offsets [n_frames+1] i32 (device), exclusive prefix of record_len
 *   w_host [host]  gc_gencomm_host_weight_floats(T) floats, packed by gencomm_b200/gencomm.py::pack_unet:
 *          T x 26 conv records (execution order; [tap][cin16][cout8] weights, bias incl. the
 *          timestep-embedding projection of that step, GroupNorm affine, nin_shortcut), then
 *          conv_in.bias[8], norm_out.weight[8], norm_out.bias[8]
 *   w_dev  [device] gc_gencomm_device_weight_floats(C) floats: conv_in [C+2][9][8], conv_out [C][9][8], conv_out.bias [C]
 *   w_cluster_dev [device, may be NULL] gc_gencomm_cluster_weight_floats(T) floats: the same T x 26 conv records in the
 *          layout the cluster kernel bulk-copies into shared memory (csrc/denoiser_cluster.cuh), packed by
 *          gencomm_b200/gencomm.py::pack_unet_cluster; NULL disables GC_PREC_CLUSTER
 *   schedule_host [host] [T][5]: sqrt_alphas_cumprod, sqrt_one_minus_alphas_cumprod,
 *          posterior_mean_coef1, posterior_mean_coef2, exp(0.5*posterior_log_variance_clipped)
 *   workspace: gc_gencomm_workspace_bytes(sumN, C, H, W) bytes (device)
 * ------------------------------------------------------------------------------------------- */
size_t gc_gencomm_host_weight_floats(int T);
size_t gc_gencomm_device_weight_floats(int C);
size_t gc_gencomm_cluster_weight_floats(int T);
size_t gc_gencomm_workspace_bytes(int total_agents, int C, int H, int W);

int gc_gencomm_sample(const float *feat, const float *cond, const int32_t *agent_offsets, int n_frames,
                      int total_agents, const float *noise0, const float *step_noise,
                      const float *w_host /*[host]*/, const float *w_dev, const float *w_cluster_dev /* or NULL */,
                      const float *schedule_host /*[host]*/, int C, int H, int W, int T, int precision /* GC_PREC_* */,
                      void *workspace, float *pred, void *stream);

/* One denoiser evaluation pred = UNet(cat[cond, x], t_index) for all agents (diagnostics / tests). */
int gc_unet_forward(const float *cond, const float *x, int total_agents, int t_index,
                    const float *w_host /*[host]*/, const float *w_dev, const float *w_cluster_dev /* or NULL */, int C,
                    int H, int W, int T, int precision /* GC_PREC_* */, void *workspace, float *pred, void *stream);

/* gc_unet_forward that also writes the activations of the evaluation to trace [device], for per-layer tests:
 * gc_unet_trace_floats(total_agents, H, W) floats holding 27 NHWC8 fp32 tensors back to back,
 *   tensor 0      hs0 = conv_in output                      [A][H][W][8]
 *   tensor 1 + l  output of middle layer l (l = 0 .. 25, the execution order of the 26 width-8 convolutions:
 *                 down.0.block.0 conv1, conv2, down.0.block.1 conv1, conv2, down.0.downsample, down.1.block.0 conv1, ...,
 *                 up.0.block.2 conv2), [A][H/2][W/2][8] for l = 4 .. 18 (tensors 5 .. 19), [A][H][W][8] otherwise.
 * pred is bit-identical to gc_unet_forward's for every precision. */
size_t gc_unet_trace_floats(int total_agents, int H, int W);
int gc_unet_trace(const float *cond, const float *x, int total_agents, int t_index,
                  const float *w_host /*[host]*/, const float *w_dev, const float *w_cluster_dev /* or NULL */, int C,
                  int H, int W, int T, int precision /* GC_PREC_* */, void *workspace, float *pred, float *trace,
                  void *stream);

/* ---------------------------------------------------------------------------------------------
 * (8f rank 1) MessageExtractorv2.forward (models/gencomm_modules/message_extractor_v2.py:114-120)
 *   = BEVDeformableExtractor.forward (:96-112): offset1 (3x3 conv C->18) -> torchvision DeformConv2d (3x3, C->64,
 *   padding 1) -> average pool + squeeze/excite -> 1x1 (64->64) + ReLU -> 1x1 (64->2).
 *   x        [sumN][C][H][W] f32, C % 64 == 0, H*W % 128 == 0
 *   packed   gc_me_packed_bytes(C) bytes written by gc_me_pack_weights from offset1.weight [18][C][3][3] and
 *            dcn1.weight [64][C][3][3] (device, f32): the bf16 B operands of the two tcgen05 implicit GEMMs
 *   params   gc_me_param_floats() floats (device): offset1.bias[18] (padded to 32), dcn1.bias[64],
 *            attn.1.weight[32][64], attn.1.bias[32], attn.3.weight[64][32], attn.3.bias[64],
 *            fuse.0.weight[64][64], fuse.0.bias[64], fuse.2.weight[2][64], fuse.2.bias[2] (padded to 8)
 *   workspace gc_me_workspace_bytes(sumN, C, H, W) bytes (device)
 *   message  [sumN][2][H][W] f32
 *   Arithmetic: the two 3x3 layers use bf16 operands with fp32 accumulation; the rest is fp32.
 * ------------------------------------------------------------------------------------------- */
size_t gc_me_param_floats(void);
size_t gc_me_packed_bytes(int C);
size_t gc_me_workspace_bytes(int total_agents, int C, int H, int W);
int gc_me_pack_weights(const float *w_offset, const float *w_dcn, int C, void *packed, void *stream);
int gc_message_extractor(const float *x, int total_agents, int C, int H, int W, const void *packed,
                         const float *params, void *workspace, float *message, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (8f rank 1) Enhancer.forward (models/gencomm_modules/enhancer.py:335-383): Enhancer_block block_1 (:316-333, attention
 *   disabled in the reference) = x + LN1(x), + FRFN(LN2(.)) (:205-250), then SplitAttn (:286-314).  Per agent; all agents
 *   of all frames in one call.
 *   x, out   [sumN][C][H][W] f32, C in {128, 256}, H*W % 128 == 0
 *   packed   gc_enhancer_packed_bytes(C) bytes written by gc_enhancer_pack_weights from block_1.mlp.partial_conv3.weight
 *            [C/4][C/4][3][3], block_1.mlp.linear1.0.weight [4C][C], block_1.mlp.linear2.0.weight [C][2C] (device, f32)
 *   params   gc_enhancer_param_floats(C) floats (device), in this order: block_1.norm1.weight/bias [C], norm2.weight/bias
 *            [C], mlp.linear1.0.bias [4C], mlp.dwconv.0.weight [2C][9], mlp.dwconv.0.bias [2C], mlp.linear2.0.bias [C],
 *            split_attn.fc1.weight [C][C], split_attn.bn1.weight/bias [C], split_attn.fc2.weight [C][C]
 *   workspace gc_enhancer_workspace_bytes(sumN, C, H, W) bytes (device)
 *   Arithmetic: the three dense layers are tcgen05 GEMMs in bf16x3 (fp32-grade); everything else fp32.
 * ------------------------------------------------------------------------------------------- */
size_t gc_enhancer_param_floats(int C);
size_t gc_enhancer_packed_bytes(int C);
size_t gc_enhancer_workspace_bytes(int total_agents, int C, int H, int W);
int gc_enhancer_pack_weights(const float *w_pconv, const float *w_lin1, const float *w_lin2, int C, void *packed,
                             void *stream);
int gc_enhancer(const float *x, int total_agents, int C, int H, int W, const void *packed, const float *params,
                void *workspace, float *out, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (8f rank 2, first slice) DoubleConv / DownsampleConv (models/sub_modules/downsample_conv.py:7-50):
 *   out = ReLU(conv3x3(ReLU(conv3x3_stride_s(x) + b1)) + b2), padding 1, stride s in {1, 2}
 *   x [sumN][c_in][H][W] f32 -> out [sumN][c_out][Ho][Wo], Ho = (H - 1) / s + 1; c_in, c_out % 64 == 0, c_out <= 256,
 *   Ho*Wo % 128 == 0.  packed: gc_double_conv_pack(double_conv.0.weight [c_out][c_in][3][3], double_conv.2.weight
 *   [c_out][c_out][3][3]); bias [2][c_out] (device).  tcgen05 implicit GEMMs in bf16x3 (fp32-grade).
 * Shared detection heads (models/heter_model_baseline.py:130-135): cls_head, reg_head, dir_head = three 1x1 Conv2d on
 *   the fused feature, evaluated as one GEMM: w [n_out][C] = their weights concatenated, n_out <= 64, bias [n_out];
 *   x [B][C][H][W] -> out [B][n_out][H][W].
 * ------------------------------------------------------------------------------------------- */
size_t gc_double_conv_packed_bytes(int c_in, int c_out);
size_t gc_double_conv_workspace_bytes(int total_agents, int c_in, int H, int W, int stride, int c_out);
int gc_double_conv_pack(const float *w1, const float *w2, int c_in, int c_out, void *packed, void *stream);
int gc_double_conv(const float *x, int total_agents, int c_in, int H, int W, int stride, int c_out, const void *packed,
                   const float *bias, void *workspace, float *out, void *stream);
/* the same layer over channel-last planes (gc_to_planes / gc_conv_planes outputs, [A][H*W][c_in]): what the shrink header
 * runs when the backbone hands its deblock outputs over as planes instead of NCHW fp32 (no layout conversion in between) */
size_t gc_double_conv_planes_workspace_bytes(int total_agents, int H, int W, int stride, int c_out);
int gc_double_conv_planes(const void *xh, const void *xl, int total_agents, int c_in, int H, int W, int stride, int c_out,
                          const void *packed, const float *bias, void *workspace, float *out, void *stream);
size_t gc_det_heads_packed_bytes(int C, int n_out);
size_t gc_det_heads_workspace_bytes(int n_frames, int C, int H, int W);
int gc_det_heads_pack(const float *w, int C, int n_out, void *packed, void *stream);
int gc_det_heads(const float *x, int n_frames, int C, int H, int W, int n_out, const void *packed, const float *bias,
                 void *workspace, float *out, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (8f rank 2) Layer primitives behind BaseBEVBackbone.forward (models/sub_modules/base_bev_backbone.py:96-124):
 *   gc_to_planes   x [A][C][HW] f32 -> channel-last bf16 value + residual planes (2 x A*HW*C*2 bytes), C % 64 == 0
 *   gc_conv_pack   w [n_out][c_in][taps] f32 (taps = 9: 3x3, row-major ky,kx; taps = 1: 1x1; BatchNorm already folded)
 *   gc_conv_planes ReLU(conv(planes) + bias): 3x3 with padding 1 and stride 1|2, or 1x1; written as the next layer's
 *                  planes (oh, ol: [A][Ho*up*Wo*up][out_ch_total] bf16, channels out_ch_off..) or as NCHW fp32 out_nchw
 *                  [A][out_ch_total][Ho*up][Wo*up], in both cases at pixel (y*up + up_dy, x*up + up_dx) -- one phase of
 *                  a ConvTranspose2d whose kernel equals its stride `up` (up = 1: an ordinary store).  up_dy = -1 (1x1 only):
 *                  ALL up * up phases in one call, `packed` = the phases' gc_conv_pack outputs back to back in the order
 *                  dy * up + dx (gc_conv_packed_bytes(1, c_in, n_out) bytes each).
 *   Output H*W must be a multiple of 128; n_out <= 256.  bf16x3 tcgen05 GEMMs (fp32-grade).
 * ------------------------------------------------------------------------------------------- */
size_t gc_conv_packed_bytes(int taps, int c_in, int n_out);
int gc_conv_pack(const float *w, int taps, int c_in, int n_out, void *packed, void *stream);
int gc_to_planes(const float *x, int total_agents, int C, int HW, void *xh, void *xl, void *stream);
int gc_conv_planes(const void *xh, const void *xl, int total_agents, int c_in, int H_in, int W_in, int stride, int taps,
                   int n_out, const void *packed, const float *bias, void *oh, void *ol, float *out_nchw,
                   int out_ch_total, int out_ch_off, int up, int up_dy, int up_dx, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (8f rank 3) VoxelPostprocessor.post_process (data_utils/post_processor/voxel_postprocessor.py:1084-1244) for the
 * ego output of an intermediate-fusion model, batched over frames: sigmoid + score threshold, delta_to_boxes3d
 * (:1351-1396), direction-classifier fix (:1156-1172), boxes_to_corners_3d + project_box3d (utils/box_utils.py:152-203,
 * :278-316), remove_large_pred_bbx / remove_bbx_abnormal_z (:1062-1112), nms_rotated (:915-960; polygon IoU of
 * utils/common_utils.py:230-252 as float64 convex clipping), mask_boxes_outside_range_numpy (:384-421).
 *   cls [B][A][H][W], reg [B][7A][H][W], dir [B][A*num_bins][H][W] (or NULL), anchors [H][W][A][7] f32
 *   (generate_anchor_box, :68-121), tfm [B][4][4] f32 row-major (cav -> ego, NULL = identity).
 *   -> boxes [B][top][8][3] f32, scores [B][top] f32 in NMS pick order (highest score first), counts [B] i32.
 *   Score ties are broken larger-anchor-index first.  No host synchronisation.
 * ------------------------------------------------------------------------------------------- */
typedef struct gcPostParams {
    float score_threshold; /* target_args.score_threshold */
    float nms_thresh;      /* nms_thresh */
    float dir_offset;      /* dir_args.dir_offset */
    int32_t num_bins;      /* dir_args.num_bins */
    int32_t order_hwl;     /* order == 'hwl' (PointPillars) : 1, 'lhw' : 0 */
    int32_t top;           /* candidates entering the NMS (the reference uses 1000; <= 1024) */
    double gt_range[6];    /* gt_range: xmin, ymin, zmin, xmax, ymax, zmax */
} gcPostParams;
size_t gc_postprocess_workspace_bytes(int n_frames, int n_anchors /* A*H*W */);
int gc_postprocess(const float *cls, const float *reg, const float *dir, const float *anchors, const float *tfm, int n_frames,
                   int A, int H, int W, const gcPostParams *params, void *workspace, float *boxes, float *scores, int *counts,
                   void *stream);

/* ---------------------------------------------------------------------------------------------
 * (8f rank 4) LiftSplatShoot.voxel_pooling (models/heter_encoders.py:161-217; cumsum trick utils/camera_utils.py:209-217):
 * geom [Nprime][3] f32 (ego-frame xyz of the B*N*D*H*W frustum points, batch-major), x [Nprime][C] f32, dx / bx [3] f32 and
 * nx [3] i32 from gen_dx_bx (camera_utils.py:129-134) -> out [B][nz*C][ny][nx] f32 (zeroed here; the reference's
 * `torch.cat(final.unbind(dim=2), 1)` layout).  Voxel indices are the reference's (fp32 sub / div, truncation); sums are
 * fp32 reductions in L2 (order differs from the reference's cumsum differences: tolerance-bounded).  With a workspace
 * (channel-last accumulation grid) and C % 4 == 0 the reductions are 128-bit (red.global.add.v4.f32) + one transpose.
 * ------------------------------------------------------------------------------------------- */
size_t gc_lss_pool_workspace_bytes(int n_batch, int C, const int *nx); /* 0 when C % 4 != 0 (scalar path, no workspace) */
int gc_lss_voxel_pooling(const float *geom, const float *x, long long n_points, int n_batch, int C, const float *dx,
                         const float *bx, const int *nx, void *workspace /* or NULL */, float *out, void *stream);

/* Deterministic variant of gc_lss_voxel_pooling (the reference's sort + cumsum is deterministic; fp32 reductions in L2 are
 * not): addends go through 40.24 fixed point and 64-bit integer reductions, which commute exactly -> bit-identical
 * results on every run; each addend is rounded to 2^-24.  workspace: gc_lss_pool_det_workspace_bytes bytes (required). */
size_t gc_lss_pool_det_workspace_bytes(int n_batch, int C, const int *nx);
int gc_lss_voxel_pooling_det(const float *geom_feats, const float *x, long long n_points, int n_batch, int C,
                             const float *dx /*[3] host*/, const float *bx /*[3] host*/, const int *nx /*[3] host*/,
                             void *workspace, float *out, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Evaluation matching: eval_utils.caluclate_tp_fp (utils/eval_utils.py) with common_utils.convert_format / compute_iou
 * (utils/common_utils.py:230-270), for n_frames frames and n_thresh IoU thresholds in one call.  Per frame and threshold:
 * sort the detections by descending score, then greedily, in that order, match each to the still-unmatched ground truth
 * of largest IoU; it is a TP when that IoU (float32, widened to double) is >= the threshold, else a FP.
 *   det_boxes [B][k_max][8][3], det_scores [B][k_max], det_counts [B] (gc_postprocess's outputs), gt_boxes [B][g_max][8][3],
 *   gt_counts [B]; polygons are the bottom-face corners 0..3 (x, y) in float64, IoU = inter / (|A| + |B| - inter) as
 *   float32 (the float64 convex clipping of gc_postprocess's NMS; shapely parity unpinned).
 *   -> sorted_scores [B][k_max] f32 (descending; 0 beyond the count), tp [B][n_thresh][k_max] u8 (1 = TP; FP = 1 - tp
 *   below the count, 0 beyond it).
 *   Ties: equal scores keep their input order (the reference's np.argsort(-score) leaves them unspecified); equal IoUs
 *   match the lowest ground-truth index (np.argmax); a NaN IoU (zero-area detection against a zero-area ground truth)
 *   makes the detection a TP matched to the first NaN, as numpy's max / argmax do.  Scores must be finite.
 *   Device counts outside [0, k_max] / [0, g_max] are clamped into that range.
 *   Argument errors (GC_EINVAL): NULL pointers, n_frames outside 1..65535, k_max or g_max outside 1..1024, n_thresh
 *   outside 1..8.  workspace: gc_eval_workspace_bytes bytes (0 for arguments outside those ranges).  No allocation, no
 *   host synchronisation.
 * ------------------------------------------------------------------------------------------- */
size_t gc_eval_workspace_bytes(int n_frames, int k_max, int g_max);
int gc_eval_match(const float *det_boxes, const float *det_scores, const int *det_counts, int k_max, const float *gt_boxes,
                  const int *gt_counts, int g_max, int n_frames, const double *iou_thresh /*[n_thresh] host*/, int n_thresh,
                  void *workspace, float *sorted_scores, uint8_t *tp, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GENCOMM_B200_H_ */
