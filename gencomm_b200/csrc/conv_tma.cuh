// Persistent TMA-fed version of the plain path of k_me_conv (implicit_gemm.cuh): stride-1 3x3 (padding 1) or 1x1 convolution over
// channel-last bf16 value + residual planes as a tcgen05 implicit GEMM in bf16x3.
//
// Why (profiles/r02ae_conv_stagers.txt): in k_me_conv 256 threads gather every [128 px x 32 ch] operand stage through registers
// (LDG -> STS -> fence.proxy.async -> 256 mbarrier arrivals).  The ncu source page of the 256-channel layer shows those threads
// busy, not waiting: STS + FENCE.VIEW.ASYNC + SYNCS.ARRIVE take as many stall samples as the wait for a free stage, L2 -> SM
// traffic sits at 28 % of peak, the tensor pipe idles half the time.  A cp.async variant of the same gather with decoupled
// epilogue warps was measured slower still (7.2 vs 6.0 ms per backbone call).  The gather is what TMA is for:
//   * the activation planes are a 4-D tensor (C, W, H, agent); the operand of tap (ky, kx) for a tile of BH rows x BW pixels
//     (BH * BW = 128) is the box {32 ch, BW, BH, 1} at (chunk * 32, x0 + kx - 1, y0 + ky - 1, agent) -- padding is TMA's
//     out-of-bounds zero fill -- written with the 64-byte swizzle, which is exactly UMMA's K-major SWIZZLE_64B operand layout
//     (row = pixel, 64 bytes = 32 channels): no thread touches the operand;
//   * one producer lane issues, per stage, two tensor loads (value + residual plane) and one bulk copy of packed weights on one
//     mbarrier; one feeder lane issues the MMAs; four epilogue warps drain one of two TMEM accumulator sets while the next
//     tile accumulates into the other.  A CTA owns an SM for the whole launch and walks tiles b, b + gridDim.x, ...
// Same packed weights (k_me_pack, split), same arithmetic and epilogues as k_me_conv: results are bit-identical.
#pragma once
#include <stdlib.h>

#include "implicit_gemm.cuh"

namespace gc {
namespace ct {

using namespace ptx;
using me::bf16_residual;
using me::gelu_erf;

constexpr int kEpi = 256;                            // warps 0-7: epilogue (warp w: TMEM lanes 32 (w % 4) .., column half w / 4)
constexpr int kThreads = kEpi + 64;                  // warp 8: feeder (MMA issue), warp 9: producer (TMA)
constexpr int kSc = 32;                              // channels per stage = one 64-byte swizzle row
constexpr int kAPlane = 128 * kSc * 2, kAStage = 2 * kAPlane;   // value + residual

#ifdef CT_TRACE                  // scripts/probe/conv_tma_trace.cu: where CTA 8's feeder / producer / epilogue spend their cycles
__device__ long long g_trace[16];
#define CT_ACC(i, expr) do { const long long t__ = clock64(); expr; if (blockIdx.x == 8) g_trace[i] += clock64() - t__; } while (0)
#define CT_SET(i, v) do { if (blockIdx.x == 8) g_trace[i] = (v); } while (0)
#else
#define CT_ACC(i, expr) do { expr; } while (0)
#define CT_SET(i, v) do { } while (0)
#endif

__host__ __device__ constexpr int b_stage_bytes(int NOUT) { return kSc * NOUT * 2 * 2; }
// plane epilogue (EPI 5, N <= 128): every warp transposes its 32 pixels x N / 2 channels (value + residual) through shared memory so
// that a store instruction writes whole 128-byte lines (4 - 8 pixels x 64 - 128 contiguous bytes) instead of 32 scattered 16-byte
// pieces -- the scattered form made the short-K layers (ConvTranspose2d phases) epilogue-bound: 6.7 k cycles per tile against 0.8 k
// cycles of MMAs (profiles/r02aj_conv_tma_trace.txt)
// (deep-K layers keep the shared memory for a deeper operand ring instead: STG is chosen per launch from the stage count)
__host__ __device__ constexpr bool stage_planes(int NOUT, int EPI) { return EPI == 5 && NOUT <= 128; }
__host__ __device__ constexpr int out_stage_bytes(int NOUT, int EPI, bool STG) { return STG && stage_planes(NOUT, EPI) ? (kEpi / 32) * 2 * 32 * NOUT : 0; }
__host__ __device__ constexpr int ring_depth(int NOUT, int EPI, bool STG) {
    return (200 * 1024 - out_stage_bytes(NOUT, EPI, STG)) / (kAStage + b_stage_bytes(NOUT)) > 8
               ? 8
               : (200 * 1024 - out_stage_bytes(NOUT, EPI, STG)) / (kAStage + b_stage_bytes(NOUT));
}
__host__ __device__ constexpr int smem_bytes(int NOUT, int EPI, bool STG) {
    return ring_depth(NOUT, EPI, STG) * (kAStage + b_stage_bytes(NOUT)) + out_stage_bytes(NOUT, EPI, STG) + 1024;
}

// H x W: the output grid; tiles of BH rows x BW pixels, BW = min(W, 128), BH = 128 / BW.  stride 2: the tensor maps traverse the
// input with element strides {1, 2, 2, 1} (box {32, 2 BW, 2 BH, 1} -> BW x BH pixels in shared memory), start (2 x0 + kx - 1, ..).
// up_dy < 0: ALL up * up phases of a ConvTranspose2d (kernel == stride == up) in one launch -- n_tiles counts (tile, phase) pairs,
// phase = t % (up * up) writes pixel (y*up + phase / up, x*up + phase % up) with the weights at wp + phase * stages * stage bytes
// (phases of one tile run on neighbouring CTAs at the same time: its operand comes from L2 once).
// EPI as in k_me_conv: 0 bias, 1 bias + GELU, 3 bias + ReLU -> fp32 [A][out_ch_total][H*up][W*up] at (y*up + up_dy, x*up + up_dx);
// 2 bias + GELU -> fp32 channel-last [A][HW][out_ch_total]; 5 bias + ReLU -> bf16 value + residual planes [A][HW*up*up][out_ch_total]
// MC: CTA pairs (cluster of 2) walk tile pairs in lock step; each CTA fetches half of every weight stage and multicasts it to both
// (half the weight bytes from L2 per SM); a ring slot is free when BOTH CTAs' MMAs on it retired (commit multicast, count 2).
template <int NOUT, int TAPS, int EPI, bool MC, bool STG>
__global__ void __launch_bounds__(kThreads, 1)
k_conv_tma(const __grid_constant__ CUtensorMap map_h, const __grid_constant__ CUtensorMap map_l, const uint4 *__restrict__ wp,
           const float *__restrict__ bias, int n_tiles, int c_in, int H, int W, int BW, int stride, int n_store, int out_ch_total, int out_ch_off,
           float *__restrict__ out, uint4 *__restrict__ oh, uint4 *__restrict__ ol, int up, int up_dy, int up_dx) {
    constexpr int NS = ring_depth(NOUT, EPI, STG);
    constexpr int kBStage = b_stage_bytes(NOUT), kBPlane = kSc * NOUT * 2;
    static_assert(NS >= 3, "ring too shallow");
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full[NS], empty[NS], acc_full[2], acc_empty[2];
    __shared__ uint32_t s_tmem;
    __shared__ float s_bias[NOUT];

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const uint32_t a_base = (smem_u32(smem_raw) + 1023u) & ~1023u;       // swizzle atoms: 512-byte aligned tiles
    const uint32_t b_base = a_base + NS * kAStage;
    const int BH = me::kPix / BW, tiles_x = W / BW, tiles_agent = tiles_x * (H / BH);
    const int chunks = c_in / kSc, stages = TAPS * chunks, HW = H * W;
    const int n_phase = up_dy < 0 ? up * up : 1;

    if (warp == 0) tmem_alloc<2 * NOUT>(&s_tmem);
    if (tid == 32) {
        for (int i = 0; i < NS; ++i) { mbar_init(smem_u32(&full[i]), 1); mbar_init(smem_u32(&empty[i]), MC ? 2 : 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&acc_full[i]), 1); mbar_init(smem_u32(&acc_empty[i]), kEpi); }
        mbar_init_fence();
    }
    for (int i = tid; i < NOUT; i += kThreads) s_bias[i] = (bias && i < n_store) ? bias[i] : 0.0f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (MC) cluster_sync_all();      // the peer's barriers exist before anything is multicast at them
    const uint32_t tmem = s_tmem;
    const long long t_begin = clock64();
    // tiles of this CTA: t0, t0 + t_step, ...; pairs take tiles (2q, 2q + 1) so that both CTAs run the same number of stages
    const int rank = MC ? (int)cluster_ctarank() : 0;
    const int t0 = MC ? 2 * ((int)blockIdx.x >> 1) + rank : (int)blockIdx.x, t_step = (int)gridDim.x;
    const int my_tiles = t0 < n_tiles ? (n_tiles - t0 + t_step - 1) / t_step : 0;

    if (warp == kEpi / 32) {
        // ---- feeder ----
        if (elect_one()) {
            constexpr uint32_t idesc = make_idesc(128, NOUT);
            int g = 0;
            for (int k = 0; k < my_tiles; ++k) {
                const int set = k & 1;
                if (k >= 2) { CT_ACC(1, mbar_wait(smem_u32(&acc_empty[set]), (uint32_t)((k >> 1) - 1) & 1u)); tc_fence_after(); }
                const uint32_t acc = tmem + (uint32_t)(set * NOUT);
                for (int s = 0; s < stages; ++s, ++g) {
                    const int sb = g % NS;
                    CT_ACC(0, mbar_wait(smem_u32(&full[sb]), (uint32_t)(g / NS) & 1u));
                    tc_fence_after();
                    const uint64_t a_d = make_desc_sw64(a_base + (uint32_t)sb * kAStage);
                    const uint64_t b_d = make_desc(b_base + (uint32_t)sb * kBStage, NOUT * 16u, 128u);
#pragma unroll
                    for (int j = 0; j < kSc / 16; ++j) {   // +1 in the address field = 16 bytes; K = 16 bf16 = 32 bytes of the row
                        const uint64_t a_hi = a_d + (uint64_t)(2 * j), a_lo = a_hi + (uint64_t)(kAPlane / 16);
                        const uint64_t b_hi = b_d + (uint64_t)(2 * j * NOUT), b_lo = b_hi + (uint64_t)(kBPlane / 16);
                        mma_bf16(acc, a_hi, b_hi, idesc, (s > 0 || j > 0) ? 1u : 0u);
                        mma_bf16(acc, a_lo, b_hi, idesc, 1u);
                        mma_bf16(acc, a_hi, b_lo, idesc, 1u);
                    }
                    if (MC) mma_commit_multicast(smem_u32(&empty[sb]), (uint16_t)3);
                    else mma_commit(smem_u32(&empty[sb]));
                }
                mma_commit(smem_u32(&acc_full[set]));
            }
        }
        __syncwarp();
    } else if (warp == kEpi / 32 + 1) {
        // ---- producer: per stage two tensor loads (value, residual plane) + the packed weights, one mbarrier ----
        if (elect_one()) {
            int g = 0;
            for (int t = t0; t < n_tiles; t += t_step) {
                const int ph = t % n_phase, tt = t / n_phase;
                const int agent = tt / tiles_agent, rem = tt - agent * tiles_agent;
                const int x0 = (rem % tiles_x) * BW, y0 = (rem / tiles_x) * BH;
                const uint4 *wph = wp + (size_t)ph * stages * (kBStage / 16);
                for (int s = 0; s < stages; ++s, ++g) {
                    const int sb = g % NS;
                    if (g >= NS) CT_ACC(2, mbar_wait(smem_u32(&empty[sb]), (uint32_t)((g / NS) - 1) & 1u));   // MMAs of stage g - NS retired
                    const int tap = s / chunks, chunk = s - tap * chunks;
                    const int ky = TAPS == 1 ? 1 : tap / 3, kx = TAPS == 1 ? 1 : tap - 3 * ky;
                    const uint32_t bar = smem_u32(&full[sb]), a_dst = a_base + (uint32_t)sb * kAStage;
                    mbar_expect_tx(bar, (uint32_t)(kAStage + kBStage));
                    tma_load_4d(a_dst, &map_h, chunk * kSc, x0 * stride + kx - 1, y0 * stride + ky - 1, agent, bar);
                    tma_load_4d(a_dst + kAPlane, &map_l, chunk * kSc, x0 * stride + kx - 1, y0 * stride + ky - 1, agent, bar);
                    if (MC)
                        bulk_copy_multicast(b_base + (uint32_t)sb * kBStage + (uint32_t)rank * (kBStage / 2),
                                            wph + (size_t)s * (kBStage / 16) + (size_t)rank * (kBStage / 32), kBStage / 2, bar, (uint16_t)3);
                    else
                        bulk_copy(b_base + (uint32_t)sb * kBStage, wph + (size_t)s * (kBStage / 16), kBStage, bar);
                }
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue: lane = pixel (row bh, column bw of the tile); warps 0-3 take the first half of the columns, 4-7 the second ----
        const size_t hw_store = (size_t)HW * up * up;
        const int q4 = warp & 3, m = q4 * 32 + lane, col0 = (warp >> 2) * (NOUT / 2);
        int k = 0;
        for (int t = t0; t < n_tiles; t += t_step, ++k) {
            const int ph = t % n_phase, tt = t / n_phase;
            const int dy = up_dy < 0 ? ph / up : up_dy, dx = up_dy < 0 ? ph % up : up_dx;
            const int agent = tt / tiles_agent, rem = tt - agent * tiles_agent;
            const int pyo = (rem / tiles_x) * BH + m / BW, pxo = (rem % tiles_x) * BW + m % BW;
            const int p_out = pyo * W + pxo;
            const size_t p_store = (size_t)(pyo * up + dy) * (W * up) + pxo * up + dx;
            const int set = k & 1;
            if (tid == 0) CT_ACC(3, mbar_wait(smem_u32(&acc_full[set]), (uint32_t)(k >> 1) & 1u));
            else mbar_wait(smem_u32(&acc_full[set]), (uint32_t)(k >> 1) & 1u);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(set * NOUT);
            if constexpr (STG && stage_planes(NOUT, EPI)) if (n_store == NOUT) {
                // this warp's 32 pixels x NOUT / 2 channels: rows of kRow = NOUT bytes per plane, 16-byte chunks XOR-swizzled by the pixel
                constexpr int kRow = NOUT, kCh = kRow / 16, kPlaneB = 32 * kRow;     // chunks per row: 8 (N = 128) or 4 (N = 64)
                const uint32_t sbuf = b_base + NS * kBStage + (uint32_t)warp * (2 * kPlaneB);
#pragma unroll 2
                for (int c16 = 0; c16 < NOUT / 2; c16 += 16) {
                    float v[16];
                    tmem_ld16(taddr + (uint32_t)(col0 + c16), v);
                    uint32_t h[8], l[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float a = fmaxf(v[2 * i] + s_bias[col0 + c16 + 2 * i], 0.0f);
                        const float b = fmaxf(v[2 * i + 1] + s_bias[col0 + c16 + 2 * i + 1], 0.0f);
                        h[i] = pack_bf16(a, b);
                        l[i] = pack_bf16(bf16_residual(a), bf16_residual(b));
                    }
                    const int cc = c16 / 8;
                    const uint32_t r0 = sbuf + (uint32_t)(lane * kRow), x0s = (uint32_t)(((cc) ^ (lane & (kCh - 1))) * 16),
                                   x1s = (uint32_t)(((cc + 1) ^ (lane & (kCh - 1))) * 16);
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(r0 + x0s), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(r0 + x1s), "r"(h[4]), "r"(h[5]), "r"(h[6]), "r"(h[7]) : "memory");
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(r0 + kPlaneB + x0s), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(r0 + kPlaneB + x1s), "r"(l[4]), "r"(l[5]), "r"(l[6]), "r"(l[7]) : "memory");
                }
                // the accumulator columns are in registers / shared memory: release the set before the global stores
                tc_fence_before();
                mbar_arrive(smem_u32(&acc_empty[set]));
                __syncwarp();
                // pixel of lane j as a uint4 index into the planes (fits 32 bits: < 2^31 16-byte vectors per plane)
                const uint32_t o_lane = (uint32_t)(((size_t)agent * hw_store + p_store) * (out_ch_total >> 3) + ((out_ch_off + col0) >> 3));
                const int chunk = lane & (kCh - 1), sub = lane / kCh;
#pragma unroll
                for (int i = 0; i < kCh; ++i) {
                    const int px = i * (32 / kCh) + sub;
                    const uint32_t o = __shfl_sync(0xffffffffu, o_lane, px) + (uint32_t)chunk;
                    const uint32_t src = sbuf + (uint32_t)(px * kRow + ((chunk ^ (px & (kCh - 1))) * 16));
                    uint4 qh, ql;
                    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(qh.x), "=r"(qh.y), "=r"(qh.z), "=r"(qh.w) : "r"(src));
                    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(ql.x), "=r"(ql.y), "=r"(ql.z), "=r"(ql.w) : "r"(src + kPlaneB));
                    oh[o] = qh;
                    ol[o] = ql;
                }
                __syncwarp();
                continue;
            }
#pragma unroll 2
            for (int c16 = col0; c16 < col0 + NOUT / 2; c16 += 16) {
                if (c16 >= n_store) break;
                float v[16];
                tmem_ld16(taddr + (uint32_t)c16, v);
                if (EPI == 5) {
                    uint32_t h[8], l[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float a = fmaxf(v[2 * i] + s_bias[c16 + 2 * i], 0.0f);
                        const float b = fmaxf(v[2 * i + 1] + s_bias[c16 + 2 * i + 1], 0.0f);
                        h[i] = pack_bf16(a, b);
                        l[i] = pack_bf16(bf16_residual(a), bf16_residual(b));
                    }
                    const size_t o = ((size_t)agent * hw_store + p_store) * (out_ch_total >> 3) + ((out_ch_off + c16) >> 3);
                    oh[o] = make_uint4(h[0], h[1], h[2], h[3]); oh[o + 1] = make_uint4(h[4], h[5], h[6], h[7]);
                    ol[o] = make_uint4(l[0], l[1], l[2], l[3]); ol[o + 1] = make_uint4(l[4], l[5], l[6], l[7]);
                } else if (EPI == 2) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = gelu_erf(v[i] + s_bias[c16 + i]);
                    float4 *dst = reinterpret_cast<float4 *>(out + ((size_t)agent * HW + p_out) * out_ch_total + out_ch_off + c16);
#pragma unroll
                    for (int i = 0; i < 4; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const int ch = c16 + i;
                        if (ch < n_store) {
                            float r = v[i] + s_bias[ch];
                            if (EPI == 1) r = gelu_erf(r);
                            if (EPI == 3) r = fmaxf(r, 0.0f);
                            out[((size_t)agent * out_ch_total + out_ch_off + ch) * hw_store + p_store] = r;
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(smem_u32(&acc_empty[set]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (tid == 0) { CT_SET(4, clock64() - t_begin); CT_SET(5, (long long)my_tiles * stages); }
    if (MC) cluster_sync_all();      // no CTA leaves while its peer may still signal its barriers
    if (warp == 0) tmem_free<2 * NOUT>(tmem);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// planes [A][H][W][C] bf16 as the 4-D tensor (C, W, H, A); box = {32 channels, BW, BH, 1} output pixels, 64-byte swizzle, zero fill
// outside; H x W is the INPUT grid, every stride-th pixel is loaded
inline bool encode_plane_map(CUtensorMap *map, const void *plane, int A, int H, int W, int C, int BW, int BH, int stride) {
    const auto encode = tensor_map_encoder();
    if (!encode) return false;
    const cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)A};
    const cuuint64_t gstride[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
    const cuuint32_t box[4] = {(cuuint32_t)kSc, (cuuint32_t)(BW * stride), (cuuint32_t)(BH * stride), 1};
    const cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void *>(plane), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// layers whose output map tiles into BH x BW = 128-pixel boxes; GC_CONV_TMA=0 disables, =1 restricts to stride 1 (A/B)
inline bool conv_tma_eligible(int stride, int C, int c_in, int H, int W, int up) {
    static int on = -1;
    if (on < 0) { const char *e = getenv("GC_CONV_TMA"); on = e ? atoi(e) : 2; }
    if (!on || (stride != 1 && !(stride == 2 && on >= 2)) || C % 8 != 0 || c_in % kSc != 0 || c_in > C) return false;
    const int BW = W < 128 ? W : 128;
    if (BW < 8 || (BW & (BW - 1)) != 0 || W % BW != 0) return false;
    return H % (128 / BW) == 0 && up >= 1;
}

template <int NOUT, int TAPS, int EPI, bool MC, bool STG>
static int launch_conv_tma_mc(cudaStream_t st, int A, const uint4 *xh, const uint4 *xl, const uint4 *wp, const float *bias, int C, int c_in,
                              int H, int W, int H_in, int W_in, int stride, int n_store, int out_ch_total, int out_ch_off, float *out,
                              uint4 *oh, uint4 *ol, int up, int up_dy, int up_dx) {
    constexpr int kSmem = smem_bytes(NOUT, EPI, STG);
    static_assert(kSmem <= 227 * 1024, "k_conv_tma: shared memory");
    static int ctas = 0;      // CTAs per launch: every SM (MC: twice the co-resident cluster count)
    if (!ctas) {
        cudaError_t e = cudaFuncSetAttribute(k_conv_tma<NOUT, TAPS, EPI, MC, STG>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        int dev = 0, n = 0;
        if (e == cudaSuccess) e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess && MC) {
            cudaLaunchConfig_t cfg = {};
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.gridDim = dim3(2 * (n / 2)); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = kSmem; cfg.attrs = at; cfg.numAttrs = 1;
            int clusters = 0;
            e = cudaOccupancyMaxActiveClusters(&clusters, k_conv_tma<NOUT, TAPS, EPI, MC, STG>, &cfg);
            n = 2 * clusters;
        }
        if (e != cudaSuccess || n <= 0) {
            (void)cudaGetLastError();
            set_error("k_conv_tma: launch set-up failed (%d)", (int)e);
            return e != cudaSuccess ? (int)e : (int)cudaErrorUnknown;
        }
        ctas = n;
    }
    const int BW = W < 128 ? W : 128, BH = 128 / BW;
    CUtensorMap mh, ml;
    const int Hi = H_in > 0 ? H_in : H, Wi = W_in > 0 ? W_in : W;
    if (!encode_plane_map(&mh, xh, A, Hi, Wi, C, BW, BH, stride) || !encode_plane_map(&ml, xl, A, Hi, Wi, C, BW, BH, stride)) {
        set_error("k_conv_tma: cuTensorMapEncodeTiled failed (A=%d H=%d W=%d C=%d stride=%d)", A, Hi, Wi, C, stride);
        return (int)cudaErrorInvalidValue;
    }
    const int n_tiles = A * (H * W / me::kPix) * (up_dy < 0 ? up * up : 1);
    int grid = n_tiles < ctas ? n_tiles : ctas;
    if (MC) grid &= ~1;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = kSmem; cfg.stream = st;
    if (MC) {
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
    }
    cudaError_t e = cudaLaunchKernelEx(&cfg, k_conv_tma<NOUT, TAPS, EPI, MC, STG>, mh, ml, wp, bias, n_tiles, c_in, H, W, BW, stride, n_store,
                                       out_ch_total, out_ch_off, out, oh, ol, up, up_dy, up_dx);
    if (e != cudaSuccess) { (void)cudaGetLastError(); set_error("k_conv_tma: %s", cudaGetErrorString(e)); return (int)e; }
    return GC_OK;
}

// weight-heavy layers (N >= 128) with an even tile count run as CTA pairs sharing every weight stage; GC_CONV_MC=0 disables
template <int NOUT, int TAPS, int EPI>
static int launch_conv_tma(cudaStream_t st, int A, const uint4 *xh, const uint4 *xl, const uint4 *wp, const float *bias, int C, int c_in,
                           int H, int W, int H_in, int W_in, int stride, int n_store, int out_ch_total, int out_ch_off, float *out,
                           uint4 *oh, uint4 *ol, int up, int up_dy, int up_dx) {
    static const bool mc_on = !(getenv("GC_CONV_MC") && getenv("GC_CONV_MC")[0] == '0');
    const int n_tiles = A * (H * W / me::kPix);
    // short-K plane layers are bound by their epilogue: staged (coalesced) stores; deep-K layers by the operand ring: deeper ring
    const bool stg = stage_planes(NOUT, EPI) && TAPS * (c_in / kSc) <= 36;
    if constexpr (NOUT >= 128) {
        if (mc_on && up_dy >= 0 && n_tiles % 2 == 0 && n_tiles >= 4) {      // (fused phases: the CTAs of a pair would need different weights)
            if (stg)
                return launch_conv_tma_mc<NOUT, TAPS, EPI, true, stage_planes(NOUT, EPI)>(st, A, xh, xl, wp, bias, C, c_in, H, W, H_in, W_in, stride,
                                                                                          n_store, out_ch_total, out_ch_off, out, oh, ol, up,
                                                                                          up_dy, up_dx);
            return launch_conv_tma_mc<NOUT, TAPS, EPI, true, false>(st, A, xh, xl, wp, bias, C, c_in, H, W, H_in, W_in, stride, n_store,
                                                                    out_ch_total, out_ch_off, out, oh, ol, up, up_dy, up_dx);
        }
    }
    if (stg)
        return launch_conv_tma_mc<NOUT, TAPS, EPI, false, stage_planes(NOUT, EPI)>(st, A, xh, xl, wp, bias, C, c_in, H, W, H_in, W_in, stride, n_store,
                                                                                   out_ch_total, out_ch_off, out, oh, ol, up, up_dy, up_dx);
    return launch_conv_tma_mc<NOUT, TAPS, EPI, false, false>(st, A, xh, xl, wp, bias, C, c_in, H, W, H_in, W_in, stride, n_store, out_ch_total,
                                                             out_ch_off, out, oh, ol, up, up_dy, up_dx);
}

}  // namespace ct
}  // namespace gc
