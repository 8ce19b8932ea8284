// Row-staged 3x3 convolution (stride 1, padding 1) on tcgen05 for the wide feature maps of the detector: the level-1 / level-2
// layers of BaseBEVBackbone (models/sub_modules/base_bev_backbone.py:96-124: 64 ch at 128 x 256, 128 ch at 64 x 128) and the
// second layer of the shrink header (models/sub_modules/downsample_conv.py:7-50).  Same arithmetic as k_me_conv's plain
// path (implicit_gemm.cuh): bf16x3 -- value + residual bf16 planes of both operands, three MMAs per product, fp32
// accumulation in TMEM -- same packed weights (k_me_pack, split), same epilogues.  What changes is the data movement.
//
// k_me_conv stages one [128 pixels x 32 channels] operand per (tap, channel chunk): every input row segment is gathered from
// L2 nine times.  The launch list of the backbone (profiles/r02u_backbone_launches.txt) shows what that costs: the four
// 64-channel layers at 128 x 256 move 2.4 GB each through L2 in 500 us = 4.8 TB/s -- L2-bandwidth bound at 155 dense
// TFLOP/s, a third of what the 256-channel layers reach with the same kernel.  Here a CTA owns R output rows x 128 pixels
// and stages, per 32-channel chunk, the R + 2 input rows it needs ONCE ([channel group][row][130 pixels] of 16-byte pixel
// vectors, x halo included); the nine taps are nine descriptor start addresses into those rows (row r + ky, pixel kx), so
// the operand traffic drops from 9x to (R + 2) / R x of the input and the staging work with it.  The weights of one
// (chunk, tap) stream through a ring of bulk copies (TMA) issued by the MMA lane.
#include <stdlib.h>

#include "common.cuh"
#include "conv_rows.cuh"
#include "implicit_gemm.cuh"

namespace gc {
namespace cr {

using namespace ptx;
using me::bf16_residual;

constexpr int kStagers = 256;     // warps 0-7: operand staging (cp.async)
constexpr int kEpi = 128;         // warps 8-11: epilogue (warp w reads TMEM lanes 32 (w % 4) ..)
constexpr int kThreads = kStagers + kEpi + 32;   // warp 12 feeds the tensor core
constexpr int kRowPx = 130;       // staged pixels per row: x0 - 1 .. x0 + 128
constexpr int kSc = 32;           // channels per chunk (4 groups of 8 = two K = 16 MMAs per plane pair)

#ifdef CR_TRACE                   // scripts/probe/conv_rows_trace.cu: where CTA 8's roles wait
__device__ long long g_trace[16];
#define CR_ACC(i, expr) do { const long long t__ = clock64(); expr; if (blockIdx.x == 8) g_trace[i] += clock64() - t__; } while (0)
#define CR_SET(i, v) do { if (blockIdx.x == 8) g_trace[i] = (v); } while (0)
#else
#define CR_ACC(i, expr) do { expr; } while (0)
#define CR_SET(i, v) do { } while (0)
#endif

// [plane hi|lo][group 4][row R+2][130 px][16 B]; the group stride is padded by 16 bytes so that the four groups of a pixel
// (consecutive threads) store to different bank quads
__host__ __device__ constexpr int group_bytes(int R) { return (R + 2) * kRowPx * 16 + 16; }
__host__ __device__ constexpr int plane_bytes(int R) { return 4 * group_bytes(R); }
__host__ __device__ constexpr int a_stage_bytes(int R) { return 2 * plane_bytes(R); }
__host__ __device__ constexpr int b_stage_bytes(int NOUT) { return 2 * kSc * NOUT * 2; }   // hi plane, lo plane (k_me_pack, split)
__host__ __device__ constexpr int smem_bytes(int NOUT, int R, int NB) { return 2 * a_stage_bytes(R) + NB * b_stage_bytes(NOUT); }

// 16-byte asynchronous copy global -> shared; bytes == 0 writes zeros (the source address must still be valid)
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, uint32_t bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Persistent: CTA b takes tiles b, b + gridDim.x, ...; tile = R output rows x 128 pixels of one agent.  Three roles run
// decoupled through mbarriers so that staging (tile k + 1), MMAs (tile k) and the epilogue (tile k - 1) overlap:
//   stagers  -> a_full[2]   -> feeder      (operand rows of one 32-channel chunk, double-buffered)
//   feeder   -> a_empty[2]  -> stagers     (tcgen05.commit once the chunk's MMAs retired)
//   feeder   -> acc_full[2] -> epilogue    (two accumulator sets of R * NOUT TMEM columns)
//   epilogue -> acc_empty[2]-> feeder
// EPI 5: bias + ReLU -> channel-last bf16 value + residual planes (the next layer's operand); EPI 3: bias + ReLU -> fp32 NCHW
template <int NOUT, int R, int NB, int EPI>
__global__ void __launch_bounds__(kThreads, 1)
k_conv_rows(const uint4 *__restrict__ xh, const uint4 *__restrict__ xl, const uint4 *__restrict__ wp, const float *__restrict__ bias,
            int n_tiles, int C, int H, int W, int out_ch_total, int out_ch_off, float *__restrict__ out, uint4 *__restrict__ oh,
            uint4 *__restrict__ ol) {
    constexpr int kGroup = group_bytes(R), kPlane = plane_bytes(R), kAStage = a_stage_bytes(R), kBStage = b_stage_bytes(NOUT);
    constexpr int kBPlane = kSc * NOUT * 2;
    constexpr int kSet = R * NOUT;                    // TMEM columns of one accumulator set
    static_assert(2 * kSet == 512, "two accumulator sets fill the 512 TMEM columns");
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *a_s = smem, *b_s = smem + 2 * kAStage;
    __shared__ __align__(8) uint64_t a_full[2], a_empty[2], b_full[NB], b_empty[NB], acc_full[2], acc_empty[2];
    __shared__ uint32_t s_tmem;
    __shared__ float s_bias[NOUT];

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int tiles_x = W / 128, tiles_agent = tiles_x * (H / R);
    const int chunks = C / kSc, C8 = C / 8, HW = H * W;

    if (warp == 0) tmem_alloc<512>(&s_tmem);
    if (tid == 32) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(smem_u32(&a_full[i]), kStagers); mbar_init(smem_u32(&a_empty[i]), 1);
            mbar_init(smem_u32(&acc_full[i]), 1); mbar_init(smem_u32(&acc_empty[i]), kEpi);
        }
        for (int i = 0; i < NB; ++i) { mbar_init(smem_u32(&b_full[i]), 1); mbar_init(smem_u32(&b_empty[i]), 1); }
        mbar_init_fence();
    }
    if (tid < NOUT) s_bias[tid] = bias[tid];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const long long t_begin = clock64();

    if (warp == (kStagers + kEpi) / 32) {
        // ---- feeder: one elected lane streams the weights and issues every MMA ----
        if (elect_one()) {
            const uint32_t a_base = smem_u32(a_s), b_base = smem_u32(b_s);
            constexpr uint32_t idesc = make_idesc(128, NOUT);
            const int my_tiles = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
            const int per_tile = chunks * 9, total = my_tiles * per_tile;
            auto load_b = [&](int s) {   // weights of step s: (chunk, tap) = stage tap * chunks + chunk of the packed tensor
                const int st = s % per_tile, c = st / 9, tap = st - 9 * c, nb = s % NB;
                bulk_load(b_base + (uint32_t)nb * kBStage, wp + (size_t)(tap * chunks + c) * (kBStage / 16), kBStage, smem_u32(&b_full[nb]));
            };
            for (int s = 0; s < NB && s < total; ++s) load_b(s);     // every buffer starts full
            int s = 0, g = 0;
            for (int k = 0; k < my_tiles; ++k) {
                const int set = k & 1;
                if (k >= 2) { CR_ACC(1, mbar_wait(smem_u32(&acc_empty[set]), (uint32_t)((k >> 1) - 1) & 1u)); tc_fence_after(); }
                const uint32_t acc0 = tmem + (uint32_t)(set * kSet);
                for (int c = 0; c < chunks; ++c, ++g) {
                    const int ab = g & 1;
                    CR_ACC(0, mbar_wait(smem_u32(&a_full[ab]), (uint32_t)(g >> 1) & 1u));
                    tc_fence_after();
                    const uint64_t a_desc0 = make_desc(a_base + (uint32_t)ab * kAStage, (uint32_t)kGroup, 128u);
#pragma unroll 1
                    for (int tap = 0; tap < 9; ++tap, ++s) {
                        const int ky = tap / 3, kx = tap - 3 * ky, nb = s % NB;
                        CR_ACC(2, mbar_wait(smem_u32(&b_full[nb]), (uint32_t)(s / NB) & 1u));
                        const uint64_t b_desc0 = make_desc(b_base + (uint32_t)nb * kBStage, NOUT * 16u, 128u);
                        const uint64_t a_tap = a_desc0 + (uint64_t)(ky * kRowPx + kx);
                        const uint32_t first = (c > 0 || tap > 0) ? 1u : 0u;
#pragma unroll
                        for (int r = 0; r < R; ++r) {
#pragma unroll
                            for (int j = 0; j < kSc / 16; ++j) {
                                // +1 in the address field = 16 bytes: (row r + ky, pixel kx) of channel groups 2j, 2j + 1
                                const uint64_t a_hi = a_tap + (uint64_t)((2 * j * kGroup) / 16 + r * kRowPx);
                                const uint64_t a_lo = a_hi + (uint64_t)(kPlane / 16);
                                const uint64_t b_hi = b_desc0 + (uint64_t)(2 * j * NOUT);
                                const uint64_t b_lo = b_hi + (uint64_t)(kBPlane / 16);
                                const uint32_t acc = acc0 + (uint32_t)(r * NOUT);
                                mma_bf16(acc, a_hi, b_hi, idesc, j > 0 ? 1u : first);
                                mma_bf16(acc, a_lo, b_hi, idesc, 1u);
                                mma_bf16(acc, a_hi, b_lo, idesc, 1u);
                            }
                        }
                        mma_commit(smem_u32(&b_empty[nb]));
                        // refill the buffer the PREVIOUS step used (its MMAs retire while this step's execute)
                        if (s >= 1 && s - 1 + NB < total) {
                            const int pb = (s - 1) % NB;
                            CR_ACC(3, mbar_wait(smem_u32(&b_empty[pb]), (uint32_t)((s - 1) / NB) & 1u));
                            load_b(s - 1 + NB);
                        }
                    }
                    mma_commit(smem_u32(&a_empty[ab]));
                }
                mma_commit(smem_u32(&acc_full[set]));
            }
        }
        __syncwarp();
    } else if (warp < kStagers / 32) {
        // ---- stagers: the R + 2 input rows of every 32-channel chunk, once, by 16-byte cp.async (zero fill outside the map) ----
        constexpr int kItems = 2 * 4 * (R + 2) * kRowPx;           // 16-byte pixel vectors per chunk
        constexpr int kIters = (kItems + kStagers - 1) / kStagers;
        const uint32_t a_base = smem_u32(a_s);
        int g = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const int agent = t / tiles_agent, rem = t - agent * tiles_agent;
            const int x0 = (rem % tiles_x) * 128, y0 = (rem / tiles_x) * R;
            const uint4 *src_plane[2] = {xh + (size_t)agent * HW * C8, xl + (size_t)agent * HW * C8};
            for (int c = 0; c < chunks; ++c, ++g) {
                const int ab = g & 1;
                if (g >= 2) {   // MMAs of chunk g - 2 retired
                    if (tid == 0) CR_ACC(4, mbar_wait(smem_u32(&a_empty[ab]), (uint32_t)((g >> 1) - 1) & 1u));
                    else mbar_wait(smem_u32(&a_empty[ab]), (uint32_t)((g >> 1) - 1) & 1u);
                }
                const uint32_t dst = a_base + (uint32_t)ab * kAStage;
#pragma unroll 5
                for (int k = 0; k < kIters; ++k) {
                    const int it = k * kStagers + tid;
                    if (it < kItems) {
                        const int gq = it & 3, pl = (it >> 2) & 1, rest = it >> 3;
                        const int row = rest / kRowPx, px = rest - row * kRowPx;
                        const int yy = y0 - 1 + row, xx = x0 - 1 + px;
                        const bool in = yy >= 0 && yy < H && xx >= 0 && xx < W;
                        const uint4 *src = src_plane[pl] + (in ? (size_t)(yy * W + xx) * C8 + c * 4 + gq : 0);
                        cp_async16(dst + (uint32_t)(pl * kPlane + gq * kGroup + (row * kRowPx + px) * 16), src, in ? 16u : 0u);
                    }
                }
                cp_async_wait_all();
                fence_async_smem();
                mbar_arrive(smem_u32(&a_full[ab]));
            }
        }
    } else {
        // ---- epilogue: warp w reads TMEM lanes 32 (w % 4) .. +31 (= pixels), every column of the tile's accumulator set ----
        const int q4 = warp & 3;
        int k = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++k) {
            const int agent = t / tiles_agent, rem = t - agent * tiles_agent;
            const int x = (rem % tiles_x) * 128 + q4 * 32 + lane, y0 = (rem / tiles_x) * R;
            const int set = k & 1;
            mbar_wait(smem_u32(&acc_full[set]), (uint32_t)(k >> 1) & 1u);
            tc_fence_after();
#pragma unroll 1
            for (int r = 0; r < R; ++r) {
                const size_t p_out = (size_t)(y0 + r) * W + x;
                const uint32_t taddr = tmem + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(set * kSet + r * NOUT);
#pragma unroll 2
                for (int c16 = 0; c16 < NOUT; c16 += 16) {
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
                        const size_t o = ((size_t)agent * HW + p_out) * (out_ch_total >> 3) + ((out_ch_off + c16) >> 3);
                        oh[o] = make_uint4(h[0], h[1], h[2], h[3]); oh[o + 1] = make_uint4(h[4], h[5], h[6], h[7]);
                        ol[o] = make_uint4(l[0], l[1], l[2], l[3]); ol[o + 1] = make_uint4(l[4], l[5], l[6], l[7]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int ch = c16 + i;
                            out[((size_t)agent * out_ch_total + out_ch_off + ch) * HW + p_out] = fmaxf(v[i] + s_bias[ch], 0.0f);
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
    if (tid == 0) CR_SET(5, clock64() - t_begin);
    if (warp == 0) tmem_free<512>(tmem);
}

template <int NOUT, int R, int NB, int EPI>
static int launch(cudaStream_t st, const ConvLayer &L) {
    constexpr int kSmem = smem_bytes(NOUT, R, NB);
    static_assert(kSmem <= 226 * 1024, "k_conv_rows: shared memory");
    static int sms = 0;
    if (!sms) {
        cudaError_t e = cudaFuncSetAttribute(k_conv_rows<NOUT, R, NB, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        int dev = 0, n = 0;
        if (e == cudaSuccess) e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess || n <= 0) { (void)cudaGetLastError(); set_error("k_conv_rows: launch set-up failed (%d)", (int)e); return e != cudaSuccess ? (int)e : (int)cudaErrorUnknown; }
        sms = n;
    }
    const int H = L.Ho(), W = L.Wo(), n_tiles = L.A * (W / 128) * (H / R);
    k_conv_rows<NOUT, R, NB, EPI><<<n_tiles < sms ? n_tiles : sms, kThreads, kSmem, st>>>(L.xh, L.xl, L.w, L.bias, n_tiles, L.c_in, H, W,
                                                                                         L.out_ch_total, L.out_ch_off, L.out, L.oh, L.ol);
    GC_LAUNCH_CHECK("k_conv_rows");
    return GC_OK;
}

}  // namespace cr

bool conv_rows_eligible(const ConvLayer &L) {
    // opt-in since k_conv_tma: the TMA-fed kernel runs the same layers faster (32 agents: 64 ch 263 vs 276 us, 128 ch 166 vs 214 us).
    // Read per call so that a test can run both paths in one process.
    const char *e = getenv("GC_CONV_ROWS");
    if (!(e && e[0] == '1')) return false;
    if (L.taps != 9 || L.stride != 1 || L.up != 1 || (L.epi != 3 && L.epi != 5) || L.c_in != L.C || L.Wo() % 128 != 0 || L.c_in % 32 != 0)
        return false;
    if (L.n_out == 64) return L.Ho() % 4 == 0;
    if (L.n_out == 128) return L.Ho() % 2 == 0;
    return false;
}

int conv_rows(cudaStream_t st, const ConvLayer &L) {
    if (L.n_out == 64) return L.epi == 5 ? cr::launch<64, 4, 3, 5>(st, L) : cr::launch<64, 4, 3, 3>(st, L);
    return L.epi == 5 ? cr::launch<128, 2, 4, 5>(st, L) : cr::launch<128, 2, 4, 3>(st, L);
}

}  // namespace gc
