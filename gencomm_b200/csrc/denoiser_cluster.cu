// Cluster-resident DiffusionUNet for sm_100a: the 26 width-8 layers of one denoiser evaluation (and, when fused,
// conv_in in front and norm_out + conv_out + the sampler update behind them) run inside ONE thread-block cluster
// per agent.  The agent's activations never leave the SMs: every 8-channel tensor lives in shared memory, split
// into 8 row bands (one per CTA of the cluster); 3x3 halos are read from the neighbouring CTA through
// distributed shared memory, GroupNorm statistics are exchanged by remote shared-memory stores, and the only
// synchronisation between layers is one cluster barrier.
//
// Replaces (paths relative to /root/reference/opencood):
//   models/gencomm_modules/unet.py:307-344 DiffusionUNet.forward, :81-138 ResnetBlock, :59-78 Downsample,
//        :40-56 Upsample, :36-37 GroupNorm(4, eps 1e-6), :31-33 swish
//   models/gencomm_modules/cond_diff.py:321-329 p_sample_loop (the T evaluations of one agent run back to back in the
//        same cluster, so x_t stays in L2 between steps)
// for the shipped denoiser shape (ch=8, ch_mult=[1,1], num_res_blocks=2, no attention) at H x W = 64 x 128.
//
// Tensor-core formulation (tcgen05, tf32 operands, fp32 accumulation in TMEM) - "input-row stationary":
//   D[128 pixels of input row i, 32] += A_i[128, 8 cin] * B_kx[8 cin, 4 blocks x 8 cout]      (one MMA per tap kx)
// where block j of B holds the weights of tap ky = 2 - j (block 3 = 0).  The 32 accumulator columns of input row i
// start at TMEM column 8 i, i.e. block j lands in the accumulator of output row i - 2 + j (kept at column
// 8 (r + 2)): one staged row feeds all three output rows it contributes to, so a 3x3 layer costs 3 MMAs per input
// row and channel group instead of 9, and the staged row is read in place for the three kx taps (descriptor start
// address shifted by one 16-byte pixel).  TMEM columns are zeroed with tcgen05.st before the first MMA.
#include <cooperative_groups.h>
#include <cuda_fp16.h>
#include <stddef.h>
#include <stdlib.h>

#include "common.cuh"
#include "denoiser_cluster.cuh"
#include "denoiser_tc.cuh"
#include "ptx.cuh"

namespace gc {
namespace cl {

namespace cg = cooperative_groups;
using namespace ptx;

constexpr int kStageWarps = 16;                    // staging + epilogue warps
constexpr int kStageThreads = kStageWarps * 32;    // 512
constexpr int kMmaWarp = kStageWarps;              // warp 16: one elected lane issues every tcgen05.mma of the CTA
constexpr int kThreads = kStageThreads + 32;       // 544
constexpr int kRowPx = 130;                        // staged pixels per operand row: x = -1 .. 128
constexpr int kFBytes = 8 * 2 * 128 * 16;          // one full-resolution raw tensor band: [8 rows][2 halves][128 px] float4
constexpr int kQBytes = 4 * 2 * 64 * 16;           // half resolution: [4 rows][2 halves][64 px] float4
constexpr int kOperBytes = 10 * 2 * kRowPx * 16;   // tf32 operand rows: cin 8: [2 planes][10 rows][130]; cin 16: [4][5][130] (ring)
constexpr int kNumBufs = 13;                       // F0..F4, Q0..Q7 (Q0-3 alias F3, Q4-7 alias F4)

// ---- shared memory carve-up (bytes from the 1024-aligned dynamic base) ----
constexpr int kOffF = 0;
constexpr int kOffOper = kOffF + 5 * kFBytes;                    // 163840
constexpr int kOffRec = kOffOper + kOperBytes;                   // 205440
constexpr int kOffStats = kOffRec + 2 * kClRecBytes;             // 219136
constexpr int kOffZeroB = kOffStats + kNumBufs * kCl * 8 * 4;    // 222464: a zero B operand (32 x 8 tf32) for the clearing MMAs
constexpr int kOffMisc = kOffZeroB + 1024;                       // 223488
constexpr int kSmemBytes = kOffMisc + 4096;

struct Misc {
    float part[kStageWarps][8];          // block reduction of the GroupNorm partial sums
    float gcoef[kStageWarps][32];        // per-warp copy of the layer's GroupNorm coefficients: ga[16], gb[16]
    uint64_t pass_bar[3];                // operand rows 4 p .. 4 p + 3 staged (16 warp arrivals)  staging warps -> MMA warp
    uint64_t free_bar[2];                // cin-16 ring: rows 0-3 / row 4 consumed (commit)         MMA warp -> staging warps
    uint64_t done_bar[2];                // output rows of phase A / B accumulated (commit) MMA warp -> epilogue
    uint64_t rec_bar[2];                 // layer record landed (bulk copy)
    uint64_t sync_bar[2];                // cluster-wide layer hand-over: 8 x 32 bytes of statistics (st.async complete_tx)
    uint32_t tmem;
};
static_assert(sizeof(Misc) <= 4096, "Misc does not fit its slot");
static_assert(kSmemBytes <= 227 * 1024, "cluster UNet kernel exceeds the shared memory of one SM");
static_assert(kClRecBytes % 16 == 0, "layer records are bulk-copied");

enum Kind { kConv = 0, kDownK = 1, kUpK = 2 };
struct LayerCfg { int8_t kind, cin, gn, res, in_a, in_b, res_a, res_b, out, half; };
enum Buf { F0 = 0, F1, F2, F3, F4, Q0, Q1, Q2, Q3, Q4, Q5, Q6, Q7 };

// Execution order of unet.py:315-340 with the buffer each tensor lives in (hs[] = skip stack):
//   F0 = hs0 (conv_in), F1 = hs1, F2 = hs2, Q0 = hs3, Q1 = hs4, Q2 = hs5; F3/F4/Q4.. = temporaries.
__constant__ LayerCfg c_layers[kClLayers] = {
    {kConv, 8, 1, kNone, F0, F0, F0, F0, F3, 0},    //  0 down.0.block.0 conv1
    {kConv, 8, 1, kIdent, F3, F3, F0, F0, F1, 0},   //  1                conv2 + x        -> hs1
    {kConv, 8, 1, kNone, F1, F1, F1, F1, F3, 0},    //  2 down.0.block.1 conv1
    {kConv, 8, 1, kIdent, F3, F3, F1, F1, F2, 0},   //  3                conv2 + x        -> hs2
    {kDownK, 8, 0, kNone, F2, F2, F2, F2, Q0, 1},   //  4 down.0.downsample               -> hs3
    {kConv, 8, 1, kNone, Q0, Q0, Q0, Q0, Q4, 1},    //  5 down.1.block.0 conv1
    {kConv, 8, 1, kIdent, Q4, Q4, Q0, Q0, Q1, 1},   //  6                conv2 + x        -> hs4
    {kConv, 8, 1, kNone, Q1, Q1, Q1, Q1, Q4, 1},    //  7 down.1.block.1 conv1
    {kConv, 8, 1, kIdent, Q4, Q4, Q1, Q1, Q2, 1},   //  8                conv2 + x        -> hs5
    {kConv, 8, 1, kNone, Q2, Q2, Q2, Q2, Q4, 1},    //  9 mid.block_1 conv1
    {kConv, 8, 1, kIdent, Q4, Q4, Q2, Q2, Q3, 1},   // 10             conv2 + x
    {kConv, 8, 1, kNone, Q3, Q3, Q3, Q3, Q4, 1},    // 11 mid.block_2 conv1
    {kConv, 8, 1, kIdent, Q4, Q4, Q3, Q3, Q5, 1},   // 12             conv2 + x
    {kConv, 16, 1, kNone, Q5, Q2, Q5, Q2, Q4, 1},   // 13 up.1.block.0 conv1 on cat(h, hs5)
    {kConv, 8, 1, kNin, Q4, Q4, Q5, Q2, Q6, 1},     // 14              conv2 + nin(cat)
    {kConv, 16, 1, kNone, Q6, Q1, Q6, Q1, Q4, 1},   // 15 up.1.block.1 conv1 on cat(h, hs4)
    {kConv, 8, 1, kNin, Q4, Q4, Q6, Q1, Q5, 1},     // 16              conv2 + nin(cat)
    {kConv, 16, 1, kNone, Q5, Q0, Q5, Q0, Q4, 1},   // 17 up.1.block.2 conv1 on cat(h, hs3)
    {kConv, 8, 1, kNin, Q4, Q4, Q5, Q0, Q6, 1},     // 18              conv2 + nin(cat)
    {kUpK, 8, 0, kNone, Q6, Q6, Q6, Q6, F3, 0},     // 19 up.1.upsample (nearest x2 + 3x3)
    {kConv, 16, 1, kNone, F3, F2, F3, F2, F4, 0},   // 20 up.0.block.0 conv1 on cat(h, hs2)
    {kConv, 8, 1, kNin, F4, F4, F3, F2, F2, 0},     // 21              conv2 + nin(cat)   (in place over hs2)
    {kConv, 16, 1, kNone, F2, F1, F2, F1, F4, 0},   // 22 up.0.block.1 conv1 on cat(h, hs1)
    {kConv, 8, 1, kNin, F4, F4, F2, F1, F3, 0},     // 23              conv2 + nin(cat)
    {kConv, 16, 1, kNone, F3, F0, F3, F0, F4, 0},   // 24 up.0.block.2 conv1 on cat(h, hs0)
    {kConv, 8, 1, kNin, F4, F4, F3, F0, F2, 0},     // 25              conv2 + nin(cat)   -> input of norm_out
};

__device__ __forceinline__ uint32_t buf_off(int id) {
    return id < 5 ? (uint32_t)(id * kFBytes)
                  : (id < 9 ? (uint32_t)(3 * kFBytes + (id - 5) * kQBytes) : (uint32_t)(4 * kFBytes + (id - 9) * kQBytes));
}

// ---- distributed shared memory ----
__device__ __forceinline__ uint32_t mapa(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ float4 ld_cluster4(uint32_t caddr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(caddr));
    return v;
}
__device__ __forceinline__ float4 lds4(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts4(uint32_t saddr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float lds1(uint32_t saddr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts1(uint32_t saddr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(saddr), "f"(v) : "memory"); }
__device__ __forceinline__ void stage_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kStageThreads) : "memory"); }   // staging warps only

// x * sigmoid(x) = h + h * tanh(h) with h = x / 2 already formed (the GroupNorm coefficients are stored pre-halved), two
// activations per MUFU: tanh.approx.f16x2 (|tanh| <= 1 in fp16: absolute error 2^-11, the tf32 operand grid).  The
// staging pass is MUFU bound (10.4 k activations per layer and CTA at 16 / clock, profiles/r02j_cluster_trace_v3.txt).
__device__ __forceinline__ void swish_half2(float &h0, float &h1) {
    const __half2 hh = __floats2half2_rn(h0, h1);
    uint32_t t;
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(t) : "r"(*reinterpret_cast<const uint32_t *>(&hh)));
    const float2 tf = __half22float2(*reinterpret_cast<const __half2 *>(&t));
    h0 = fmaf(h0, tf.x, h0);
    h1 = fmaf(h1, tf.y, h1);
}

struct Ctx {
    uint32_t smem;        // shared::cta address of the carve-up base
    uint32_t rank;        // CTA rank in the cluster = row band
    uint32_t ph_pass, ph_free, ph_done, ph_rec, ph_sync;   // mbarrier phase parities, one bit per barrier (uniform per CTA)
    uint32_t sync_n;      // cluster hand-overs so far (parity selects sync_bar)
    int tid, warp, lane;
    long long *trace;     // GC_CL_DEBUG & 32: per-layer clock64 timeline of CTA 0: [layer][16]
    int trace_row;
    int dbg;
};
#define GC_TRACE(c, k) do { if ((c).trace != nullptr && (c).tid == 0) (c).trace[(c).trace_row * 16 + (k)] = clock64(); } while (0)
#define MISC_ADDR(c, member) ((c).smem + kOffMisc + (uint32_t)offsetof(Misc, member))
constexpr uint32_t kTmem = 0u;   // the CTA owns all 512 columns (one CTA per SM): the allocation starts at column 0, checked at start
// (Four independent accumulator sets, one per row of a pass, were tried against the 70 cycles per MMA of
// profiles/r02n_cluster_trace_v3_1.txt and measured slower: the MMAs retire 70 cycles after the last issue -- the pipe is
// never backed up; the cost is the dependent uniform-datapath chain that builds each descriptor, profiles/r02o_*.)

__device__ __forceinline__ void wait_bit(uint32_t bar, uint32_t &bits, int k) {
    mbar_wait(bar, (bits >> k) & 1u);
    bits ^= 1u << k;
}

// ------------------------------------------------------------------------------------------------
// Cluster-wide hand-over between layers.  Producer side (end of a layer, staging warps): per-CTA partial GroupNorm sums of
// the tile just produced, block-reduced in a fixed order, pushed to the statistics slot `out_buf` of all 8 CTAs with
// st.async; every push completes 32 bytes on the destination's sync_bar.  Consumer side (start of the next layer): wait for
// 8 x 32 bytes = every CTA of the cluster has finished the previous layer (its raw rows are in its shared memory, and it
// no longer reads anything this layer overwrites), then re-arm the barrier for its next use.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void push_stats(Ctx &c, float (&q8)[8], int out_buf, float *gstats) {
    // halving butterfly: 4 + 2 + 1 exchanges leave value v = 4 b4 + 2 b3 + b2 (lane bits) in each lane, 2 more finish it
    {
        const bool hi = c.lane & 16;
        float k0 = hi ? q8[4] : q8[0], k1 = hi ? q8[5] : q8[1], k2 = hi ? q8[6] : q8[2], k3 = hi ? q8[7] : q8[3];
        const float s0 = hi ? q8[0] : q8[4], s1 = hi ? q8[1] : q8[5], s2 = hi ? q8[2] : q8[6], s3 = hi ? q8[3] : q8[7];
        k0 += __shfl_xor_sync(0xffffffffu, s0, 16); k1 += __shfl_xor_sync(0xffffffffu, s1, 16);
        k2 += __shfl_xor_sync(0xffffffffu, s2, 16); k3 += __shfl_xor_sync(0xffffffffu, s3, 16);
        const bool h8 = c.lane & 8;
        float m0 = h8 ? k2 : k0, m1 = h8 ? k3 : k1;
        const float t0 = h8 ? k0 : k2, t1 = h8 ? k1 : k3;
        m0 += __shfl_xor_sync(0xffffffffu, t0, 8); m1 += __shfl_xor_sync(0xffffffffu, t1, 8);
        const bool h4 = c.lane & 4;
        float r = h4 ? m1 : m0;
        const float u = h4 ? m0 : m1;
        r += __shfl_xor_sync(0xffffffffu, u, 4);
        r += __shfl_xor_sync(0xffffffffu, r, 2);
        r += __shfl_xor_sync(0xffffffffu, r, 1);
        if ((c.lane & 3) == 0) {
            const int v = ((c.lane >> 4) & 1) * 4 + ((c.lane >> 3) & 1) * 2 + ((c.lane >> 2) & 1);
            sts1(MISC_ADDR(c, part) + (uint32_t)(c.warp * 8 + v) * 4u, r);
        }
    }
    stage_bar();      // every staging warp has finished its epilogue: raw rows stored, partial sums in shared memory
    {   // all accumulators have been read: zero the 104 columns for the next layer (warp = lane quarter x 32-column slice)
        const int slice = c.warp >> 2;
        const uint32_t ta = kTmem + ((uint32_t)((c.warp & 3) * 32) << 16) + 32u * (uint32_t)slice;
        if (slice < 3) {
#pragma unroll
            for (int j = 0; j < 4; ++j) tmem_zero8(ta + 8u * j);
        } else {
            tmem_zero8(ta);
        }
    }
    if (c.warp == 0 && c.lane < 16) {
        const int peer = c.lane >> 1, half = c.lane & 1;
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int w = 0; w < kStageWarps; ++w) {
            const float4 p = lds4(MISC_ADDR(c, part) + (uint32_t)(w * 8 + half * 4) * 4u);
            t.x += p.x; t.y += p.y; t.z += p.z; t.w += p.w;
        }
        const uint32_t dst = c.smem + kOffStats + (uint32_t)(((out_buf * kCl) + (int)c.rank) * 8 + half * 4) * 4u;
        st_async4(mapa(dst, (uint32_t)peer), t, mapa(MISC_ADDR(c, sync_bar) + (c.sync_n & 1u) * 8u, (uint32_t)peer));
        if (gstats != nullptr && peer == 0) *reinterpret_cast<float4 *>(gstats + c.rank * 8 + half * 4) = t;
    }
    tmem_wait_st();
    tc_fence_before();   // ordered before the next layer's MMAs through this warp's arrival on its first pass barrier
    ++c.sync_n;
}

// Consumer side: wait for hand-over number n (pushes are numbered by c.sync_n).
__device__ __forceinline__ void sync_wait(Ctx &c, uint32_t n) {
    const int par = (int)(n & 1u);
    wait_bit(MISC_ADDR(c, sync_bar) + (uint32_t)par * 8u, c.ph_sync, par);
    // re-arm for hand-over n + 2: no peer can push it before this CTA has pushed n + 1, which every thread here precedes
    if (c.tid == 0) mbar_expect_tx(MISC_ADDR(c, sync_bar) + (uint32_t)par * 8u, kCl * 32u);
}

// GroupNorm(4 groups) coefficients of the layer input from the cluster-wide partial sums (fixed order -> every warp of
// every CTA computes identical values); each warp keeps its own copy: no block-wide barrier.  unet.py:36-37: eps 1e-6.
__device__ __forceinline__ void gn_coeffs_warp(const Ctx &c, const LayerCfg &L, uint32_t rec_saddr) {
    if (c.lane < L.cin) {
        const int ch = c.lane, cc = ch & 7;
        const uint32_t st = c.smem + kOffStats + (uint32_t)((ch < 8 ? L.in_a : L.in_b) * kCl * 8) * 4u;
        float s = 0.0f, ss = 0.0f;
        if (L.cin == 8) {
            const int p = cc >> 1;
#pragma unroll
            for (int r = 0; r < kCl; ++r) { s += lds1(st + (uint32_t)(r * 8 + 2 * p) * 4u); ss += lds1(st + (uint32_t)(r * 8 + 2 * p + 1) * 4u); }
        } else {
            const int p = (cc >> 2) * 2;
#pragma unroll
            for (int r = 0; r < kCl; ++r) {
                s += lds1(st + (uint32_t)(r * 8 + 2 * p) * 4u) + lds1(st + (uint32_t)(r * 8 + 2 * p + 2) * 4u);
                ss += lds1(st + (uint32_t)(r * 8 + 2 * p + 1) * 4u) + lds1(st + (uint32_t)(r * 8 + 2 * p + 3) * 4u);
            }
        }
        const float inv_cnt = 1.0f / ((L.half ? 32.0f * 64.0f : 64.0f * 128.0f) * (L.cin == 8 ? 2.0f : 4.0f));
        const float mean = s * inv_cnt;
        const float var = fmaxf(ss * inv_cnt - mean * mean, 0.0f);
        const float rstd = rsqrtf(var + 1e-6f);
        const float gamma = lds1(rec_saddr + (uint32_t)(kClRecGamma + ch) * 4u), beta = lds1(rec_saddr + (uint32_t)(kClRecBeta + ch) * 4u);
        const uint32_t g = MISC_ADDR(c, gcoef) + (uint32_t)(c.warp * 32) * 4u;
        sts1(g + (uint32_t)ch * 4u, 0.5f * (gamma * rstd));                       // pre-halved: see swish_half2
        sts1(g + (uint32_t)(16 + ch) * 4u, 0.5f * (beta - mean * gamma * rstd));
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// Staging side of a tensor-core layer.  Warp w owns pixel chunk w & 3 (32 pixels) of row 4 p + (w >> 2) in pass p: it reads
// the raw input (own band or the neighbour's halo row through DSMEM), applies GroupNorm + swish, writes the fp32 (tf32)
// pixel halves into the operand row and arrives on the row's barrier; the MMA warp issues the row as soon as its four
// chunks are in.  cin 16 layers keep 5 rows in flight (ring): row i >= 5 waits until the MMAs of row i - 5 have retired.
// ------------------------------------------------------------------------------------------------
template <int CG, bool HALF, bool UP, bool GN>
__device__ __forceinline__ void stage_layer(Ctx &c, const LayerCfg &L) {
    constexpr int PXW = HALF ? 64 : 128, R = HALF ? 4 : 8, NR = R + 2, HRES = HALF ? 32 : 64;
    constexpr int SPXW = UP ? 64 : PXW, SR = UP ? 4 : R;             // source tensor geometry
    constexpr int PROWS = CG == 1 ? 10 : 5;                          // slot rows per operand plane
    constexpr int NPASS = (NR + 3) / 4;
    const int chunk = c.warp & 3, rsel = c.warp >> 2;
    const int y0 = (int)c.rank * R;
    const int px = chunk * 32 + c.lane;                              // interior pixel of this thread (operand column px + 1)
    const bool px_ok = px < PXW;
    float4 ga[CG][2], gb[CG][2];
    if (GN) {
        const uint32_t g = MISC_ADDR(c, gcoef) + (uint32_t)(c.warp * 32) * 4u;
#pragma unroll
        for (int cg = 0; cg < CG; ++cg) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                ga[cg][h] = lds4(g + (uint32_t)(cg * 8 + h * 4) * 4u);
                gb[cg][h] = lds4(g + (uint32_t)(16 + cg * 8 + h * 4) * 4u);
            }
        }
    }
    auto row_valid = [&](int i) { const int gy = y0 - 1 + i; return i < NR && gy >= 0 && gy < HRES; };
    auto load_row = [&](int i, float4 (&v)[CG][2]) {
#pragma unroll
        for (int cg = 0; cg < CG; ++cg) v[cg][0] = v[cg][1] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!row_valid(i) || !px_ok) return;
        const int gy = y0 - 1 + i;
        const int sx = UP ? (px >> 1) : px;
        int sy = UP ? ((gy >> 1) - (int)c.rank * SR) : (i - 1);       // source row relative to this CTA's band
        uint32_t srank = c.rank;
        if (sy < 0) { srank = c.rank - 1; sy += SR; } else if (sy >= SR) { srank = c.rank + 1; sy -= SR; }
        // own band: plain LDS.  ld.shared::cluster is a ~20 B/cycle path even for the CTA's own memory (measured: 950 cycles
        // per 16 KB pass, profiles/r02m_cluster_trace.txt), so only the two halo rows go through it
#pragma unroll
        for (int cg = 0; cg < CG; ++cg) {
            const uint32_t a = c.smem + kOffF + buf_off(cg == 0 ? L.in_a : L.in_b) + (uint32_t)((sy * 2) * SPXW + sx) * 16u;
            if (srank == c.rank) {                                    // warp-uniform
                v[cg][0] = lds4(a);
                v[cg][1] = lds4(a + SPXW * 16u);
            } else {
                const uint32_t r = mapa(a, srank);
                v[cg][0] = ld_cluster4(r);
                v[cg][1] = ld_cluster4(r + SPXW * 16u);
            }
        }
    };
    // Row at a time, the next row's loads in flight while the current one is activated and stored.  (Loading and
    // activating all three rows first was measured slower, 331 vs 303 us per step: profiles/r02q_cluster_trace.txt.)
#define GC_TRACE2(k) do { if (c.trace != nullptr && c.tid == 0) c.trace[(kClLayers + c.trace_row) * 16 + (k)] = clock64(); } while (0)
    float4 cur[CG][2], nxt[CG][2];
    GC_TRACE2(0);
    load_row(rsel, cur);
#pragma unroll
    for (int p = 0; p < NPASS; ++p) {
        const int i = 4 * p + rsel;
        if (p + 1 < NPASS) load_row(i + 4, nxt);
        // cin-16 ring: rows 5-7 reuse the slots of rows 0-2 (MMAs of pass 0 retired), rows 8-9 those of rows 3-4
        if (CG == 2 && p >= 1) wait_bit(MISC_ADDR(c, free_bar) + (uint32_t)(p - 1) * 8u, c.ph_free, p - 1);
        if (row_valid(i) && px_ok) {                                  // row validity is warp-uniform
            const int slot = CG == 1 ? i : i % 5;
#pragma unroll
            for (int cg = 0; cg < CG; ++cg) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float4 u = cur[cg][h];
                    if (GN) {   // ga / gb carry the factor 1/2 of x sigmoid(x) = h + h tanh(h), h = x / 2
                        u.x = fmaf(u.x, ga[cg][h].x, gb[cg][h].x); u.y = fmaf(u.y, ga[cg][h].y, gb[cg][h].y);
                        u.z = fmaf(u.z, ga[cg][h].z, gb[cg][h].z); u.w = fmaf(u.w, ga[cg][h].w, gb[cg][h].w);
                        swish_half2(u.x, u.y);
                        swish_half2(u.z, u.w);
                    }
                    const uint32_t o = c.smem + kOffOper + (uint32_t)(((cg * 2 + h) * PROWS + slot) * kRowPx) * 16u;
                    sts4(o + (uint32_t)(px + 1) * 16u, u);
                    // x halo columns (padding applies after the activation): pixel -1 and pixel PXW
                    if (px == 0) sts4(o, make_float4(0.f, 0.f, 0.f, 0.f));
                    if (px == PXW - 1) sts4(o + (uint32_t)(PXW + 1) * 16u, make_float4(0.f, 0.f, 0.f, 0.f));
                }
            }
        }
        fence_async_smem();      // generic-proxy stores -> async proxy (tensor core)
        __syncwarp();
        if (c.lane == 0) mbar_arrive(MISC_ADDR(c, pass_bar) + (uint32_t)p * 8u);
        GC_TRACE2(1 + p);
        if (p + 1 < NPASS) {
#pragma unroll
            for (int cg = 0; cg < CG; ++cg) { cur[cg][0] = nxt[cg][0]; cur[cg][1] = nxt[cg][1]; }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// MMA warp: one elected lane, per layer: clear the accumulator columns (D = A * 0), then per staged row and channel group
// three MMAs (taps kx) of M = 128, N = 32, K = 8 (tf32) into TMEM columns 8 i .. 8 i + 31.
// ------------------------------------------------------------------------------------------------
template <int CG, bool HALF>
__device__ __forceinline__ void mma_layer(Ctx &c, uint32_t rec_saddr) {
    constexpr int R = HALF ? 4 : 8, NR = R + 2, HRES = HALF ? 32 : 64, NRA = R / 2 + 2;
    constexpr int PROWS = CG == 1 ? 10 : 5, NPASS = (NR + 3) / 4;
    constexpr uint32_t kPlane = PROWS * kRowPx * 16u;
    constexpr uint32_t idesc = make_idesc_tf32(128, 32);
    const int y0 = (int)c.rank * R;
    const uint64_t a_base = make_desc(c.smem + kOffOper, kPlane, 128u);
    const uint64_t b_base = make_desc(rec_saddr, 512u, 128u);
    // fully unrolled: every row index is a compile-time constant, so each descriptor is the base plus an immediate
#pragma unroll
    for (int p = 0; p < NPASS; ++p) {
        wait_bit(MISC_ADDR(c, pass_bar) + (uint32_t)p * 8u, c.ph_pass, p);   // one wait per pass: a try_wait costs ~100 cycles
        fence_async_smem();
        tc_fence_after();
        if (c.trace != nullptr) c.trace[c.trace_row * 16 + 5 + p] = clock64();
        // descriptors = loop-invariant base + small offset (one independent 64-bit add each: the address field cannot
        // carry, everything lives below 256 KB); a chain of mask / shift / or per MMA costs ~60 cycles on the uniform pipe
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int i = 4 * p + r;
            const int gy = y0 - 1 + i;
            if (i < NR && gy >= 0 && gy < HRES) {
                const int slot = CG == 1 ? i : i % 5;
#pragma unroll
                for (int cg = 0; cg < CG; ++cg) {
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)   // +1 in the address field = one 16-byte pixel; B: 2048 B per kx, 1024 B per group
                        mma_tf32(kTmem + 8u * i, a_base + (uint64_t)(cg * 2 * (kPlane / 16u) + slot * kRowPx + kx),
                                 b_base + (uint64_t)(kx * 128 + cg * 64), idesc, 1u);
                }
            }
        }
        if (CG == 2 && NPASS == 3 && p == 1) mma_commit(MISC_ADDR(c, free_bar) + 8u);      // rows 3, 4 retired: slots free for rows 8, 9
        if ((NRA - 1) / 4 == p) mma_commit(MISC_ADDR(c, done_bar));                         // rows 0 .. NRA-1 issued
        if (CG == 2 && p == 0) mma_commit(MISC_ADDR(c, free_bar));                          // slots 0-2 free for rows 5-7
    }
    mma_commit(MISC_ADDR(c, done_bar) + 8u);
    if (c.trace != nullptr) {   // debug: when do the accumulators actually complete?
        c.trace[c.trace_row * 16 + 8] = clock64();
        mbar_wait(MISC_ADDR(c, done_bar) + 8u, (c.ph_done >> 1) & 1u);
        c.ph_done ^= 2u;
        c.trace[c.trace_row * 16 + 10] = clock64();
    }
}

// ------------------------------------------------------------------------------------------------
// Epilogue (staging warps), phase by phase: thread = pixel x of one output row; bias, residual / nin_shortcut, raw output
// into this CTA's band, GroupNorm partial sums.
// ------------------------------------------------------------------------------------------------
template <bool HALF>
__device__ __forceinline__ void epilogue_layer(Ctx &c, const LayerCfg &L, uint32_t rec_saddr, float *gout, float (&q8)[8]) {
    constexpr int PXW = HALF ? 64 : 128, R = HALF ? 4 : 8;
    const int y0 = (int)c.rank * R;
    const int q = c.warp & 3, hsel = c.warp >> 2;      // lane quarter of TMEM, row within the phase
    const int px = q * 32 + c.lane;
    float bias[8];
    {
        const float4 b0 = lds4(rec_saddr + kClRecBias * 4u), b1 = lds4(rec_saddr + kClRecBias * 4u + 16u);
        bias[0] = b0.x; bias[1] = b0.y; bias[2] = b0.z; bias[3] = b0.w; bias[4] = b1.x; bias[5] = b1.y; bias[6] = b1.z; bias[7] = b1.w;
    }
    const uint32_t out_base = c.smem + kOffF + buf_off(L.out);
    const uint32_t ra_base = c.smem + kOffF + buf_off(L.res_a), rb_base = c.smem + kOffF + buf_off(L.res_b);
#pragma unroll
    for (int ph = 0; ph < 2; ++ph) {
        wait_bit(MISC_ADDR(c, done_bar) + (uint32_t)ph * 8u, c.ph_done, ph);
        tc_fence_after();
        GC_TRACE(c, 9 + 2 * ph);
        if (px >= PXW || hsel >= R / 2) continue;      // warp-uniform (half resolution: 4 of the 16 warps work)
        const int r0 = ph * (R / 2) + hsel;
        float a[8];
        tmem_ld8(kTmem + ((uint32_t)(q * 32) << 16) + 8u * (r0 + 2), a);
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] += bias[i];
        const uint32_t poff = (uint32_t)((r0 * 2) * PXW + px) * 16u;
        if (L.res != kNone) {
            const float4 a0 = lds4(ra_base + poff), a1 = lds4(ra_base + poff + PXW * 16u);
            if (L.res == kIdent) {
                a[0] += a0.x; a[1] += a0.y; a[2] += a0.z; a[3] += a0.w;
                a[4] += a1.x; a[5] += a1.y; a[6] += a1.z; a[7] += a1.w;
            } else {
                const float4 b0 = lds4(rb_base + poff), b1 = lds4(rb_base + poff + PXW * 16u);
                const float xr[16] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w,
                                      b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                const float4 n0 = lds4(rec_saddr + kClRecNinB * 4u), n1 = lds4(rec_saddr + kClRecNinB * 4u + 16u);
                float sh[8] = {n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, n1.z, n1.w};
#pragma unroll
                for (int ci = 0; ci < 16; ++ci) {
                    const float4 w0 = lds4(rec_saddr + (uint32_t)(kClRecNinW + ci * 8) * 4u);
                    const float4 w1 = lds4(rec_saddr + (uint32_t)(kClRecNinW + ci * 8 + 4) * 4u);
                    sh[0] = fmaf(xr[ci], w0.x, sh[0]); sh[1] = fmaf(xr[ci], w0.y, sh[1]);
                    sh[2] = fmaf(xr[ci], w0.z, sh[2]); sh[3] = fmaf(xr[ci], w0.w, sh[3]);
                    sh[4] = fmaf(xr[ci], w1.x, sh[4]); sh[5] = fmaf(xr[ci], w1.y, sh[5]);
                    sh[6] = fmaf(xr[ci], w1.z, sh[6]); sh[7] = fmaf(xr[ci], w1.w, sh[7]);
                }
#pragma unroll
                for (int o = 0; o < 8; ++o) a[o] += sh[o];
            }
        }
        const float4 o0 = make_float4(a[0], a[1], a[2], a[3]), o1 = make_float4(a[4], a[5], a[6], a[7]);
        sts4(out_base + poff, o0);
        sts4(out_base + poff + PXW * 16u, o1);
        if (gout != nullptr) {   // last layer of the unfused variant: the raw tensor also goes to global memory (NHWC8)
            float4 *dst = reinterpret_cast<float4 *>(gout + ((size_t)(y0 + r0) * PXW + px) * 8);
            dst[0] = o0;
            dst[1] = o1;
        }
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            q8[2 * p] += a[2 * p] + a[2 * p + 1];
            q8[2 * p + 1] += a[2 * p] * a[2 * p] + a[2 * p + 1] * a[2 * p + 1];
        }
    }
    tc_fence_before();
}

// down.0.downsample (unet.py:59-78): pad (0,1,0,1) + 3x3 stride 2, no GroupNorm, on CUDA cores (thread = output pixel).
__device__ __forceinline__ void down_layer(Ctx &c, const LayerCfg &L, uint32_t rec_saddr, float (&q8)[8]) {
    const bool act = c.tid < 256;                      // 4 rows x 64 output pixels; the other warps only join the reduction
    if (!act) return;
    const int r = (c.tid >> 6) & 3, ox = c.tid & 63;
    float acc[8];
    {
        const float4 b0 = lds4(rec_saddr + kClRecBias * 4u), b1 = lds4(rec_saddr + kClRecBias * 4u + 16u);
        acc[0] = b0.x; acc[1] = b0.y; acc[2] = b0.z; acc[3] = b0.w; acc[4] = b1.x; acc[5] = b1.y; acc[6] = b1.z; acc[7] = b1.w;
    }
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        int sy = 2 * r + ky;                              // full-resolution row relative to this CTA's band (0..8)
        uint32_t srank = c.rank;
        if (sy >= 8) { srank = c.rank + 1; sy -= 8; }
        const bool row_ok = srank < (uint32_t)kCl;        // row 64 is the zero padding
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int sx = 2 * ox + kx;
            if (!row_ok || sx >= 128) continue;
            const uint32_t a = c.smem + kOffF + buf_off(L.in_a) + (uint32_t)((sy * 2) * 128 + sx) * 16u;
            float4 v0, v1;
            if (srank == c.rank) { v0 = lds4(a); v1 = lds4(a + 128u * 16u); }
            else { const uint32_t ra = mapa(a, srank); v0 = ld_cluster4(ra); v1 = ld_cluster4(ra + 128u * 16u); }
            const float vv[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
            const uint32_t w = rec_saddr + (uint32_t)((ky * 3 + kx) * 64) * 4u;   // [tap][cin][cout]
#pragma unroll
            for (int ci = 0; ci < 8; ++ci) {
                const float4 w0 = lds4(w + (uint32_t)(ci * 8) * 4u), w1 = lds4(w + (uint32_t)(ci * 8 + 4) * 4u);
                acc[0] = fmaf(vv[ci], w0.x, acc[0]); acc[1] = fmaf(vv[ci], w0.y, acc[1]);
                acc[2] = fmaf(vv[ci], w0.z, acc[2]); acc[3] = fmaf(vv[ci], w0.w, acc[3]);
                acc[4] = fmaf(vv[ci], w1.x, acc[4]); acc[5] = fmaf(vv[ci], w1.y, acc[5]);
                acc[6] = fmaf(vv[ci], w1.z, acc[6]); acc[7] = fmaf(vv[ci], w1.w, acc[7]);
            }
        }
    }
    const uint32_t poff = (uint32_t)((r * 2) * 64 + ox) * 16u, out_base = c.smem + kOffF + buf_off(L.out);
    sts4(out_base + poff, make_float4(acc[0], acc[1], acc[2], acc[3]));
    sts4(out_base + poff + 64u * 16u, make_float4(acc[4], acc[5], acc[6], acc[7]));
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        q8[2 * p] = acc[2 * p] + acc[2 * p + 1];
        q8[2 * p + 1] = acc[2 * p] * acc[2 * p] + acc[2 * p + 1] * acc[2 * p + 1];
    }
}

// The 26 middle layers of one UNet evaluation.  rec_g: this step's layer records in global memory.  On entry the input
// tensor (F0) and its statistics have been pushed (hand-over c.sync_n - 1 is in flight).
__device__ __forceinline__ void middle_layers(Ctx &c, const float *rec_g, float *gout, float *gstats) {
    if (c.tid == 32) {   // records 0 and 1; record l + 2 follows at the end of layer l (a full layer ahead of its use)
        bulk_load(c.smem + kOffRec, rec_g, kClRecBytes, MISC_ADDR(c, rec_bar));
        bulk_load(c.smem + kOffRec + kClRecBytes, rec_g + kClRecFloats, kClRecBytes, MISC_ADDR(c, rec_bar) + 8u);
    }
#pragma unroll 1
    for (int l = 0; l < kClLayers; ++l) {
        const LayerCfg L = c_layers[l];
        const int rb = l & 1;
        c.trace_row = l;
        GC_TRACE(c, 0);
        wait_bit(MISC_ADDR(c, rec_bar) + (uint32_t)rb * 8u, c.ph_rec, rb);
        GC_TRACE(c, 1);
        const uint32_t rec_saddr = c.smem + kOffRec + (uint32_t)(rb * kClRecBytes);
        if (c.warp == kMmaWarp) {
            // ---- MMA warp ----
            // its phase bookkeeping of the hand-over / done barriers is not needed; row and free bits are tracked by the
            // elected lane only (the same lane is elected every time: the warp stays converged)
            if (L.kind != kDownK && elect_one()) {
                if (L.half) {
                    if (L.cin == 8) mma_layer<1, true>(c, rec_saddr); else mma_layer<2, true>(c, rec_saddr);
                } else {
                    if (L.cin == 8) mma_layer<1, false>(c, rec_saddr); else mma_layer<2, false>(c, rec_saddr);
                }
            }
            __syncwarp();
            ++c.sync_n;
            continue;
        }
        // ---- staging / epilogue warps ----
        sync_wait(c, c.sync_n - 1);       // the producers of this layer's inputs are done, everywhere in the cluster
        GC_TRACE(c, 2);
        if (L.gn) gn_coeffs_warp(c, L, rec_saddr);
        GC_TRACE(c, 3);
        float q8[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) q8[i] = 0.0f;
        const bool last = l == kClLayers - 1;
        if (L.kind == kDownK) {
            down_layer(c, L, rec_saddr, q8);
        } else {
            if (L.kind == kUpK) stage_layer<1, false, true, false>(c, L);
            else if (L.half) { if (L.cin == 8) stage_layer<1, true, false, true>(c, L); else stage_layer<2, true, false, true>(c, L); }
            else { if (L.cin == 8) stage_layer<1, false, false, true>(c, L); else stage_layer<2, false, false, true>(c, L); }
            GC_TRACE(c, 4);
            if (L.half) epilogue_layer<true>(c, L, rec_saddr, nullptr, q8);
            else epilogue_layer<false>(c, L, rec_saddr, last ? gout : nullptr, q8);
        }
        GC_TRACE(c, 12);
        push_stats(c, q8, L.out, last ? gstats : nullptr);
        // every staging warp is past this layer's epilogue and its MMAs have retired: the record buffer is free
        if (c.tid == 32 && l + 2 < kClLayers)
            bulk_load(c.smem + kOffRec + (uint32_t)(rb * kClRecBytes), rec_g + (size_t)(l + 2) * kClRecFloats, kClRecBytes,
                      MISC_ADDR(c, rec_bar) + (uint32_t)rb * 8u);
        GC_TRACE(c, 13);
    }
}

// ------------------------------------------------------------------------------------------------
// Unfused variant: h0 = conv_in output (NHWC8, global) -> 26 layers -> input of norm_out (NHWC8, global) + its
// per-band GroupNorm partial sums [A][8 bands][8] for k_conv_out_tc.  One cluster per agent (grid-stride).
// ------------------------------------------------------------------------------------------------
__global__ void __cluster_dims__(kCl, 1, 1) __launch_bounds__(kThreads, 1)
k_unet_middle_cluster(const float *__restrict__ h0, const float *__restrict__ rec_g, float *__restrict__ out,
                      float *__restrict__ stats_out, int n_agents, int dbg, long long *trace) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    Ctx c;
    c.smem = smem_u32(smem_raw);
    c.tid = threadIdx.x;
    c.warp = __shfl_sync(0xffffffffu, c.tid >> 5, 0);   // warp-uniform by construction (role dispatch branches on it)
    c.lane = c.tid & 31;
    c.rank = blockIdx.x % kCl;
    c.trace = (blockIdx.x == 1 && (dbg & 32)) ? trace : nullptr;
    c.trace_row = 0;
    c.dbg = dbg;
    c.ph_pass = c.ph_free = c.ph_done = c.ph_rec = c.ph_sync = 0u;
    c.sync_n = 0u;
    const int n_clusters = gridDim.x / kCl, cluster_id = blockIdx.x / kCl;
    Misc *misc = reinterpret_cast<Misc *>(smem_raw + kOffMisc);

    if (c.warp == 0) tmem_alloc<512>(&misc->tmem);
    if (c.tid == 32) {
        for (int i = 0; i < 3; ++i) mbar_init(MISC_ADDR(c, pass_bar) + 8u * i, kStageWarps);
        for (int i = 0; i < 2; ++i) mbar_init(MISC_ADDR(c, free_bar) + 8u * i, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(MISC_ADDR(c, done_bar) + 8u * i, 1); mbar_init(MISC_ADDR(c, rec_bar) + 8u * i, 1);
            mbar_init(MISC_ADDR(c, sync_bar) + 8u * i, 1);
        }
        mbar_init_fence();
        mbar_expect_tx(MISC_ADDR(c, sync_bar), kCl * 32u);          // hand-overs 0 and 1
        mbar_expect_tx(MISC_ADDR(c, sync_bar) + 8u, kCl * 32u);
    }
    // operand rows, the zero B operand: finite values everywhere (the clearing MMAs multiply whatever is there by zero)
    for (int i = c.tid; i < (kOperBytes + 1024) / 16; i += kThreads)
        sts4(c.smem + (i < kOperBytes / 16 ? kOffOper + i * 16 : kOffZeroB + (i - kOperBytes / 16) * 16), make_float4(0.f, 0.f, 0.f, 0.f));
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (misc->tmem != kTmem) __trap();                  // the whole tensor memory of the SM: the allocation starts at column 0
    cluster_arrive();                                   // barriers initialised everywhere before anyone pushes
    cluster_wait();

    for (int agent = cluster_id; agent < n_agents; agent += n_clusters) {
        if (c.warp != kMmaWarp) {
            // ---- load this CTA's band of h0 into F0 and publish its GroupNorm partial sums ----
            const int q = c.warp & 3, hsel = c.warp >> 2, px = q * 32 + c.lane, r0 = hsel * 2;
            float q8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) q8[i] = 0.0f;
            float4 v[2][2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const float4 *src = reinterpret_cast<const float4 *>(h0 + (((size_t)agent * 64 + c.rank * 8 + r0 + r) * 128 + px) * 8);
                v[r][0] = __ldg(src);
                v[r][1] = __ldg(src + 1);
            }
            // the previous agent's layers read F0 as a halo until their layer 24; this CTA has seen the hand-over of layer 24
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const uint32_t poff = (uint32_t)(((r0 + r) * 2) * 128 + px) * 16u;
                sts4(c.smem + kOffF + buf_off(F0) + poff, v[r][0]);
                sts4(c.smem + kOffF + buf_off(F0) + poff + 128u * 16u, v[r][1]);
                const float a[8] = {v[r][0].x, v[r][0].y, v[r][0].z, v[r][0].w, v[r][1].x, v[r][1].y, v[r][1].z, v[r][1].w};
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    q8[2 * p] += a[2 * p] + a[2 * p + 1];
                    q8[2 * p + 1] += a[2 * p] * a[2 * p] + a[2 * p + 1] * a[2 * p + 1];
                }
            }
            push_stats(c, q8, F0, nullptr);
        } else {
            ++c.sync_n;
        }
        middle_layers(c, rec_g, out + (size_t)agent * 64 * 128 * 8, stats_out + (size_t)agent * kCl * 8);
        // the hand-over of layer 25 must be consumed before the next agent's F0 load: a neighbour reads this CTA's F0 / F2
        // rows until it has finished layer 24 / 25
        // (every hand-over is waited for exactly once: this is the wait of layer 25's)
        if (c.warp != kMmaWarp) sync_wait(c, c.sync_n - 1);
    }
    tc_fence_before();
    __syncthreads();
    cluster_arrive();                                   // no CTA exits while a peer may still push into its shared memory
    cluster_wait();
    if (c.warp == 0) tmem_free<512>(kTmem);
}

}  // namespace cl

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool unet_cluster_eligible(int C, int H, int W) {
    (void)C;
    return H == 64 && W == 128;
}

static int cluster_grid(const void *kernel, size_t smem, int n_agents, int *n_clusters) {
    static int cached = -1;
    if (cached < 0) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { (void)cudaGetLastError(); set_error("unet cluster kernel: cudaFuncSetAttribute failed (%d)", (int)e); return (int)e; }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(kCl, 1, 1);
        cfg.blockDim = dim3(cl::kThreads, 1, 1);
        cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kCl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int n = 0;
        e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
        if (e != cudaSuccess || n <= 0) { (void)cudaGetLastError(); set_error("unet cluster kernel: no active cluster fits (%d)", (int)e); return e != cudaSuccess ? (int)e : GC_EUNSUPPORTED; }
        cached = n;
    }
    *n_clusters = n_agents < cached ? n_agents : cached;
    return GC_OK;
}

int unet_middle_cluster(cudaStream_t st, int A, const float *h0, const float *rec_dev, float *out, float *stats_out) {
    int n_clusters = 0;
    if (int rc = cluster_grid((const void *)cl::k_unet_middle_cluster, cl::kSmemBytes, A, &n_clusters)) return rc;
    static int dbg = -1;
    if (dbg < 0) { const char *e = getenv("GC_CL_DEBUG"); dbg = e ? atoi(e) : 0; }
    static long long *trace = nullptr;
    if ((dbg & 32) && trace == nullptr) {
        cudaMalloc(&trace, 2 * kClLayers * 16 * sizeof(long long));
        cudaMemset(trace, 0, 2 * kClLayers * 16 * sizeof(long long));
    }
    cl::k_unet_middle_cluster<<<n_clusters * kCl, cl::kThreads, cl::kSmemBytes, st>>>(h0, rec_dev, out, stats_out, A, dbg, trace);
    if (trace != nullptr) {   // debug only: dump the timeline of the last agent CTA 0 processed
        cudaStreamSynchronize(st);
        long long h[2 * kClLayers * 16];
        cudaMemcpy(h, trace, sizeof(h), cudaMemcpyDeviceToHost);
        for (int l = 0; l < kClLayers; ++l) {
            fprintf(stderr, "trace layer %2d:", l);
            for (int k = 1; k < 16; ++k) fprintf(stderr, " %lld", h[l * 16 + k] ? h[l * 16 + k] - h[l * 16] : -1);
            fprintf(stderr, "  | stage:");
            for (int k = 0; k < 14; ++k) fprintf(stderr, " %lld", h[(kClLayers + l) * 16 + k] ? h[(kClLayers + l) * 16 + k] - h[l * 16] : -1);
            fprintf(stderr, "\n");
        }
    }
    GC_LAUNCH_CHECK("k_unet_middle_cluster");
    return GC_OK;
}

}  // namespace gc
