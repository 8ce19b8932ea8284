// Tiled, TMA-staged warp + regroup + Max/Att fusion for sm_100a (the fast path of gc_warp_fuse).
//
// Same operator and numerics as warp_fuse.cu (reference: fusion_in_one.py:53-151,
// torch_transformation_utils.py:323-332); this file is about data movement.  Round-1a ncu of the first
// TMA version (one 32x32 tile, one channel per barrier round trip, AttFusion in two passes) showed 61 warp
// instructions per sampled warp-element and 1.55x algorithmic DRAM traffic: issue bound and re-reading.
// This version:
//
//   * CTA = TW x TH output pixels (16 x 8) of one frame, G thread groups per pixel (each group owns every
//     G-th channel) + one producer warp.  The bilinear taps are computed once per (pixel, agent) -- group g
//     takes agents g, g+G, .. -- from float64 base-grid coordinates computed once per tile row/column, and
//     exchanged through shared memory.
//   * The source footprint of the tile under agent j's affine map fits a BW x BH box for any isometry.
//     ONE 3-D TMA copy per (agent, stage) brings that box for CHS consecutive channel planes
//     (cp.async.bulk.tensor.3d, out-of-bounds elements zero-filled == grid_sample padding_mode='zeros';
//     an agent that is out of view is simply an all-zero box).  When the ego's taps are exactly the identity
//     (theta = I) it uses a tight TW x TH box instead: no halo.
//   * full/empty mbarrier ring between the producer warp and the consumer warps.
//   * Hot loop (fast_loop): compile-time agent count, every agent's weights + ONE shared-memory byte address
//     in registers, channels of a stage unrolled: a sample is 4 LDS with immediate offsets + 4 FMA.
//   * AttFusion in ONE pass over HBM: sampled vectors of the non-identity agents are parked in shared
//     memory ([agent][channel][pixel], conflict free) while the ego-row scores accumulate; after the
//     softmax the weighted sum is formed from shared memory (the identity agent is re-read from L2).
//     If the park does not fit (large C x N) the kernel degrades to two passes through the ring.
//   * Affine maps that are not near-isometries can overflow the box: such an agent is detected per tile
//     and the tile runs generic_loop, which samples that agent straight from global memory.
//
// Requirements checked by the host: W % 4 == 0 and 16-byte aligned base (TMA global strides), at most
// kTileMaxN agents per frame.  Otherwise gc_warp_fuse uses the gather kernels of warp_fuse.cu.
#include <stdlib.h>

#include "ptx.cuh"
#include "warp_common.cuh"

namespace gc {

using namespace ptx;

constexpr int kTileMaxN = 5;
constexpr int kMaxStages = 4;
constexpr int kDynSmemBytes = 224 * 1024;

constexpr int isqrt_ceil(int v) {
    int r = 0;
    while (r * r < v) ++r;
    return r;
}

template <int TW_, int TH_, int G_, int KC_, int CTAS_ = 1>
struct TileCfg {
    static constexpr int TW = TW_, TH = TH_, G = G_, KC = KC_, CTAS = CTAS_;
    static constexpr int kSmemBytes = CTAS == 1 ? kDynSmemBytes : 110 * 1024;   // dynamic shared memory per CTA
    static constexpr int P = TW * TH;                  // pixels per tile
    static constexpr int CHS = G * KC;                 // channel planes per pipeline stage
    static constexpr int kConsumers = P * G;
    static constexpr int kThreads = kConsumers + 32;   // + producer warp
    // x0 = floor(ix) spans at most ceil(diagonal) + 1 values over the tile, + 1 for the x0+1 tap
    static constexpr int EXT = isqrt_ceil((TW - 1) * (TW - 1) + (TH - 1) * (TH - 1)) + 2;
    static constexpr int BW = (EXT + 3 + 3) & ~3;      // + up to 3 columns: box x origin floored to 16 bytes
    static constexpr int BH = EXT;
    static constexpr int BOXF = BW * BH;
    // scratch = max(tap exchange [N][6][P], score reduction [G][N][P]) floats
    static constexpr int kScratch = kTileMaxN * P * (G > 6 ? G : 6);
    static_assert(P % 32 == 0 && TW % 4 == 0, "tile rows must be 16-byte multiples, groups warp aligned");
    static_assert((CHS * BOXF * 4) % 128 == 0 && (CHS * P * 4) % 128 == 0, "TMA destinations are 128-byte aligned");
    static_assert((kScratch * 4) % 128 == 0, "ring must stay 128-byte aligned");
    static_assert(kThreads <= 1024, "block too large");
    static_assert((P & (P - 1)) == 0, "P must be a power of two");
};

struct TapS {
    float w_nw, w_ne, w_sw, w_se;
    int x0, y0;   // clamped to [-2, W] / [-2, H]: anything clamped has both taps out of bounds (zero)
};

__device__ __forceinline__ TapS make_tap_xy(const double *__restrict__ th, double xs, double ys, int H, int W) {
    const float gx = (float)(xs * th[0] + ys * th[1] + th[2]);
    const float gy = (float)(xs * th[3] + ys * th[4] + th[5]);
    const float ix = __fmaf_rn(gx + 1.0f, (float)W, -1.0f) * 0.5f;
    const float iy = __fmaf_rn(gy + 1.0f, (float)H, -1.0f) * 0.5f;
    const float fx = floorf(ix), fy = floorf(iy);
    const float ex = (fx + 1.0f) - ix, wx = ix - fx;
    const float sy = (fy + 1.0f) - iy, ny_ = iy - fy;
    TapS t;
    t.w_nw = ex * sy; t.w_ne = wx * sy; t.w_sw = ex * ny_; t.w_se = wx * ny_;
    t.x0 = (int)fminf(fmaxf(fx, -2.0f), (float)W);
    t.y0 = (int)fminf(fmaxf(fy, -2.0f), (float)H);
    if (!(ix == ix) || !(iy == iy)) {   // NaN transform: contributes zeros
        t.w_nw = t.w_ne = t.w_sw = t.w_se = 0.0f;
        t.x0 = t.y0 = -2;
    }
    return t;
}

enum AgentPath { kPathIdent = 1, kPathBox = 2, kPathGather = 3 };

// everything the consumer loops need, by value
struct TileCtx {
    uint32_t ring_addr, stage_bytes, park_addr, full_addr, empty_addr;
    int stages, chunks, C, n;
    bool park_mode, active;
    int lane, g, p;
    float sqrt_c;
    float *scratch;
    float *dst;            // out + (first output plane of the CTA + g) * plane + pix
    const float *src_pix;  // feat + a0 * C * plane + pix
    size_t plane, pix;
};

// softmax over the ego-row scores after combining the G channel groups in a fixed order
// (score / sqrt(C), fusion_in_one.py:42-43).  score[] holds the attention weights on return.
template <int N, class Cfg>
__device__ __forceinline__ void att_softmax(const TileCtx &x, float (&score)[N]) {
    constexpr int G = Cfg::G, P = Cfg::P;
#pragma unroll
    for (int j = 0; j < N; ++j) x.scratch[(x.g * N + j) * P + x.p] = score[j];
    consumer_sync<Cfg::kConsumers>();
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        float t = 0.0f;
#pragma unroll
        for (int gg = 0; gg < G; ++gg) t += x.scratch[(gg * N + j) * P + x.p];
        score[j] = __fdiv_rn(t, x.sqrt_c);
        mx = fmaxf(mx, score[j]);
    }
    float den = 0.0f;
#pragma unroll
    for (int j = 0; j < N; ++j) { score[j] = expf(score[j] - mx); den += score[j]; }
#pragma unroll
    for (int j = 0; j < N; ++j) score[j] = __fdiv_rn(score[j], den);
}

// ------------------------------------------------------------------------------------------------
// Hot loop: exactly N agents, agent 0 through the tight identity slab (IDENT0) or a box, agents 1..N-1 boxes.
// ------------------------------------------------------------------------------------------------
template <int MODE, int N, bool IDENT0, class Cfg>
__device__ __forceinline__ void fast_loop(const TileCtx &x, const float (&wt)[kTileMaxN][4], const uint32_t (&ta)[kTileMaxN]) {
    constexpr int G = Cfg::G, KC = Cfg::KC, P = Cfg::P, CHS = Cfg::CHS, BW = Cfg::BW, BOXF = Cfg::BOXF;
    constexpr int kParked = IDENT0 ? N - 1 : N;   // agents whose sampled vectors are parked (ATT)
    const int total = x.chunks * ((MODE == GC_FUSE_ATT && !x.park_mode) ? 2 : 1);
    const size_t dst_step = (size_t)G * x.plane;
    const uint32_t slot_stride = (uint32_t)x.C * P * 4u;
    float *dst = x.dst;
    float score[N];
#pragma unroll
    for (int j = 0; j < N; ++j) score[j] = 0.0f;

    int s = 0, chunk = 0, c0 = x.g;
    uint32_t parity = 0;
    uint32_t pk0 = x.park_addr + (uint32_t)(x.g * P + x.p) * 4u;   // park address of (slot 0, channel c0, pixel p)
    for (int it = 0; it < total; ++it) {
        const bool second = MODE == GC_FUSE_ATT && it >= x.chunks;
        mbar_wait(x.full_addr + 8u * s, parity);
        const uint32_t sb = x.ring_addr + (uint32_t)s * x.stage_bytes;
        uint32_t a[N], pk[N];
#pragma unroll
        for (int j = 0; j < N; ++j) { a[j] = sb + ta[j]; pk[j] = pk0 + (uint32_t)(IDENT0 ? j - 1 : j) * slot_stride; }
        static_for<KC>([&](auto kc_) {
            constexpr int kc = decltype(kc_)::value;
            if (c0 + G * kc < x.C) {   // warp-uniform; false only in the last chunk when C % CHS != 0
                float v[N];
                static_for<N>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    if (j == 0 && IDENT0) {
                        v[j] = lds<kc * G * P * 4>(a[j]);
                    } else {
                        constexpr int o = kc * G * BOXF * 4;
                        float acc = lds<o>(a[j]) * wt[j][0];
                        acc = __fmaf_rn(lds<o + 4>(a[j]), wt[j][1], acc);
                        acc = __fmaf_rn(lds<o + BW * 4>(a[j]), wt[j][2], acc);
                        acc = __fmaf_rn(lds<o + BW * 4 + 4>(a[j]), wt[j][3], acc);
                        v[j] = acc;
                    }
                });
                if (MODE == GC_FUSE_WARP_ONLY) {
#pragma unroll
                    for (int j = 0; j < N; ++j)
                        if (x.active) dst[(size_t)j * x.C * x.plane] = v[j];
                    dst += dst_step;
                } else if (MODE == GC_FUSE_MAX) {
                    float m = v[0];
#pragma unroll
                    for (int j = 1; j < N; ++j) m = fmaxf(m, v[j]);
                    if (x.active) *dst = m;
                    dst += dst_step;
                } else if (!second) {   // scores s_j += <w_0, w_j>; park the sampled vectors
#pragma unroll
                    for (int j = 0; j < N; ++j) score[j] = __fmaf_rn(v[0], v[j], score[j]);
                    if (x.park_mode) {
                        static_for<N>([&](auto j_) {
                            constexpr int j = decltype(j_)::value;
                            if (!(j == 0 && IDENT0)) sts<kc * G * P * 4>(pk[j], v[j]);
                        });
                    }
                } else {                // two-pass variant: out = sum_j a_j w_j
                    float acc = 0.0f;
#pragma unroll
                    for (int j = 0; j < N; ++j) acc = __fmaf_rn(score[j], v[j], acc);
                    if (x.active) *dst = acc;
                    dst += dst_step;
                }
            }
        });
        __syncwarp();   // this warp is done with the stage
        if (x.lane == 0) mbar_arrive(x.empty_addr + 8u * s);
        if (++s == x.stages) { s = 0; parity ^= 1u; }
        c0 += CHS; pk0 += CHS * P * 4;
        if (++chunk == x.chunks) {
            chunk = 0; c0 = x.g;
            if (MODE == GC_FUSE_ATT && !second) att_softmax<N, Cfg>(x, score);
        }
    }

    if (MODE == GC_FUSE_ATT && x.park_mode) {
        // out = sum_j a_j w_j from the parked vectors; the identity ego is re-read from global memory (L2 hits)
        uint32_t pkb = x.park_addr + (uint32_t)(x.g * P + x.p) * 4u;
        const float *sp = x.src_pix + (size_t)x.g * x.plane;
#pragma unroll 4
        for (int c = x.g; c < x.C; c += G) {
            float acc = 0.0f;
            static_for<N>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                float v;
                if (j == 0 && IDENT0) v = x.active ? __ldg(sp) : 0.0f;
                else v = lds<0>(pkb + (uint32_t)(IDENT0 ? j - 1 : j) * slot_stride);
                acc = __fmaf_rn(score[j], v, acc);
            });
            if (x.active) *dst = acc;
            dst += dst_step; sp += dst_step; pkb += G * P * 4;
        }
    }
    (void)kParked;
}

// ------------------------------------------------------------------------------------------------
// Generic loop: any mix of identity / box / gather agents (tiles where some affine map overflows its box).
// ------------------------------------------------------------------------------------------------
template <int MODE, class Cfg>
__device__ __forceinline__ void generic_loop(const TileCtx &x, const float (&wt)[kTileMaxN][4], const uint32_t (&ta)[kTileMaxN],
                                          const int (&goff)[kTileMaxN], unsigned m_ident, unsigned m_box, unsigned gvalid,
                                          const int *park_slot, bool use_ring, int W) {
    constexpr int NMAX = kTileMaxN, G = Cfg::G, KC = Cfg::KC, P = Cfg::P, CHS = Cfg::CHS, BW = Cfg::BW, BOXF = Cfg::BOXF;
    const int n = x.n, C = x.C;
    const int total = x.chunks * ((MODE == GC_FUSE_ATT && !x.park_mode) ? 2 : 1);
    const size_t plane = x.plane, dst_step = (size_t)G * plane;
    const float *src = x.src_pix - x.pix;   // plane base of the frame's first agent
    float *dst = x.dst;
    float score[NMAX];
#pragma unroll
    for (int j = 0; j < NMAX; ++j) score[j] = 0.0f;

    int s = 0, chunk = 0;
    uint32_t parity = 0;
    for (int it = 0; it < total; ++it) {
        const bool second = it >= x.chunks;
        if (use_ring) mbar_wait(x.full_addr + 8u * s, parity);
        const uint32_t sb = x.ring_addr + (uint32_t)s * x.stage_bytes;
#pragma unroll
        for (int kc = 0; kc < KC; ++kc) {
            const int c = chunk * CHS + x.g + G * kc;
            if (c < C) {   // warp-uniform
                float v[NMAX];
#pragma unroll
                for (int j = 0; j < NMAX; ++j) {
                    v[j] = 0.0f;
                    if (j >= n) continue;
                    if ((m_box >> j) & 1u) {
                        const uint32_t q = sb + ta[j] + (uint32_t)(kc * G * BOXF * 4);
                        float acc = lds<0>(q) * wt[j][0];
                        acc = __fmaf_rn(lds<4>(q), wt[j][1], acc);
                        acc = __fmaf_rn(lds<BW * 4>(q), wt[j][2], acc);
                        acc = __fmaf_rn(lds<BW * 4 + 4>(q), wt[j][3], acc);
                        v[j] = acc;
                    } else if ((m_ident >> j) & 1u) {
                        v[j] = lds<0>(sb + ta[j] + (uint32_t)(kc * G * P * 4));
                    } else {
                        Tap t;
                        t.w_nw = wt[j][0]; t.w_ne = wt[j][1]; t.w_sw = wt[j][2]; t.w_se = wt[j][3];
                        t.off = goff[j]; t.valid = (gvalid >> (4 * j)) & 15u;
                        v[j] = sample(src + ((size_t)j * C + c) * plane, t, W);
                    }
                }
                if (MODE == GC_FUSE_WARP_ONLY) {
#pragma unroll
                    for (int j = 0; j < NMAX; ++j)
                        if (j < n && x.active) dst[(size_t)j * C * plane] = v[j];
                    dst += dst_step;
                } else if (MODE == GC_FUSE_MAX) {
                    float m = v[0];
#pragma unroll
                    for (int j = 1; j < NMAX; ++j) if (j < n) m = fmaxf(m, v[j]);
                    if (x.active) *dst = m;
                    dst += dst_step;
                } else if (!second) {
#pragma unroll
                    for (int j = 0; j < NMAX; ++j) {
                        if (j < n) {
                            score[j] = __fmaf_rn(v[0], v[j], score[j]);
                            if (x.park_mode && park_slot[j] >= 0)
                                sts<0>(x.park_addr + (uint32_t)(((size_t)park_slot[j] * C + c) * P + x.p) * 4u, v[j]);
                        }
                    }
                } else {
                    float acc = 0.0f;
#pragma unroll
                    for (int j = 0; j < NMAX; ++j) if (j < n) acc = __fmaf_rn(score[j], v[j], acc);
                    if (x.active) *dst = acc;
                    dst += dst_step;
                }
            }
        }
        if (use_ring) {
            __syncwarp();
            if (x.lane == 0) mbar_arrive(x.empty_addr + 8u * s);
            if (++s == x.stages) { s = 0; parity ^= 1u; }
        }
        if (++chunk == x.chunks) {
            chunk = 0;
            if (MODE == GC_FUSE_ATT && !second) {
                // like att_softmax, for a run-time agent count
#pragma unroll
                for (int j = 0; j < NMAX; ++j) if (j < n) x.scratch[(x.g * NMAX + j) * P + x.p] = score[j];
                consumer_sync<Cfg::kConsumers>();
                float mx = -INFINITY;
#pragma unroll
                for (int j = 0; j < NMAX; ++j) {
                    if (j < n) {
                        float t = 0.0f;
#pragma unroll
                        for (int gg = 0; gg < G; ++gg) t += x.scratch[(gg * NMAX + j) * P + x.p];
                        score[j] = __fdiv_rn(t, x.sqrt_c);
                        mx = fmaxf(mx, score[j]);
                    }
                }
                float den = 0.0f;
#pragma unroll
                for (int j = 0; j < NMAX; ++j) if (j < n) { score[j] = expf(score[j] - mx); den += score[j]; }
#pragma unroll
                for (int j = 0; j < NMAX; ++j) score[j] = (j < n) ? __fdiv_rn(score[j], den) : 0.0f;
            }
        }
    }
    if (MODE == GC_FUSE_ATT && x.park_mode) {
        for (int c = x.g; c < C; c += G) {
            float acc = 0.0f;
#pragma unroll
            for (int j = 0; j < NMAX; ++j) {
                if (j < n) {
                    float v = 0.0f;
                    if ((m_ident >> j) & 1u) v = x.active ? __ldg(x.src_pix + ((size_t)j * C + c) * plane) : 0.0f;
                    else v = lds<0>(x.park_addr + (uint32_t)(((size_t)park_slot[j] * C + c) * P + x.p) * 4u);
                    acc = __fmaf_rn(score[j], v, acc);
                }
            }
            if (x.active) *dst = acc;
            dst += dst_step;
        }
    }
}

// MODE: GC_FUSE_WARP_ONLY, GC_FUSE_MAX, GC_FUSE_ATT; grid = (tiles x, tiles y, frame)
template <int MODE, class Cfg>
__global__ void __launch_bounds__(Cfg::kThreads, Cfg::CTAS)
k_fuse_tile(const __grid_constant__ CUtensorMap tmap_box, const __grid_constant__ CUtensorMap tmap_id,
            const float *__restrict__ feat, const int32_t *__restrict__ agent_offsets,
            const double *__restrict__ theta, int L, int C, int H, int W, float sqrt_c, int cap_floats,
            float *__restrict__ out) {
    constexpr int NMAX = kTileMaxN;
    constexpr int TW = Cfg::TW, TH = Cfg::TH, G = Cfg::G, P = Cfg::P, CHS = Cfg::CHS;
    constexpr int BW = Cfg::BW, BH = Cfg::BH, BOXF = Cfg::BOXF, kConsumers = Cfg::kConsumers;

    extern __shared__ uint8_t smem_raw[];
    // [scratch: tap exchange, later the score reduction][ring: stages * stage_floats][park: n_park * C * P]
    float *const scratch = reinterpret_cast<float *>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
    const uint32_t ring_addr = smem_u32(scratch) + Cfg::kScratch * 4u;
    __shared__ uint64_t full_bar[kMaxStages], empty_bar[kMaxStages];
    __shared__ double s_xs[TW], s_ys[TH];
    __shared__ int s_bx[NMAX], s_by[NMAX], s_path[NMAX], s_off[NMAX], s_park[NMAX];
    __shared__ int s_stage_floats, s_stages, s_park_mode, s_n_ring, s_any_gather;
    __shared__ unsigned s_ident;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool is_consumer = tid < kConsumers;
    const int p = tid % P, g = tid / P;           // g == G for the producer warp
    const int w0 = blockIdx.x * TW, h0 = blockIdx.y * TH;
    const int w = w0 + p % TW, h = h0 + p / TW;
    const bool active = is_consumer && w < W && h < H;
    const int b = blockIdx.z;
    const int a0 = __ldg(agent_offsets + b);
    const int n = min(min(__ldg(agent_offsets + b + 1) - a0, NMAX), L);
    const double *th_base = theta + (size_t)b * L * L * 6;   // row [b][0][j]
    const uint32_t full_addr = smem_u32(full_bar), empty_addr = smem_u32(empty_bar);

    // ---- base grid coordinates of the tile's columns / rows (float64, ATen linspace_from_neg_one) ------
    if (tid < TW) s_xs[tid] = base_coord(min(w0 + tid, W - 1), W);
    else if (tid < TW + TH) s_ys[tid - TW] = base_coord(min(h0 + tid - TW, H - 1), H);
    if (tid == 0) {
        for (int s = 0; s < kMaxStages; ++s) { mbar_init(full_addr + 8u * s, 1); mbar_init(empty_addr + 8u * s, kConsumers / 32); }
        mbar_init_fence();
        s_ident = 0xFFFFFFFFu;
    }
    __syncthreads();

    // ---- taps: group g computes agents j = g, g+G, ... for its pixel and publishes them ---------------
    // scratch as [j][k][p], k = w_nw, w_ne, w_sw, w_se, x0, y0
    if (is_consumer) {
        const double xs = s_xs[p % TW], ys = s_ys[p / TW];
        unsigned ident = 0xFFFFFFFFu;
        for (int j = g; j < n; j += G) {
            const TapS t = make_tap_xy(th_base + j * 6, xs, ys, H, W);
            float *q = scratch + (size_t)j * 6 * P + p;
            q[0] = t.w_nw; q[P] = t.w_ne; q[2 * P] = t.w_sw; q[3 * P] = t.w_se;
            q[4 * P] = __int_as_float(t.x0); q[5 * P] = __int_as_float(t.y0);
            const bool id = !active || (t.x0 == w && t.y0 == h && t.w_nw == 1.0f && t.w_ne == 0.0f &&
                                        t.w_sw == 0.0f && t.w_se == 0.0f);
            if (!id) ident &= ~(1u << j);
        }
        ident = __reduce_and_sync(0xffffffffu, ident);
        if (lane == 0 && ident != 0xFFFFFFFFu) atomicAnd(&s_ident, ident);
    }
    __syncthreads();

    // ---- per-agent path + box of this tile (warp 0, lane j), then the shared-memory plan ---------------
    if (warp == 0) {
        int path = 0, bx = 0, by = 0;
        if (lane < n) {
            if (lane == 0 && (s_ident & 1u)) {   // only the ego takes the tight identity slab
                path = kPathIdent; bx = w0; by = h0;
            } else {
                // the affine map is linear and rounding monotone: extremes of x0 / y0 are at the tile corners
                const int pw1 = min(TW - 1, W - 1 - w0), ph1 = min(TH - 1, H - 1 - h0);
                int minx = INT_MAX, maxx = INT_MIN, miny = INT_MAX, maxy = INT_MIN;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int pc = ((k & 2) ? ph1 : 0) * TW + ((k & 1) ? pw1 : 0);
                    const int x0 = __float_as_int(scratch[((size_t)lane * 6 + 4) * P + pc]);
                    const int y0 = __float_as_int(scratch[((size_t)lane * 6 + 5) * P + pc]);
                    minx = min(minx, x0); maxx = max(maxx, x0);
                    miny = min(miny, y0); maxy = max(maxy, y0);
                }
                bx = minx & ~3;   // floor to a multiple of 4 (two's complement): 16-byte aligned box start
                by = miny;
                // an out-of-view agent is a box of TMA zero fill; only an oversized footprint needs the gather path
                path = (maxx - bx + 2 <= BW && maxy - miny + 2 <= BH) ? kPathBox : kPathGather;
            }
        }
        const unsigned m_id = __ballot_sync(0xffffffffu, path == kPathIdent);
        const unsigned m_box = __ballot_sync(0xffffffffu, path == kPathBox);
        const unsigned m_ga = __ballot_sync(0xffffffffu, path == kPathGather);
        const unsigned below = (1u << lane) - 1u;
        if (lane < NMAX) {
            s_bx[lane] = bx; s_by[lane] = by; s_path[lane] = path;
            // stage layout: the identity slab first, then the boxes
            s_off[lane] = path == kPathIdent ? 0 : CHS * P * __popc(m_id) + CHS * BOXF * __popc(m_box & below);
            const unsigned m_park = m_box | m_ga;
            s_park[lane] = (MODE == GC_FUSE_ATT && ((m_park >> lane) & 1u)) ? __popc(m_park & below) : -1;
        }
        if (lane == 0) {
            const int n_id = __popc(m_id), n_box = __popc(m_box), n_park = MODE == GC_FUSE_ATT ? __popc(m_box | m_ga) : 0;
            const int stage_floats = CHS * (n_id * P + n_box * BOXF);
            const long long park_floats = (long long)n_park * C * P;
            const int min_ring = stage_floats * (stage_floats ? 2 : 0);
            const int park_mode = MODE == GC_FUSE_ATT && park_floats + min_ring <= cap_floats;
            int stages = 0;
            if (stage_floats) {
                stages = (int)((cap_floats - (park_mode ? park_floats : 0)) / stage_floats);
                stages = stages > kMaxStages ? kMaxStages : stages;   // host guarantees >= 1
            }
            s_stage_floats = stage_floats; s_stages = stages; s_park_mode = park_mode;
            s_n_ring = n_id + n_box; s_any_gather = m_ga != 0;
        }
    }
    __syncthreads();

    const int stage_floats = s_stage_floats, stages = s_stages;
    const bool park_mode = s_park_mode != 0, use_ring = s_n_ring > 0;
    const int chunks = (C + CHS - 1) / CHS;
    const size_t plane = (size_t)H * W;

    // ---- producer warp ----------------------------------------------------------------------------------
    if (!is_consumer) {
        if (lane == 0 && use_ring) {
            const int total = chunks * ((MODE == GC_FUSE_ATT && !park_mode) ? 2 : 1);
            int s = 0, chunk = 0;
            uint32_t parity = 1;   // first lap: the slots are free
            const uint32_t tx_bytes = (uint32_t)stage_floats * 4u;
            for (int it = 0; it < total; ++it) {
                mbar_wait(empty_addr + 8u * s, parity);
                mbar_expect_tx(full_addr + 8u * s, tx_bytes);
                const uint32_t dst = ring_addr + (uint32_t)s * tx_bytes;
                for (int j = 0; j < n; ++j) {
                    const int path = s_path[j];
                    if (path == kPathIdent)
                        tma_load_box(dst + s_off[j] * 4u, &tmap_id, s_bx[j], s_by[j], (a0 + j) * C + chunk * CHS, full_addr + 8u * s);
                    else if (path == kPathBox)
                        tma_load_box(dst + s_off[j] * 4u, &tmap_box, s_bx[j], s_by[j], (a0 + j) * C + chunk * CHS, full_addr + 8u * s);
                }
                if (++s == stages) { s = 0; parity ^= 1u; }
                if (++chunk == chunks) chunk = 0;
            }
        }
        return;
    }

    // ---- consumers: fold the per-agent geometry into one shared-memory byte offset --------------------
    float wt[NMAX][4];
    uint32_t ta[NMAX];       // byte offset inside a stage of this thread's first tap for channel slot g (ring agents)
    int goff[NMAX];          // gather agents: y0 * W + x0
    unsigned m_ident = 0, m_box = 0, gvalid = 0;
#pragma unroll
    for (int j = 0; j < NMAX; ++j) {
        wt[j][0] = wt[j][1] = wt[j][2] = wt[j][3] = 0.0f;
        ta[j] = 0; goff[j] = 0;
        if (j < n) {
            const int path = s_path[j];
            if (path == kPathIdent) {
                m_ident |= 1u << j;
                ta[j] = (uint32_t)(s_off[j] + g * P + p) * 4u;
            } else {
                const float *q = scratch + (size_t)j * 6 * P + p;
                wt[j][0] = q[0]; wt[j][1] = q[P]; wt[j][2] = q[2 * P]; wt[j][3] = q[3 * P];
                const int x0 = __float_as_int(q[4 * P]), y0 = __float_as_int(q[5 * P]);
                if (path == kPathBox) {
                    m_box |= 1u << j;
                    ta[j] = (uint32_t)(s_off[j] + g * BOXF + (y0 - s_by[j]) * BW + (x0 - s_bx[j])) * 4u;
                } else {
                    const bool xin0 = x0 >= 0 && x0 < W, xin1 = x0 + 1 >= 0 && x0 + 1 < W;
                    const bool yin0 = y0 >= 0 && y0 < H, yin1 = y0 + 1 >= 0 && y0 + 1 < H;
                    const unsigned v = ((xin0 && yin0) ? 1u : 0u) | ((xin1 && yin0) ? 2u : 0u) |
                                       ((xin0 && yin1) ? 4u : 0u) | ((xin1 && yin1) ? 8u : 0u);
                    gvalid |= (active ? v : 0u) << (4 * j);
                    goff[j] = y0 * W + x0;
                }
            }
        }
    }
    consumer_sync<kConsumers>();   // every tap has been read: scratch may be reused for the score reduction

    TileCtx x;
    x.ring_addr = ring_addr; x.stage_bytes = (uint32_t)stage_floats * 4u;
    x.park_addr = ring_addr + (uint32_t)stages * x.stage_bytes;
    x.full_addr = full_addr; x.empty_addr = empty_addr;
    x.stages = stages; x.chunks = chunks; x.C = C; x.n = n;
    x.park_mode = park_mode; x.active = active; x.lane = lane; x.g = g; x.p = p;
    x.sqrt_c = sqrt_c; x.scratch = scratch; x.plane = plane;
    const size_t pix = (size_t)(active ? h : 0) * W + (active ? w : 0);
    x.src_pix = feat + (size_t)a0 * C * plane + pix; x.pix = pix;
    // this thread's first channel is g; consecutive channels of the thread are G planes apart
    x.dst = out + ((size_t)(MODE == GC_FUSE_WARP_ONLY ? a0 : b) * C + g) * plane + pix;

    if (s_any_gather || n < 1) {
        generic_loop<MODE, Cfg>(x, wt, ta, goff, m_ident, m_box, gvalid, s_park, use_ring, W);
        return;
    }
    const bool id0 = (m_ident & 1u) != 0;
#define GC_FAST(N)                                                                   \
    case N:                                                                          \
        if (id0) fast_loop<MODE, N, true, Cfg>(x, wt, ta);                            \
        else fast_loop<MODE, N, false, Cfg>(x, wt, ta);                               \
        break;
    switch (n) {
        GC_FAST(1) GC_FAST(2) GC_FAST(3) GC_FAST(4) GC_FAST(5)
        default: break;
    }
#undef GC_FAST
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static bool encode_map(CUtensorMap *map, const float *feat, int W, int H, long long planes, int bw, int bh, int bc) {
    const auto encode = tensor_map_encoder();
    if (!encode) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)planes};
    const cuuint64_t gstride[2] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4};
    const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bc};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(feat), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int MODE, class Cfg>
static int launch_tile(cudaStream_t st, const float *feat, const int32_t *off, int n_frames, int total_agents,
                       const double *theta, int L, int C, int H, int W, float *out) {
    // worst-case stage (all agents through boxes) must fit at least once after the scratch
    const int cap_floats = (Cfg::kSmemBytes - 128) / 4 - Cfg::kScratch;
    if (Cfg::CHS * kTileMaxN * Cfg::BOXF > cap_floats) return 1;
    CUtensorMap map_box, map_id;
    const long long planes = (long long)total_agents * C;
    if (!encode_map(&map_box, feat, W, H, planes, Cfg::BW, Cfg::BH, Cfg::CHS)) return 1;
    if (!encode_map(&map_id, feat, W, H, planes, Cfg::TW, Cfg::TH, Cfg::CHS)) return 1;
    auto kern = k_fuse_tile<MODE, Cfg>;
    static bool configured = false;   // one attribute call per instantiation
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            set_error("k_fuse_tile: cudaFuncSetAttribute failed (%d)", (int)e);
            return (int)e;
        }
        configured = true;
    }
    const dim3 grid((W + Cfg::TW - 1) / Cfg::TW, (H + Cfg::TH - 1) / Cfg::TH, n_frames);
    if (grid.y > 65535 || grid.z > 65535) return 1;
    const float sqrt_c = (float)sqrt((double)C);
    kern<<<grid, Cfg::kThreads, Cfg::kSmemBytes, st>>>(map_box, map_id, feat, off, theta, L, C, H, W, sqrt_c, cap_floats, out);
    GC_LAUNCH_CHECK("k_fuse_tile");
    return GC_OK;
}

// Returns GC_OK when the tiled path was launched, 1 when the configuration is not eligible (caller falls
// back to the gather kernels), or an error code.  nmax: upper bound on the agents of any one frame.
int warp_fuse_tile(const float *feat, const int32_t *agent_offsets, int n_frames, int total_agents,
                   const double *theta, int L, int C, int H, int W, int mode, int nmax, float *out,
                   cudaStream_t st) {
    if ((W & 3) != 0 || ((uintptr_t)feat & 15) != 0) return 1;
    if (nmax > kTileMaxN) return 1;
    if ((long long)total_agents * C >= (1ll << 31)) return 1;
    using Cfg2 = TileCfg<16, 8, 4, 2>;   // 8 channel planes per stage
    using Cfg1 = TileCfg<16, 8, 4, 1>;   // 4 channel planes per stage (5 agents: the park needs the room)
    if (mode == GC_FUSE_WARP_ONLY)
        return launch_tile<GC_FUSE_WARP_ONLY, Cfg2>(st, feat, agent_offsets, n_frames, total_agents, theta, L, C, H, W, out);
    using CfgX = TileCfg<16, 8, 2, 2, 2>;   // experiment: 2 CTAs per SM
    const char *ex = getenv("GC_TILE_X");
    if (mode == GC_FUSE_MAX && ex && ex[0] == '1')
        return launch_tile<GC_FUSE_MAX, CfgX>(st, feat, agent_offsets, n_frames, total_agents, theta, L, C, H, W, out);
    if (mode == GC_FUSE_MAX)
        return launch_tile<GC_FUSE_MAX, Cfg2>(st, feat, agent_offsets, n_frames, total_agents, theta, L, C, H, W, out);
    if (nmax <= 4)
        return launch_tile<GC_FUSE_ATT, Cfg2>(st, feat, agent_offsets, n_frames, total_agents, theta, L, C, H, W, out);
    return launch_tile<GC_FUSE_ATT, Cfg1>(st, feat, agent_offsets, n_frames, total_agents, theta, L, C, H, W, out);
}

}  // namespace gc
