// Persistent, TMA-staged warp + regroup + Max/Att fusion for sm_100a (the fast path of gc_warp_fuse).
//
// Same operator and numerics as warp_fuse.cu (reference: fusion_in_one.py:53-151,
// torch_transformation_utils.py:323-332); this file is about data movement.
//
// Round-1c ncu of the per-tile kernel (one CTA per 16x8 tile, 1 CTA/SM because of the 224 KB ring+park): 29 % of
// the stall samples were consumers waiting on the TMA full barrier, 19 % of all instructions were per-tile setup,
// and the TMA pipeline idled during every tile's setup and AttFusion epilogue.  This version:
//
//   * ONE persistent CTA per SM walks tiles t = blockIdx.x, += gridDim.x.  The producer warp derives each tile's
//     source boxes itself (from the four tile corners of every agent's affine map) and keeps the ring full ACROSS
//     tile boundaries: while the consumers run tile t's epilogue and tile t+1's setup, tile t+1's channel planes
//     are already in flight.
//   * A stage slot has a fixed size (n_bound agents x CHS channel planes x one BW x BH box): no per-tile ring
//     re-planning, no block-wide barriers between producer and consumers except the mbarrier ring.
//   * Consumers (P pixels x G channel groups) compute their own bilinear taps in registers (float64 affine, the
//     grid rounded to float32, ATen's float32 unnormalise/floor/weights); only the per-tile box origins go through
//     shared memory (consumer warp 0 -> all consumers, named barrier, double buffered).
//   * Hot loop as before: compile-time agent count, per-agent weights + ONE shared-memory byte address in registers;
//     a sample is 4 LDS with immediate offsets + 4 FMA.  AttFusion in one pass over HBM (sampled vectors of the
//     non-identity agents parked in shared memory while the ego-row scores accumulate).
//   * The source footprint of a tile under a near-isometry fits the BW x BH box (TMA zero fill == grid_sample
//     padding_mode='zeros').  A tile where some affine map overflows its box is a "slow tile": the producer skips
//     it and the consumers gather straight from global memory (rare: non-isometric transforms only).
//
// Requirements checked by the host: W % 4 == 0 and 16-byte aligned base (TMA global strides; the probe
// scripts/probes/tma_align.cu shows the innermost TMA start coordinate must be a multiple of 16 bytes), at most
// kTileMaxN agents per frame.  Otherwise gc_warp_fuse uses the gather kernels of warp_fuse.cu.
#include <stdlib.h>

#include "ptx.cuh"
#include "warp_common.cuh"

namespace gc {
namespace persist {

using namespace ptx;

constexpr int kTileMaxN = 8;
constexpr int kMaxStages = 8;
constexpr int kGeomSlots = 4;   // tiles of geometry the geometry warp may run ahead
constexpr int kDynSmemBytes = 224 * 1024;

constexpr int isqrt_ceil(int v) {
    int r = 0;
    while (r * r < v) ++r;
    return r;
}

template <int TW_, int TH_, int G_, int KC_>
struct Cfg {
    static constexpr int TW = TW_, TH = TH_, G = G_, KC = KC_;
    static constexpr int P = TW * TH;                  // pixels per tile
    static constexpr int CHS = G * KC;                 // channel planes per pipeline stage
    static constexpr int kConsumers = P * G;
    static constexpr int kThreads = kConsumers + 64;   // + producer warp + geometry warp
    // x0 = floor(ix) spans at most ceil(diagonal) + 1 values over the tile, + 1 for the x0+1 tap
    static constexpr int EXT = isqrt_ceil((TW - 1) * (TW - 1) + (TH - 1) * (TH - 1)) + 2;
    static constexpr int BW = (EXT + 3 + 3) & ~3;      // + up to 3 columns: box x origin floored to 16 bytes
    static constexpr int BH = EXT;
    static constexpr int BOXF = BW * BH;
    static constexpr int kAgentFloats = (CHS * BOXF + 31) & ~31;   // per-agent region of a stage slot (128-byte aligned)
    static constexpr int kScratch = kTileMaxN * P * G;   // AttFusion score reduction [G][N][P]
    // tensor-memory park: one thread per pixel owning 4 consecutive channels per stage, lanes = pixel % 128
    static constexpr bool kTmemOK = G == 1 && KC == 4 && P % 128 == 0;
    static_assert(P % 32 == 0 && TW % 4 == 0, "tile rows must be 16-byte multiples, groups warp aligned");
    static_assert(kConsumers % 32 == 0, "whole consumer warps");
    static_assert(kThreads <= 1024, "block too large");
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

enum AgentPath { kPathNone = 0, kPathIdent = 1, kPathBox = 2, kPathGather = 3 };

struct Geom {   // per (tile, agent): which box the producer loads
    int bx, by, path;
};

// Warp-cooperative geometry of one tile: lane j < n returns agent j's box.  Deterministic in (theta, tile), so the
// producer warp and consumer warp 0 evaluate it independently and agree.  All 32 lanes must call it.
template <class C_>
__device__ __forceinline__ Geom tile_geom(int lane, int n, const double *__restrict__ th_base, int w0, int h0, int H, int W) {
    constexpr int TW = C_::TW, TH = C_::TH, P = C_::P, BW = C_::BW, BH = C_::BH;
    Geom g;
    g.bx = 0; g.by = 0; g.path = kPathNone;
    const int pw1 = min(TW - 1, W - 1 - w0), ph1 = min(TH - 1, H - 1 - h0);
    if (lane < n) {
        // the affine map is linear and rounding monotone: extremes of x0 / y0 are at the tile corners
        const double *th = th_base + lane * 6;
        int minx = INT_MAX, maxx = INT_MIN, miny = INT_MAX, maxy = INT_MIN;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const TapS t = make_tap_xy(th, base_coord(w0 + ((k & 1) ? pw1 : 0), W), base_coord(h0 + ((k & 2) ? ph1 : 0), H), H, W);
            minx = min(minx, t.x0); maxx = max(maxx, t.x0);
            miny = min(miny, t.y0); maxy = max(maxy, t.y0);
        }
        g.bx = minx & ~3;   // floor to a multiple of 4 (two's complement): 16-byte aligned box start
        g.by = miny;
        // an out-of-view agent is a box of TMA zero fill; only an oversized footprint needs the gather path
        g.path = (maxx - g.bx + 2 <= BW && maxy - miny + 2 <= BH) ? kPathBox : kPathGather;
    }
    // the ego takes the tight identity slab when every pixel of the tile samples exactly itself
    const double *t0 = th_base;
    const bool ident_theta = n > 0 && t0[0] == 1.0 && t0[1] == 0.0 && t0[2] == 0.0 && t0[3] == 0.0 && t0[4] == 1.0 && t0[5] == 0.0;
    if (ident_theta) {   // warp-uniform
        bool ok = true;
        for (int p = lane; p < P; p += 32) {
            const int w = w0 + p % TW, h = h0 + p / TW;
            if (w < W && h < H) {
                const TapS t = make_tap_xy(t0, base_coord(w, W), base_coord(h, H), H, W);
                ok = ok && t.x0 == w && t.y0 == h && t.w_nw == 1.0f && t.w_ne == 0.0f && t.w_sw == 0.0f && t.w_se == 0.0f;
            }
        }
        ok = __all_sync(0xffffffffu, ok);
        if (ok && lane == 0) { g.path = kPathIdent; g.bx = w0; g.by = h0; }
    }
    return g;
}

// everything the consumer loops need
struct Ctx {
    uint32_t ring_addr, slot_bytes, park_addr, full_addr, empty_addr;
    int stages, chunks, C;
    bool park_mode, active;
    bool park_tmem;        // the park lives in tensor memory (G == 1, KC == 4 configurations)
    uint32_t tmem_park;    // TMEM address of (this thread's lane, column of park slot 0 / channel 0 of its pixel set)
    int lane, g, p;
    float sqrt_c;
    float *scratch;
    float *dst;            // out + (first output plane of the tile + g) * plane + pix
    const float *src_pix;  // feat + a0 * C * plane + pix
    size_t plane;
    int s;                 // ring position, persists across tiles
    uint32_t parity;
};

// softmax over the ego-row scores after combining the G channel groups in a fixed order
// (score / sqrt(C), fusion_in_one.py:42-43).  score[] holds the attention weights on return.
template <int N, class C_>
__device__ __forceinline__ void att_softmax(const Ctx &x, float (&score)[N]) {
    constexpr int G = C_::G, P = C_::P;
    if (G > 1) {
#pragma unroll
        for (int j = 0; j < N; ++j) x.scratch[(x.g * N + j) * P + x.p] = score[j];
        consumer_sync<C_::kConsumers>();
    }
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        float t = score[j];   // G == 1: the thread already holds the full dot product
        if (G > 1) {
            t = 0.0f;
#pragma unroll
            for (int gg = 0; gg < G; ++gg) t += x.scratch[(gg * N + j) * P + x.p];
        }
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
// Hot loop of one tile: exactly N agents, agent 0 through the tight identity slab (IDENT0) or a box.
// ------------------------------------------------------------------------------------------------
template <int MODE, int N, bool IDENT0, class C_>
__device__ __forceinline__ void fast_loop(Ctx &x, const float (&wt)[kTileMaxN][4], const uint32_t (&ta)[kTileMaxN]) {
    constexpr int G = C_::G, KC = C_::KC, P = C_::P, CHS = C_::CHS, BW = C_::BW, BOXF = C_::BOXF;
    constexpr bool kTmemOK = C_::kTmemOK;
    const int total = x.chunks * ((MODE == GC_FUSE_ATT && !x.park_mode) ? 2 : 1);
    const size_t dst_step = (size_t)G * x.plane;
    const uint32_t slot_stride = (uint32_t)x.C * P * 4u;
    float *dst = x.dst;
    float score[N];
#pragma unroll
    for (int j = 0; j < N; ++j) score[j] = 0.0f;

    int s = x.s, chunk = 0, c0 = x.g;
    uint32_t parity = x.parity;
    uint32_t pk0 = x.park_addr + (uint32_t)(x.g * P + x.p) * 4u;   // park address of (slot 0, channel c0, pixel p)
    for (int it = 0; it < total; ++it) {
        const bool second = MODE == GC_FUSE_ATT && it >= x.chunks;
        mbar_wait(x.full_addr + 8u * s, parity);
        const uint32_t sb = x.ring_addr + (uint32_t)s * x.slot_bytes;
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
                    if (kTmemOK && x.park_tmem) {
                        // tensor-memory park: 4 columns per channel = the (up to 4) parked agents of this pixel
                        if (x.park_mode) {
                            constexpr int o = IDENT0 ? 1 : 0;   // first parked agent
                            // with at most 3 parked agents the fourth column carries the identity ego, so the output
                            // pass below never goes back to global memory (r02: 16 dependent L2 round trips per tile)
                            constexpr bool kEgoCol = IDENT0 && N <= 4;
                            tmem_st4(x.tmem_park + (uint32_t)((c0 + G * kc) * 4), v[o < N ? o : 0], v[o + 1 < N ? o + 1 : 0],
                                     v[o + 2 < N ? o + 2 : 0], kEgoCol ? v[0] : v[o + 3 < N ? o + 3 : 0]);
                        }
                    } else if (x.park_mode) {
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
            chunk = 0; c0 = x.g; pk0 = x.park_addr + (uint32_t)(x.g * P + x.p) * 4u;
            if (MODE == GC_FUSE_ATT && !second) att_softmax<N, C_>(x, score);
        }
    }
    x.s = s; x.parity = parity;

    if constexpr (kTmemOK && MODE == GC_FUSE_ATT) {
        if (x.park_tmem && x.park_mode) {
            // out = sum_j a_j w_j from the vectors parked in tensor memory: one 16-column load = 4 channels x 4 agents;
            // two loads in flight per iteration (C % 8 == 0 takes the unrolled body)
            constexpr int o = IDENT0 ? 1 : 0;
            constexpr bool kEgoCol = IDENT0 && N <= 4;
            tmem_wait_st();
            const float *sp = x.src_pix;
            auto emit = [&](const float (&pv)[16], const float (&ego)[4], float *d) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float acc = 0.0f;
#pragma unroll
                    for (int j = 0; j < N; ++j) {
                        const float v = (j == 0 && IDENT0) ? (kEgoCol ? pv[i * 4 + 3] : ego[i]) : pv[i * 4 + (j - o < 0 ? 0 : j - o)];
                        acc = __fmaf_rn(score[j], v, acc);
                    }
                    if (x.active) d[(size_t)i * x.plane] = acc;
                }
            };
            int c = 0;
            for (; c + 8 <= x.C; c += 8) {
                float pa[16], pb[16], ea[4] = {0.f, 0.f, 0.f, 0.f}, eb[4] = {0.f, 0.f, 0.f, 0.f};
                tmem_ld16_nowait(x.tmem_park + (uint32_t)(c * 4), pa);
                tmem_ld16_nowait(x.tmem_park + (uint32_t)(c * 4 + 16), pb);
                if (IDENT0 && !kEgoCol) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        ea[i] = x.active ? __ldg(sp + (size_t)i * x.plane) : 0.0f;
                        eb[i] = x.active ? __ldg(sp + (size_t)(i + 4) * x.plane) : 0.0f;
                    }
                }
                tmem_wait_ld();
                emit(pa, ea, dst);
                emit(pb, eb, dst + 4 * x.plane);
                dst += 8 * x.plane; sp += 8 * x.plane;
            }
            for (; c < x.C; c += 4) {   // C % 4 == 0 in this mode
                float pv[16], ego[4] = {0.f, 0.f, 0.f, 0.f};
                tmem_ld16_nowait(x.tmem_park + (uint32_t)(c * 4), pv);
                if (IDENT0 && !kEgoCol) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) ego[i] = x.active ? __ldg(sp + (size_t)i * x.plane) : 0.0f;
                }
                tmem_wait_ld();
                emit(pv, ego, dst);
                dst += 4 * x.plane; sp += 4 * x.plane;
            }
            return;
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
}

// ------------------------------------------------------------------------------------------------
// Slow tile: every agent sampled straight from global memory (some affine map overflows its box).
// ------------------------------------------------------------------------------------------------
template <int MODE, class C_>
__device__ __forceinline__ void gather_tile(const Ctx &x, int n, const double *__restrict__ th_base, int w, int h, int H, int W) {
    constexpr int NMAX = kTileMaxN, G = C_::G, P = C_::P;
    const int C = x.C;
    const size_t plane = x.plane;
    const size_t pix = x.active ? (size_t)h * W + w : 0;
    const float *src = x.src_pix - pix;   // plane base of the frame's first agent
    Tap tap[NMAX];
    const double xs = base_coord(min(w, W - 1), W), ys = base_coord(min(h, H - 1), H);
#pragma unroll
    for (int j = 0; j < NMAX; ++j) {
        if (j < n) {
            tap[j] = make_tap(th_base + j * 6, xs, ys, H, W);
            if (!x.active) tap[j].valid = 0;
        } else {
            tap[j].valid = 0; tap[j].off = 0;
            tap[j].w_nw = tap[j].w_ne = tap[j].w_sw = tap[j].w_se = 0.0f;
        }
    }
    float *dst = x.dst;
    const size_t dst_step = (size_t)G * plane;
    if (MODE == GC_FUSE_WARP_ONLY) {
        for (int c = x.g; c < C; c += G, dst += dst_step) {
#pragma unroll
            for (int j = 0; j < NMAX; ++j)
                if (j < n && x.active) dst[(size_t)j * C * plane] = sample(src + ((size_t)j * C + c) * plane, tap[j], W);
        }
    } else if (MODE == GC_FUSE_MAX) {
        for (int c = x.g; c < C; c += G, dst += dst_step) {
            float m = 0.0f;
#pragma unroll
            for (int j = 0; j < NMAX; ++j) {
                if (j < n) {
                    const float v = sample(src + ((size_t)j * C + c) * plane, tap[j], W);
                    m = (j == 0) ? v : fmaxf(m, v);
                }
            }
            if (x.active) *dst = m;
        }
    } else {
        float score[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; ++j) score[j] = 0.0f;
        for (int c = x.g; c < C; c += G) {
            const float v0 = sample(src + (size_t)c * plane, tap[0], W);
#pragma unroll
            for (int j = 0; j < NMAX; ++j) {
                if (j < n) {
                    const float v = (j == 0) ? v0 : sample(src + ((size_t)j * C + c) * plane, tap[j], W);
                    score[j] = __fmaf_rn(v0, v, score[j]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < NMAX; ++j) if (j < n) x.scratch[(x.g * NMAX + j) * P + x.p] = score[j];
        consumer_sync<C_::kConsumers>();
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
        for (int c = x.g; c < C; c += G, dst += dst_step) {
            float acc = 0.0f;
#pragma unroll
            for (int j = 0; j < NMAX; ++j)
                if (j < n) acc = __fmaf_rn(score[j], sample(src + ((size_t)j * C + c) * plane, tap[j], W), acc);
            if (x.active) *dst = acc;
        }
    }
}

struct LaunchPlan {
    int tiles_x, tiles_y, n_tiles;
    int stages, slot_floats, park_slots;   // park_slots: agents whose sampled vectors fit the park (ATT), 0 = two passes
    int n_bound;
    int park_tmem;   // 1: the AttFusion park lives in tensor memory (no shared memory taken from the ring)
};

// MODE: GC_FUSE_WARP_ONLY, GC_FUSE_MAX, GC_FUSE_ATT; grid = min(n_tiles, #SM) persistent CTAs
template <int MODE, class C_>
__global__ void __launch_bounds__(C_::kThreads, 1)
k_fuse_persist(const __grid_constant__ CUtensorMap tmap_box, const __grid_constant__ CUtensorMap tmap_id,
               const float *__restrict__ feat, const int32_t *__restrict__ agent_offsets,
               const double *__restrict__ theta, int L, int C, int H, int W, float sqrt_c, LaunchPlan plan,
               float *__restrict__ out) {
    constexpr int NMAX = kTileMaxN;
    constexpr int TW = C_::TW, TH = C_::TH, P = C_::P, CHS = C_::CHS;
    constexpr int BW = C_::BW, BOXF = C_::BOXF, kConsumers = C_::kConsumers;

    extern __shared__ uint8_t smem_raw[];
    // [ring: stages * slot][park: park_slots * C * P][scratch: G * NMAX * P (ATT)]
    uint8_t *const base = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
    const uint32_t ring_addr = smem_u32(base);
    const uint32_t slot_bytes = (uint32_t)plan.slot_floats * 4u;
    const uint32_t park_addr = ring_addr + (uint32_t)plan.stages * slot_bytes;
    float *const scratch = reinterpret_cast<float *>(base + (size_t)plan.stages * slot_bytes +
                                                     (plan.park_tmem ? 0 : (size_t)plan.park_slots * C * P * 4));
    __shared__ __align__(8) uint64_t full_bar[kMaxStages], empty_bar[kMaxStages];
    __shared__ __align__(8) uint64_t gfull_bar[kGeomSlots], gempty_bar[kGeomSlots];
    __shared__ int s_geom[kGeomSlots][NMAX][3];
    __shared__ int s_slow[kGeomSlots];
    __shared__ uint32_t s_tmem;

    const int tid = threadIdx.x, lane = tid & 31;
    const bool is_consumer = tid < kConsumers;
    const uint32_t full_addr = smem_u32(full_bar), empty_addr = smem_u32(empty_bar);
    const uint32_t gfull_addr = smem_u32(gfull_bar), gempty_addr = smem_u32(gempty_bar);
    const int chunks = (C + CHS - 1) / CHS;
    const size_t plane = (size_t)H * W;
    const int tiles_per_frame = plan.tiles_x * plan.tiles_y;

    if (tid == 0) {
        for (int s = 0; s < kMaxStages; ++s) { mbar_init(full_addr + 8u * s, 1); mbar_init(empty_addr + 8u * s, kConsumers / 32); }
        for (int s = 0; s < kGeomSlots; ++s) { mbar_init(gfull_addr + 8u * s, 1); mbar_init(gempty_addr + 8u * s, kConsumers / 32 + 1); }
        mbar_init_fence();
    }
    // tensor memory as a 256 KB per-SM scratchpad (AttFusion park, lane = pixel % 128): all 512 columns, 1 CTA per SM
    if (MODE == GC_FUSE_ATT && plan.park_tmem && tid < 32) tmem_alloc<512>(&s_tmem);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    // ---- geometry warp: box origins / paths of the tiles ahead, published through a small ring so that neither the
    // producer nor the consumers have the float64 corner evaluation (and the per-tile identity check) on their path
    if (tid >= kConsumers + 32) {
        int slot = 0;
        uint32_t parity = 1;   // first lap: the slots are free
        for (int t = blockIdx.x; t < plan.n_tiles; t += gridDim.x) {
            const int b = t / tiles_per_frame, r = t - b * tiles_per_frame;
            const int w0 = (r % plan.tiles_x) * TW, h0 = (r / plan.tiles_x) * TH;
            const int a0 = __ldg(agent_offsets + b);
            const int n = min(min(__ldg(agent_offsets + b + 1) - a0, plan.n_bound), L);
            const Geom gm = tile_geom<C_>(lane, n, theta + (size_t)b * L * L * 6, w0, h0, H, W);
            const bool slow = __any_sync(0xffffffffu, gm.path == kPathGather) || n < 1;
            mbar_wait(gempty_addr + 8u * slot, parity);
            if (lane < NMAX) { s_geom[slot][lane][0] = gm.bx; s_geom[slot][lane][1] = gm.by; s_geom[slot][lane][2] = gm.path; }
            if (lane == 0) s_slow[slot] = slow ? 1 : 0;
            __syncwarp();
            if (lane == 0) mbar_arrive(gfull_addr + 8u * slot);
            if (++slot == kGeomSlots) { slot = 0; parity ^= 1u; }
        }
        return;
    }

    // ---- producer: one thread keeps the ring full, across tile boundaries -------------------------------------
    if (!is_consumer) {
        if (lane != 0) return;
        int s = 0, slot = 0;
        uint32_t parity = 1, gparity = 0;   // ring slots start free; geometry slots start empty
        for (int t = blockIdx.x; t < plan.n_tiles; t += gridDim.x) {
            const int b = t / tiles_per_frame;
            const int a0 = __ldg(agent_offsets + b);
            const int n = min(min(__ldg(agent_offsets + b + 1) - a0, plan.n_bound), L);
            mbar_wait(gfull_addr + 8u * slot, gparity);
            const bool slow = s_slow[slot] != 0;
            int bx[NMAX], by[NMAX], path[NMAX];
#pragma unroll
            for (int j = 0; j < NMAX; ++j) { bx[j] = s_geom[slot][j][0]; by[j] = s_geom[slot][j][1]; path[j] = s_geom[slot][j][2]; }
            mbar_arrive(gempty_addr + 8u * slot);
            if (++slot == kGeomSlots) { slot = 0; gparity ^= 1u; }
            if (slow) continue;   // consumers gather this tile from global memory
            const int n_id = path[0] == kPathIdent ? 1 : 0;
            const int parked = n - n_id;
            const bool park_mode = MODE == GC_FUSE_ATT && parked <= plan.park_slots;
            const int total = chunks * ((MODE == GC_FUSE_ATT && !park_mode) ? 2 : 1);
            const uint32_t tx_bytes = (uint32_t)CHS * (uint32_t)(n_id * P + (n - n_id) * BOXF) * 4u;
            int chunk = 0;
            for (int it = 0; it < total; ++it) {
                mbar_wait(empty_addr + 8u * s, parity);
                mbar_expect_tx(full_addr + 8u * s, tx_bytes);
                const uint32_t dst = ring_addr + (uint32_t)s * slot_bytes;
#pragma unroll
                for (int j = 0; j < NMAX; ++j) {
                    if (j < n)
                        tma_load_box(dst + (uint32_t)(j * C_::kAgentFloats) * 4u, path[j] == kPathIdent ? &tmap_id : &tmap_box,
                                     bx[j], by[j], (a0 + j) * C + chunk * CHS, full_addr + 8u * s);
                }
                if (++s == plan.stages) { s = 0; parity ^= 1u; }
                if (++chunk == chunks) chunk = 0;
            }
        }
        return;
    }

    // ---- consumers ------------------------------------------------------------------------------------------
    const int p = tid % P, g = tid / P;
    Ctx x;
    x.ring_addr = ring_addr; x.slot_bytes = slot_bytes; x.park_addr = park_addr;
    x.full_addr = full_addr; x.empty_addr = empty_addr;
    x.stages = plan.stages; x.chunks = chunks; x.C = C;
    x.lane = lane; x.g = g; x.p = p; x.sqrt_c = sqrt_c; x.plane = plane;
    x.s = 0; x.parity = 0;
    x.park_tmem = MODE == GC_FUSE_ATT && plan.park_tmem != 0;
    // lane quadrant of this warp = (tid / 32) % 4 = (p / 32) % 4 because P % 128 == 0; pixel set p / 128 owns its own columns
    x.tmem_park = x.park_tmem ? s_tmem + ((uint32_t)(((tid >> 5) & 3) * 32) << 16) + (uint32_t)((p / 128) * C * 4) : 0u;

    int slot = 0, it_tile = 0;
    uint32_t gparity = 0;
    for (int t = blockIdx.x; t < plan.n_tiles; t += gridDim.x, it_tile ^= 1) {
        const int b = t / tiles_per_frame, r = t - b * tiles_per_frame;
        const int w0 = (r % plan.tiles_x) * TW, h0 = (r / plan.tiles_x) * TH;
        const int w = w0 + p % TW, h = h0 + p / TW;
        const bool active = w < W && h < H;
        const int a0 = __ldg(agent_offsets + b);
        const int n = min(min(__ldg(agent_offsets + b + 1) - a0, plan.n_bound), L);
        const double *th_base = theta + (size_t)b * L * L * 6;   // row [b][0][j]
        const size_t pix = (size_t)(active ? h : 0) * W + (active ? w : 0);
        x.active = active;
        x.src_pix = feat + (size_t)a0 * C * plane + pix;
        // this thread's first channel is g; consecutive channels of the thread are G planes apart
        x.dst = out + ((size_t)(MODE == GC_FUSE_WARP_ONLY ? a0 : b) * C + g) * plane + pix;
        x.scratch = scratch + it_tile * C_::kScratch;   // double buffered: a warp may run one tile ahead of another

        // own taps for every agent (independent of the tile geometry, overlaps the wait below)
        const double xs = base_coord(min(w, W - 1), W), ys = base_coord(min(h, H - 1), H);
        float wt[NMAX][4];
        int tx0[NMAX], ty0[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; ++j) {
            wt[j][0] = wt[j][1] = wt[j][2] = wt[j][3] = 0.0f;
            tx0[j] = ty0[j] = 0;
            if (j < n) {
                const TapS tp = make_tap_xy(th_base + j * 6, xs, ys, H, W);
                wt[j][0] = tp.w_nw; wt[j][1] = tp.w_ne; wt[j][2] = tp.w_sw; wt[j][3] = tp.w_se;
                tx0[j] = tp.x0; ty0[j] = tp.y0;
            }
        }
        // geometry of this tile from the geometry warp
        mbar_wait(gfull_addr + 8u * slot, gparity);
        const bool slow = s_slow[slot] != 0;
        const bool id0 = s_geom[slot][0][2] == kPathIdent;
        uint32_t ta[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; ++j) {
            ta[j] = (uint32_t)(j * C_::kAgentFloats) * 4u;
            if (j < n) {
                if (j == 0 && id0) {
                    ta[j] += (uint32_t)(g * P + p) * 4u;
                } else {
                    // inactive threads of a partial tile may fall outside the box: keep their address inside it
                    const int dx = active ? tx0[j] - s_geom[slot][j][0] : 0, dy = active ? ty0[j] - s_geom[slot][j][1] : 0;
                    ta[j] += (uint32_t)(g * BOXF + dy * BW + dx) * 4u;
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(gempty_addr + 8u * slot);
        if (++slot == kGeomSlots) { slot = 0; gparity ^= 1u; }

        if (slow) {
            if (n >= 1) gather_tile<MODE, C_>(x, n, th_base, w, h, H, W);
            continue;
        }
        const int parked = n - (id0 ? 1 : 0);
        x.park_mode = MODE == GC_FUSE_ATT && parked <= plan.park_slots;

#define GC_FAST(N)                                                                   \
    case N:                                                                          \
        if (id0) fast_loop<MODE, N, true, C_>(x, wt, ta);                             \
        else fast_loop<MODE, N, false, C_>(x, wt, ta);                                \
        break;
        switch (n) {
            GC_FAST(1) GC_FAST(2) GC_FAST(3) GC_FAST(4) GC_FAST(5) GC_FAST(6) GC_FAST(7) GC_FAST(8)
            default: break;
        }
#undef GC_FAST
    }
    if (MODE == GC_FUSE_ATT && plan.park_tmem) {   // every consumer is done with tensor memory
        tc_fence_before();
        consumer_sync<kConsumers>();
        if (tid < 32) tmem_free<512>(s_tmem);
    }
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

static int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
        (void)cudaGetLastError();
    }
    return n;
}

template <int MODE, class C_>
static int launch(cudaStream_t st, const float *feat, const int32_t *off, int n_frames, int total_agents,
                  const double *theta, int L, int C, int H, int W, int n_bound, float *out) {
    LaunchPlan plan;
    plan.tiles_x = (W + C_::TW - 1) / C_::TW;
    plan.tiles_y = (H + C_::TH - 1) / C_::TH;
    const long long n_tiles = (long long)plan.tiles_x * plan.tiles_y * n_frames;
    if (n_tiles >= (1ll << 30)) return 1;
    plan.n_tiles = (int)n_tiles;
    plan.n_bound = n_bound;
    plan.slot_floats = n_bound * C_::kAgentFloats;
    const long long cap = (kDynSmemBytes - 128) / 4;   // floats
    const long long scratch = MODE == GC_FUSE_ATT ? 2 * C_::kScratch : 0;   // double buffered by tile parity
    plan.park_slots = 0;
    plan.park_tmem = 0;
    if (MODE == GC_FUSE_ATT && C_::kTmemOK && C % 4 == 0 && n_bound > 1 && n_bound <= 5 &&
        (long long)(C_::P / 128) * C * 4 <= 512 && !getenv("GC_FUSE_NO_TMEM")) {   // 4 columns per (pixel set, channel)
        plan.park_tmem = 1;               // 512 columns x 128 lanes x 32 bit of tensor memory hold the park
        plan.park_slots = n_bound - 1;
    } else if (MODE == GC_FUSE_ATT) {
        // park the sampled vectors of all agents but the ego (normally the identity map) when that leaves at least
        // two ring stages; otherwise (and for tiles whose ego is not the identity) AttFusion takes two passes
        const long long park = (long long)(n_bound - 1) * C * C_::P;
        if (cap - scratch - park >= 2ll * plan.slot_floats) plan.park_slots = n_bound - 1;
    }
    const long long ring = cap - scratch - (plan.park_tmem ? 0 : (long long)plan.park_slots * C * C_::P);
    long long stages = ring / plan.slot_floats;
    if (stages < 2) return 1;
    plan.stages = (int)(stages > kMaxStages ? kMaxStages : stages);

    CUtensorMap map_box, map_id;
    const long long planes = (long long)total_agents * C;
    if (!encode_map(&map_box, feat, W, H, planes, C_::BW, C_::BH, C_::CHS)) return 1;
    if (!encode_map(&map_id, feat, W, H, planes, C_::TW, C_::TH, C_::CHS)) return 1;
    auto kern = k_fuse_persist<MODE, C_>;
    static bool configured = false;   // one attribute call per instantiation
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynSmemBytes);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            set_error("k_fuse_persist: cudaFuncSetAttribute failed (%d)", (int)e);
            return (int)e;
        }
        configured = true;
    }
    const int grid = plan.n_tiles < sm_count() ? plan.n_tiles : sm_count();
    const float sqrt_c = (float)sqrt((double)C);
    kern<<<grid, C_::kThreads, kDynSmemBytes, st>>>(map_box, map_id, feat, off, theta, L, C, H, W, sqrt_c, plan, out);
    GC_LAUNCH_CHECK("k_fuse_persist");
    return GC_OK;
}

}  // namespace persist

// Returns GC_OK when the persistent tiled path was launched, 1 when the configuration is not eligible (caller
// falls back to the gather kernels), or an error code.  nmax: upper bound on the agents of any one frame.
int warp_fuse_persist(const float *feat, const int32_t *agent_offsets, int n_frames, int total_agents,
                      const double *theta, int L, int C, int H, int W, int mode, int nmax, float *out,
                      cudaStream_t st) {
    using namespace persist;
    if ((W & 3) != 0 || ((uintptr_t)feat & 15) != 0) return 1;
    if (nmax > kTileMaxN || nmax < 1) return 1;
    if ((long long)total_agents * C >= (1ll << 31)) return 1;
    // variant table (GC_FUSE_CFG=<k> overrides the default of a mode; measured on B200 in profiles/)
    int variant = -1;
    if (const char *e = getenv("GC_FUSE_CFG")) variant = atoi(e);
#define GC_LAUNCH(MODE, ...) launch<MODE, Cfg<__VA_ARGS__>>(st, feat, agent_offsets, n_frames, total_agents, theta, L, C, H, W, nmax, out)
#define GC_VARIANTS(MODE, DEFAULT)                                                  \
    switch (variant < 0 ? DEFAULT : variant) {                                      \
        case 2: return GC_LAUNCH(MODE, 16, 8, 2, 2);                                \
        case 4: return GC_LAUNCH(MODE, 16, 16, 1, 2);                               \
        case 5: return GC_LAUNCH(MODE, 16, 16, 1, 4);                               \
        case 6: return GC_LAUNCH(MODE, 16, 8, 1, 4);                                \
        default: return GC_LAUNCH(MODE, 16, 16, 1, 2);                              \
    }
    // defaults from the B200 sweep profiles/r01g_bench_fuse_cfg*.txt: 16x16 tiles, one thread per pixel; 4 channels per
    // thread and stage while the slot (n_bound boxes) leaves >= 3 stages, 2 channels for frames with more than 5 agents
    const int dflt = nmax > 5 ? 4 : 5;
    if (mode == GC_FUSE_WARP_ONLY) { GC_VARIANTS(GC_FUSE_WARP_ONLY, (nmax > 5 ? 4 : 4)) }
    if (mode == GC_FUSE_MAX) { GC_VARIANTS(GC_FUSE_MAX, dflt) }
    // AttFusion: the one-pass TMEM park needs (P / 128) * 4C <= 512 columns: 16x16 tiles up to C = 64; beyond that two
    // passes through the ring.  Variant 6 (16x8 tiles, one pass up to C = 128) measured the same as two passes on
    // 16x16 tiles at 4x128x64x128 (0.094 vs 0.097 ms, profiles/r02e_bench_fuse.txt): that shape is wave-quantisation
    // and latency bound (256 tiles on 148 SMs), not pass-count bound -- kept selectable, not the default.
    GC_VARIANTS(GC_FUSE_ATT, dflt)
#undef GC_VARIANTS
#undef GC_LAUNCH
}

}  // namespace gc
