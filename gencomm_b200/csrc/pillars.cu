// PointPillars front end for sm_100a: voxelize -> PillarVFE -> PointPillarScatter.
//
// Replaces (paths relative to /root/reference/opencood):
//   data_utils/pre_processor/sp_voxel_preprocessor.py:62-85  (spconv Point2VoxelCPU3d, CPU, sequential)
//   models/sub_modules/pillar_vfe.py:105-155 (+ PFNLayer :31-53)
//   models/sub_modules/point_pillar_scatter.py:19-76
//
// Design (DESIGN.md section 3): the spconv voxelizer is a sequential first-come algorithm; its
// result is reproduced exactly by an order-preserving parallel formulation:
//   1. k_cell_assign : cell id per point; cell_code[cell] = min point index (atomicMin).
//   2. k_pillar_count/k_pillar_assign : a point is the "first point" of its cell iff
//      cell_code[cell] == its index.  Pillar id = number of first-points with a smaller index
//      (block counts + in-block ballot scan) == spconv's creation order; ids >= max_voxels are
//      dropped exactly like spconv's `num_voxels >= max_voxels` test.
//   3. k_slot_insert : the first 32 points of a pillar in input order == the 32 smallest point
//      indices of the cell: a conserving atomicMin insertion chain over 32 slots per pillar
//      (order-independent final state -> deterministic).
//   4. k_canvas<...> : canvas-stationary writer.  One CTA owns 128 consecutive cells of one canvas
//      row, evaluates the PFN for the occupied ones (one warp per pillar, one lane per channel
//      pair, loop over the <=32 valid points only) and stores every canvas byte exactly once with
//      128-bit coalesced stores.  No memset, no pillar_features round trip.
// All of it is HBM-bound integer/byte work + ~1 kFLOP per pillar; no tensor cores.
#include <cuda_bf16.h>

#include "common.cuh"
#include "ptx.cuh"

#include <stdlib.h>
#include <string.h>

namespace gc {

using namespace ptx;

// ------------------------------------------------------------------------------------------------
// agent lookup: largest a with off[a] <= g
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int find_segment(const int32_t *__restrict__ off, int n, int g) {
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(off + mid) <= g) lo = mid; else hi = mid;
    }
    return lo;
}

struct GeomDev {
    float rmin[3];
    float voxel[3];
    int grid[3];
    int max_voxels;
    int ncell;
};

// ------------------------------------------------------------------------------------------------
// 1. cell assignment.  c_j = floor((p_j - min_j) / voxel_j) in IEEE fp32 (no FMA contraction, true
//    division) -- spconv's arithmetic, SURVEY.md App. A.1.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_cell_assign(const float4 *__restrict__ points, const int32_t *__restrict__ point_offsets, int n_agents,
              int total_points, GeomDev g, uint32_t *__restrict__ cell_code, int32_t *__restrict__ point_cell) {
    const int gi = blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= total_points) return;
    if (gi >= __ldg(point_offsets + n_agents)) { point_cell[gi] = -1; return; }
    const int a = find_segment(point_offsets, n_agents, gi);
    const float4 p = __ldg(points + gi);
    const float pv[3] = {p.x, p.y, p.z};
    int c[3];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const float f = floorf(__fdiv_rn(__fsub_rn(pv[j], g.rmin[j]), g.voxel[j]));
        ok = ok && (f >= 0.0f) && (f < (float)g.grid[j]);   // false for NaN
        c[j] = (int)f;
    }
    int cell = -1;
    if (ok) {
        cell = (c[2] * g.grid[1] + c[1]) * g.grid[0] + c[0];
        atomicMin(cell_code + (size_t)a * g.ncell + cell, (uint32_t)(gi - __ldg(point_offsets + a)));
    }
    point_cell[gi] = cell;
}

// ------------------------------------------------------------------------------------------------
// 2. pillar ranking.  grid = (blocks_per_agent, n_agents), 256 threads x 4 items = 1024 points,
//    item-major order i = blk*1024 + item*256 + tid.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool is_first_point(const int32_t *__restrict__ point_cell, const uint32_t *codes,
                                               int base, int i, int n) {
    if (i >= n) return false;
    const int c = point_cell[base + i];
    if (c < 0) return false;
    return codes[c] == (uint32_t)i;   // plain load: codes are rewritten by other CTAs of k_pillar_assign
}

__global__ void __launch_bounds__(256)
k_pillar_count(const int32_t *__restrict__ point_offsets, const int32_t *__restrict__ point_cell,
               const uint32_t *__restrict__ cell_code, int ncell, int blocks_per_agent,
               int32_t *__restrict__ block_counts) {
    const int a = blockIdx.y;
    const int base = __ldg(point_offsets + a);
    const int n = __ldg(point_offsets + a + 1) - base;
    const int i0 = blockIdx.x * 1024;
    int cnt = 0;
    if (i0 < n) {
        const uint32_t *codes = cell_code + (size_t)a * ncell;
#pragma unroll
        for (int it = 0; it < 4; ++it)
            cnt += is_first_point(point_cell, codes, base, i0 + it * 256 + threadIdx.x, n) ? 1 : 0;
    }
    const int total = __syncthreads_count(cnt & 1) + 2 * __syncthreads_count(cnt & 2) + 4 * __syncthreads_count(cnt & 4);
    if (threadIdx.x == 0) block_counts[(size_t)a * blocks_per_agent + blockIdx.x] = total;
}

__global__ void __launch_bounds__(256)
k_pillar_assign(const int32_t *__restrict__ point_offsets, const int32_t *__restrict__ point_cell,
                uint32_t *__restrict__ cell_code, int ncell, int max_voxels, int blocks_per_agent,
                const int32_t *__restrict__ block_counts, uint32_t *__restrict__ slots,
                int32_t *__restrict__ pillar_cell, int32_t *__restrict__ n_pillars) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int a = blockIdx.y;
    const int base = __ldg(point_offsets + a);
    const int n = __ldg(point_offsets + a + 1) - base;
    const int i0 = blockIdx.x * 1024;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int32_t *bc = block_counts + (size_t)a * blocks_per_agent;

    if (blockIdx.x == 0 && warp == 1) {   // total number of occupied cells of this agent
        int t = 0;
        for (int k = lane; k < blocks_per_agent; k += 32) t += bc[k];
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) t += __shfl_xor_sync(0xffffffffu, t, m);
        if (lane == 0) n_pillars[a] = t < max_voxels ? t : max_voxels;
    }
    if (i0 >= n) return;   // uniform per block

    if (warp == 0) {       // exclusive prefix of the preceding blocks
        int t = 0;
        for (int k = lane; k < (int)blockIdx.x; k += 32) t += bc[k];
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) t += __shfl_xor_sync(0xffffffffu, t, m);
        if (lane == 0) s_base = t;
    }
    uint32_t *codes = cell_code + (size_t)a * ncell;
    bool flag[4];
    int cellv[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int i = i0 + it * 256 + threadIdx.x;
        flag[it] = is_first_point(point_cell, codes, base, i, n);
        cellv[it] = flag[it] ? point_cell[base + i] : -1;
    }
    __syncthreads();
    int running = s_base;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const unsigned bal = __ballot_sync(0xffffffffu, flag[it]);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const int v = s_warp[w];
            before += (w < warp) ? v : 0;
            total += v;
        }
        if (flag[it]) {
            const int pid = running + before + __popc(bal & ((1u << lane) - 1u));
            if (pid < max_voxels) {
                codes[cellv[it]] = kPillarBit | (uint32_t)pid;
                const size_t gp = (size_t)a * max_voxels + pid;
                pillar_cell[gp] = cellv[it];
                uint4 *s = reinterpret_cast<uint4 *>(slots + gp * 32);
                const uint4 e = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
#pragma unroll
                for (int k = 0; k < 8; ++k) s[k] = e;
            } else {
                codes[cellv[it]] = kDropped;
            }
        }
        running += total;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// 3. slot insertion: conserving atomicMin chain.  Each atomicMin(slot, v) leaves min(slot, v) in the
//    slot and carries max(slot, v) on, so the multiset {slots} U {carried} is invariant and the final
//    slot contents are the 32 smallest indices in ascending order, whatever the interleaving.
// ------------------------------------------------------------------------------------------------
// grid = (n_agents, chunks): blockIdx.x (fastest-scheduled) is the agent, blockIdx.y the 256-point chunk, so
// the machine sweeps every agent's points in index order.  Late (large-index) points of a crowded cell then
// find 32 smaller indices already in place and leave without a single atomic.
__global__ void __launch_bounds__(256)
k_slot_insert(const int32_t *__restrict__ point_offsets, const int32_t *__restrict__ point_cell,
              const uint32_t *__restrict__ cell_code, int ncell, int max_voxels, uint32_t *__restrict__ slots) {
    const int a = blockIdx.x;
    const int base = __ldg(point_offsets + a);
    const int i = blockIdx.y * blockDim.x + threadIdx.x;
    if (i >= __ldg(point_offsets + a + 1) - base) return;
    const int c = __ldg(point_cell + base + i);
    if (c < 0) return;
    const uint32_t code = __ldg(cell_code + (size_t)a * ncell + c);
    if (code >= kDropped) return;
    uint32_t *s = slots + ((size_t)a * max_voxels + (code & ~kPillarBit)) * 32;
    uint32_t v = (uint32_t)i;
    // The slot array is sorted ascending at every instant and its values only ever decrease, so a slot
    // observed below v stays below v and atomicMin(slot, v) there is a no-op: skip all of them.  The
    // snapshot is read through L2 (ld.cg); a stale (larger) value only skips less.
    int k0 = 0;
    const uint4 *s4 = reinterpret_cast<const uint4 *>(s);
    // ascending order: stop at the first quad that holds a slot >= v (most pillars hold a handful of points,
    // so one 16-byte read instead of the whole 128-byte row)
#pragma unroll 1
    for (int q = 0; q < 8; ++q) {
        const uint4 u = __ldcg(s4 + q);
        const int below = (u.x < v) + (u.y < v) + (u.z < v) + (u.w < v);
        k0 += below;
        if (below < 4) break;
    }
#pragma unroll 1
    for (int k = k0; k < 32; ++k) {
        const uint32_t old = atomicMin(s + k, v);
        if (old == kEmpty) break;
        v = old > v ? old : v;
        if ((k & 3) == 3 && __ldcg(s + 31) < v) break;   // 32 smaller indices already present
    }
}

// ------------------------------------------------------------------------------------------------
// 2+3 fused (the default voxelizer since round 2): pillar ranking and slot insertion in ONE pass over the
// points, k_pillar_build.  grid = (n_agents, chunks) with the agent fastest, 256 threads x IT points, item-major
// order like k_pillar_assign.  Every dependency of a block points at a block with a lower linear index of the same
// agent (the hardware dispatches blocks in linear order, the assumption every decoupled look-back scan makes):
//   a. first-point flags (cell_code[cell] == i after k_cell_assign2), block total published at once with
//      st.release into block_flags (kEmpty = not yet; cleared by k_cell_assign2) -- no dependency;
//   b. warp 0 sums the totals of all preceding blocks of the agent (ld.relaxed polls, four in flight per lane)
//      = first pillar id of the block;
//   c. first points: pillar id (creation order), pillar_cell, slot row = {i, empty x 31} -- the first point of
//      a cell is its smallest index, i.e. slot 0 for good -- one __threadfence, then kPillarBit|pid into cell_code;
//   d. every other point polls (ld.relaxed, then one __threadfence as the acquire) until its cell carries the pillar
//      bit -- published by this block or an earlier one, after step b of that block -- and runs the conserving
//      atomicMin chain of k_slot_insert.  The chains of a thread are interleaved so that their L2 round trips overlap.
// Same final workspace as k_pillar_count + k_pillar_assign + k_slot_insert, bit for bit (the chain's final
// state does not depend on the interleaving; tests/test_voxelizer_model_cpu.py walks random interleavings of the
// protocol on the CPU).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// 1'. k_cell_assign with two points per thread (two independent load -> divide -> atomic chains) that also
//     clears the look-back flags of k_pillar_build.
__global__ void __launch_bounds__(256)
k_cell_assign2(const float4 *__restrict__ points, const int32_t *__restrict__ point_offsets, int n_agents,
               int total_points, GeomDev g, uint32_t *__restrict__ cell_code, int32_t *__restrict__ point_cell,
               uint32_t *__restrict__ block_flags, int n_flags) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_flags) block_flags[t] = kEmpty;
    const int valid_points = __ldg(point_offsets + n_agents);
    float4 p[2];
    int gi[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        gi[u] = blockIdx.x * 512 + u * 256 + threadIdx.x;
        if (gi[u] < total_points && gi[u] < valid_points) p[u] = __ldg(points + gi[u]);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        if (gi[u] >= total_points) continue;
        if (gi[u] >= valid_points) { point_cell[gi[u]] = -1; continue; }
        const int a = find_segment(point_offsets, n_agents, gi[u]);
        const float pv[3] = {p[u].x, p[u].y, p[u].z};
        int c[3];
        bool ok = true;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const float f = floorf(__fdiv_rn(__fsub_rn(pv[j], g.rmin[j]), g.voxel[j]));
            ok = ok && (f >= 0.0f) && (f < (float)g.grid[j]);   // false for NaN
            c[j] = (int)f;
        }
        int cell = -1;
        if (ok) {
            cell = (c[2] * g.grid[1] + c[1]) * g.grid[0] + c[0];
            atomicMin(cell_code + (size_t)a * g.ncell + cell, (uint32_t)(gi[u] - __ldg(point_offsets + a)));
        }
        point_cell[gi[u]] = cell;
    }
}

__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// grid = (n_agents, chunks): blockIdx.x (dispatched fastest) is the agent, blockIdx.y the chunk of 256*IT points, so
// the machine sweeps every agent's points in index order (late points of a crowded cell find 32 smaller indices in
// place and leave without an atomic) and every block a block waits for -- same agent, lower chunk -- has a lower
// linear index.  IT = points per thread: more independent chains per thread, but a wider in-flight index window.
template <int IT, int NT>
__global__ void __launch_bounds__(NT)
k_pillar_build(const int32_t *__restrict__ point_offsets, const int32_t *__restrict__ point_cell,
               uint32_t *__restrict__ cell_code, int ncell, int max_voxels, int blocks_per_agent,
               uint32_t *__restrict__ block_flags, uint32_t *__restrict__ slots, int32_t *__restrict__ pillar_cell,
               int32_t *__restrict__ n_pillars) {
    constexpr int NW = NT / 32;
    __shared__ int s_warp[IT][NW];
    __shared__ int s_base;
    const int a = blockIdx.x;
    const int chunk = blockIdx.y;
    const int base = __ldg(point_offsets + a);
    const int n = __ldg(point_offsets + a + 1) - base;
    const int i0 = chunk * (NT * IT);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *codes = cell_code + (size_t)a * ncell;
    uint32_t *bf = block_flags + (size_t)a * blocks_per_agent;

    // a. flags
    int cellv[IT];
    uint32_t cv[IT];
    bool flag[IT];
    unsigned bal[IT];
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        const int i = i0 + it * NT + threadIdx.x;
        cellv[it] = i < n ? __ldg(point_cell + base + i) : -1;
    }
#pragma unroll
    for (int it = 0; it < IT; ++it) cv[it] = cellv[it] >= 0 ? __ldcg(codes + cellv[it]) : kEmpty;
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        flag[it] = cellv[it] >= 0 && cv[it] == (uint32_t)(i0 + it * NT + threadIdx.x);
        bal[it] = __ballot_sync(0xffffffffu, flag[it]);
        if (lane == 0) s_warp[it][warp] = __popc(bal[it]);
    }
    __syncthreads();
    // b. publish the block total, then look back
    if (warp == 0) {
        int total = lane < IT * NW ? (&s_warp[0][0])[lane] : 0;
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) total += __shfl_xor_sync(0xffffffffu, total, m);
        if (lane == 0) st_release_u32(bf + chunk, (uint32_t)total);
        int t = 0;
        for (int k0 = 0; k0 < chunk; k0 += 128) {   // four polls in flight per lane
            uint32_t v[4];
            bool again = true;
            while (again) {
                again = false;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int k = k0 + u * 32 + lane;
                    v[u] = k < chunk ? ld_relaxed_u32(bf + k) : 0u;
                    again = again || v[u] == kEmpty;
                }
            }
            t += (int)(v[0] + v[1] + v[2] + v[3]);
        }
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) t += __shfl_xor_sync(0xffffffffu, t, m);
        if (lane == 0) {
            s_base = t;
            if (chunk == blocks_per_agent - 1) n_pillars[a] = t + total < max_voxels ? t + total : max_voxels;
        }
    }
    __syncthreads();
    // c. first points open their pillars: rows first, one fence, then the codes
    int running = s_base;
    uint32_t newcode[IT];
    bool opened = false;
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            const int v = s_warp[it][w];
            before += (w < warp) ? v : 0;
            total += v;
        }
        if (flag[it]) {
            const int pid = running + before + __popc(bal[it] & ((1u << lane) - 1u));
            if (pid < max_voxels) {
                const size_t gp = (size_t)a * max_voxels + pid;
                pillar_cell[gp] = cellv[it];
                uint4 *s = reinterpret_cast<uint4 *>(slots + gp * 32);
                const uint4 e = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
                __stcg(s, make_uint4((uint32_t)(i0 + it * NT + threadIdx.x), kEmpty, kEmpty, kEmpty));
#pragma unroll
                for (int k = 1; k < 8; ++k) __stcg(s + k, e);
                newcode[it] = kPillarBit | (uint32_t)pid;
            } else {
                newcode[it] = kDropped;
            }
            opened = true;
        }
        running += total;
    }
    if (opened) {
        __threadfence();   // rows visible device-wide before any code that points at them
#pragma unroll
        for (int it = 0; it < IT; ++it)
            if (flag[it]) st_relaxed_u32(codes + cellv[it], newcode[it]);
    }
    // d. the other points: wait for the pillar of their cell, then insert
    bool act[IT];
    bool waiting = false;
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        act[it] = cellv[it] >= 0 && !flag[it];
        waiting = waiting || (act[it] && !(cv[it] & kPillarBit));
    }
    while (waiting) {
        waiting = false;
#pragma unroll
        for (int it = 0; it < IT; ++it)
            if (act[it] && !(cv[it] & kPillarBit)) cv[it] = ld_relaxed_u32(codes + cellv[it]);
#pragma unroll
        for (int it = 0; it < IT; ++it) waiting = waiting || (act[it] && !(cv[it] & kPillarBit));
    }
    __threadfence();       // acquire side: the rows are read after the codes
    uint32_t *srow[IT];
    uint32_t v[IT];
    int k[IT];
    uint4 q0[IT];
    uint32_t last[IT];
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        act[it] = act[it] && cv[it] < kDropped;
        srow[it] = slots + ((size_t)a * max_voxels + (cv[it] & ~kPillarBit)) * 32;
        v[it] = (uint32_t)(i0 + it * NT + threadIdx.x);
        if (act[it]) {
            q0[it] = __ldcg(reinterpret_cast<const uint4 *>(srow[it]));
            last[it] = __ldcg(srow[it] + 31);
        }
    }
    // The row is ascending at every instant and its values only decrease: a slot seen below v stays below v
    // (see k_slot_insert), so the chain may start at the number of slots seen below v.  Two round trips at most:
    // {first quad, last slot} -- a full row of smaller indices (late point of a crowded cell) or a free slot among
    // the first four (most pillars hold a handful of points) ends the search -- then the other seven quads at once.
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        k[it] = 0;
        if (!act[it]) continue;
        if (last[it] < v[it]) { act[it] = false; continue; }   // 32 smaller indices in place
        const uint4 u = q0[it];
        k[it] = (u.x < v[it]) + (u.y < v[it]) + (u.z < v[it]) + (u.w < v[it]);
        if (k[it] == 4) {
            uint4 r[7];
#pragma unroll
            for (int q = 0; q < 7; ++q) r[q] = __ldcg(reinterpret_cast<const uint4 *>(srow[it]) + 1 + q);
#pragma unroll
            for (int q = 0; q < 7; ++q)
                k[it] += (r[q].x < v[it]) + (r[q].y < v[it]) + (r[q].z < v[it]) + (r[q].w < v[it]);
            if (k[it] >= 32) act[it] = false;
        }
    }
    bool any = false;
#pragma unroll
    for (int it = 0; it < IT; ++it) any = any || act[it];
    while (any) {
        uint32_t old[IT];
#pragma unroll
        for (int it = 0; it < IT; ++it)
            if (act[it]) old[it] = atomicMin(srow[it] + k[it], v[it]);
        any = false;
#pragma unroll
        for (int it = 0; it < IT; ++it) {
            if (!act[it]) continue;
            if (old[it] == kEmpty) { act[it] = false; continue; }
            v[it] = old[it] > v[it] ? old[it] : v[it];
            if (++k[it] == 32) { act[it] = false; continue; }
            if ((k[it] & 3) == 0 && __ldcg(srow[it] + 31) < v[it]) { act[it] = false; continue; }
            any = true;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// PFN evaluation for one pillar by one warp ("kernel order", mirrored by oracle/pillar_ref.c).
// Lane l owns output channels l and l+32; lane s also holds point s of the pillar.
// ------------------------------------------------------------------------------------------------
struct PfnLane {     // packed row of the pfn table, see include/gencomm_b200.h
    float a0, a1, a2, a3, b0, b1, b2, d0, d1, d2, shift, pad;
};

__device__ __forceinline__ PfnLane load_pfn(const float *__restrict__ pfn, int ch) {
    const float4 *r = reinterpret_cast<const float4 *>(pfn + ch * 16);
    const float4 a = __ldg(r), b = __ldg(r + 1), c = __ldg(r + 2);
    PfnLane w;
    w.a0 = a.x; w.a1 = a.y; w.a2 = a.z; w.a3 = a.w;
    w.b0 = b.x; w.b1 = b.y; w.b2 = b.z; w.d0 = b.w;
    w.d1 = c.x; w.d2 = c.y; w.shift = c.z; w.pad = c.w;
    return w;
}

__device__ __forceinline__ float tree_sum(float v) {
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, m));
    return v;
}

__device__ __forceinline__ float pfn_bias(const PfnLane &w, float cx, float cy, float cz, float mx, float my, float mz) {
    float b = __fmaf_rn(w.b0, cx, w.shift);
    b = __fmaf_rn(w.b1, cy, b);
    b = __fmaf_rn(w.b2, cz, b);
    b = __fmaf_rn(w.d0, mx, b);
    b = __fmaf_rn(w.d1, my, b);
    b = __fmaf_rn(w.d2, mz, b);
    return b;
}

__device__ __forceinline__ float pfn_point(const PfnLane &w, float xr, float yr, float zr, float pi) {
    float acc = __fmaf_rn(w.a2, zr, __fmul_rn(w.a3, pi));
    acc = __fmaf_rn(w.a1, yr, acc);
    return __fmaf_rn(w.a0, xr, acc);
}

__device__ __forceinline__ float pfn_finish(const PfnLane &w, float best, float b, int n) {
    float o = fmaxf(__fadd_rn(best, b), 0.0f);
    if (n < 32) o = fmaxf(o, w.pad);   // padded slots contribute relu(bn(0)) = max(shift, 0), pillar_vfe.py:46
    return o;
}

// p: this lane's point (ignored when lane >= n); returns the two channel maxima of the pillar.
// stage: 32 float4 of shared memory private to the calling warp.  The decorated points are exchanged through it
// (one broadcast LDS.128 per point instead of four shuffles); arithmetic and order are unchanged.
__device__ __forceinline__ float2 pfn_pillar(const PfnLane &wa, const PfnLane &wb, float4 p, int n, float cx,
                                             float cy, float cz, float4 *__restrict__ stage) {
    const int lane = threadIdx.x & 31;
    const bool valid = lane < n;
    const float xr = valid ? __fsub_rn(p.x, cx) : 0.0f;
    const float yr = valid ? __fsub_rn(p.y, cy) : 0.0f;
    const float zr = valid ? __fsub_rn(p.z, cz) : 0.0f;
    const float pi = valid ? p.w : 0.0f;
    __syncwarp();                                   // every lane is done reading the previous pillar's points
    stage[lane] = make_float4(xr, yr, zr, pi);
    const float inv_n = __frcp_rn((float)n);
    const float mx = __fmul_rn(tree_sum(xr), inv_n);
    const float my = __fmul_rn(tree_sum(yr), inv_n);
    const float mz = __fmul_rn(tree_sum(zr), inv_n);
    const float ba = pfn_bias(wa, cx, cy, cz, mx, my, mz);
    const float bb = pfn_bias(wb, cx, cy, cz, mx, my, mz);
    float best_a = -INFINITY, best_b = -INFINITY;
    __syncwarp();                                   // staged points visible to the whole warp
#pragma unroll 4
    for (int s = 0; s < n; ++s) {
        const float4 q = stage[s];
        best_a = fmaxf(best_a, pfn_point(wa, q.x, q.y, q.z, q.w));
        best_b = fmaxf(best_b, pfn_point(wb, q.x, q.y, q.z, q.w));
    }
    return make_float2(pfn_finish(wa, best_a, ba, n), pfn_finish(wb, best_b, bb, n));
}

// ------------------------------------------------------------------------------------------------
// Standalone PillarVFE on reference-shaped voxel tensors: one warp per pillar.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_pillar_vfe(const float4 *__restrict__ voxels, const int32_t *__restrict__ num_points,
             const int4 *__restrict__ coords, int n_pillars, const float *__restrict__ pfn, float vx, float vy,
             float vz, float ox, float oy, float oz, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (m >= n_pillars) return;   // warp-uniform
    const PfnLane wa = load_pfn(pfn, lane), wb = load_pfn(pfn, lane + 32);
    int n = __ldg(num_points + m);
    n = n < 0 ? 0 : (n > 32 ? 32 : n);
    const int4 c = __ldg(coords + m);   // (b, z, y, x)
    const float cx = __fadd_rn(__fmul_rn((float)c.w, vx), ox);
    const float cy = __fadd_rn(__fmul_rn((float)c.z, vy), oy);
    const float cz = __fadd_rn(__fmul_rn((float)c.y, vz), oz);
    __shared__ float4 s_stage[8][32];
    const float4 p = __ldg(voxels + (size_t)m * 32 + lane);
    const float2 r = pfn_pillar(wa, wb, p, n, cx, cy, cz, s_stage[threadIdx.x >> 5]);
    out[(size_t)m * 64 + lane] = r.x;
    out[(size_t)m * 64 + lane + 32] = r.y;
}

// ------------------------------------------------------------------------------------------------
// Reference-shaped voxel tensors out of the workspace (SpVoxelPreprocessor.preprocess + collate).
// One warp per (compact) pillar.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_voxel_gather(const float4 *__restrict__ points, const int32_t *__restrict__ point_offsets, int n_agents,
               GeomDev g, const uint32_t *__restrict__ slots, const int32_t *__restrict__ pillar_cell,
               const int32_t *__restrict__ pillar_offsets, int total_pillars, float4 *__restrict__ voxels,
               int4 *__restrict__ coords, int32_t *__restrict__ num_points) {
    const int lane = threadIdx.x & 31;
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (m >= total_pillars) return;
    const int a = find_segment(pillar_offsets, n_agents, m);
    const size_t gp = (size_t)a * g.max_voxels + (m - __ldg(pillar_offsets + a));
    const uint32_t idx = __ldg(slots + gp * 32 + lane);
    const bool valid = idx != kEmpty;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) p = __ldg(points + __ldg(point_offsets + a) + idx);
    voxels[(size_t)m * 32 + lane] = p;
    const unsigned bal = __ballot_sync(0xffffffffu, valid);
    if (lane == 0) {
        const int cell = __ldg(pillar_cell + gp);
        const int x = cell % g.grid[0];
        const int y = (cell / g.grid[0]) % g.grid[1];
        const int z = cell / (g.grid[0] * g.grid[1]);
        coords[m] = make_int4(a, z, y, x);
        num_points[m] = __popc(bal);
    }
}

// ------------------------------------------------------------------------------------------------
// 4. canvas-stationary writer.  grid = (ceil(nx/128), ny, n_batch), 256 threads.
//    Src::occupied(code) / Src::features(...) select between
//      FeatSrc  : pillar_features rows looked up through a dense cell->row map   (PointPillarScatter)
//      FusedSrc : PFN evaluated from the voxelizer workspace                     (fused front end)
// ------------------------------------------------------------------------------------------------
constexpr int kTileX = 128;
constexpr int kTileStride = kTileX + 4;   // floats; keeps rows 16-byte aligned

struct FeatSrc {
    const float *feat;        // [M][C]
    const int32_t *cell_map;  // [n_batch][ny*nx], -1 = empty
    int C;
    static constexpr bool kFused = false;
    __device__ __forceinline__ int code(int b, int cell, int ncell) const {
        return __ldg(cell_map + (size_t)b * ncell + cell);
    }
    __device__ __forceinline__ static bool occupied(int code) { return code >= 0; }
};

struct FusedSrc {
    const float4 *points;
    const int32_t *point_offsets;
    const uint32_t *cell_code;
    const uint32_t *slots;
    const float *pfn;
    int max_voxels;
    float vx, vy, ox, oy, cz;   // cz = centre of z-cell 0
    static constexpr bool kFused = true;
    __device__ __forceinline__ int code(int b, int cell, int ncell) const {
        return (int)__ldg(cell_code + (size_t)b * ncell + cell);
    }
    // kPillarBit|pid is a negative int below kDropped (-2) and kEmpty (-1)
    __device__ __forceinline__ static bool occupied(int code) { return code < -2; }
};

template <class Src>
__global__ void __launch_bounds__(256, 4)
k_canvas(Src src, int nx, int ny, int C, float *__restrict__ canvas) {
    __shared__ __align__(16) float tile[64 * kTileStride];
    __shared__ int s_code[kTileX];
    __shared__ int s_list[kTileX];
    __shared__ unsigned s_mask[4];
    __shared__ float4 s_stage[8][32];   // per-warp point exchange of pfn_pillar

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int x0 = blockIdx.x * kTileX, y = blockIdx.y, b = blockIdx.z;
    const int ncell = nx * ny;

    if (t < kTileX) {
        const int x = x0 + t;
        const int code = (x < nx) ? src.code(b, y * nx + x, ncell) : -1;
        const bool occ = (x < nx) && Src::occupied(code);
        s_code[t] = code;
        const unsigned bal = __ballot_sync(0xffffffffu, occ);
        if (lane == 0) s_mask[warp] = bal;
    }
    __syncthreads();
    const unsigned m0 = s_mask[0], m1 = s_mask[1], m2 = s_mask[2], m3 = s_mask[3];
    const int n_occ = __popc(m0) + __popc(m1) + __popc(m2) + __popc(m3);
    if (t < kTileX) {
        const unsigned mine = warp == 0 ? m0 : warp == 1 ? m1 : warp == 2 ? m2 : m3;
        if ((mine >> lane) & 1u) {
            int pos = __popc(mine & ((1u << lane) - 1u));
            pos += (warp > 0 ? __popc(m0) : 0) + (warp > 1 ? __popc(m1) : 0) + (warp > 2 ? __popc(m2) : 0);
            s_list[pos] = t;
        }
    }
    __syncthreads();

    const bool vec_ok = (nx & 3) == 0;
    const size_t plane = (size_t)ny * nx;

    for (int c0 = 0; c0 < C; c0 += 64) {
        // the tile starts as zeros (empty cells); the load phase overwrites the occupied columns, so the store
        // phase is a plain shared -> global copy (no per-quad occupancy selects)
        {
            float4 *t4 = reinterpret_cast<float4 *>(tile);
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = t; i < 64 * kTileStride / 4; i += 256) t4[i] = z;
        }
        __syncthreads();
        // ---- load phase: one warp per occupied cell -------------------------------------------
        if constexpr (!Src::kFused) {
            const Src &fs = src;
            for (int k = warp; k < n_occ; k += 8) {
                const int xc = s_list[k];
                const float *row = fs.feat + (size_t)s_code[xc] * C + c0;
                if (c0 + lane < C) tile[lane * kTileStride + xc] = __ldg(row + lane);
                if (c0 + lane + 32 < C) tile[(lane + 32) * kTileStride + xc] = __ldg(row + lane + 32);
            }
        } else {
            const Src &fs = src;
            if (warp < n_occ) {   // warp-uniform; skips the weight loads for empty tiles
                const PfnLane wa = load_pfn(fs.pfn, lane), wb = load_pfn(fs.pfn, lane + 32);
                const int pbase = __ldg(fs.point_offsets + b);
                const float cy = __fadd_rn(__fmul_rn((float)y, fs.vy), fs.oy);
                // two-stage software pipeline over this warp's pillars: slot indices two ahead, point one ahead
                auto slot_of = [&](int k) -> uint32_t {
                    const unsigned pid = (unsigned)s_code[s_list[k]] & ~kPillarBit;
                    return __ldg(fs.slots + ((size_t)b * fs.max_voxels + pid) * 32 + lane);
                };
                auto point_of = [&](uint32_t idx) -> float4 {
                    return idx != kEmpty ? __ldg(fs.points + pbase + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
                };
                uint32_t idx_cur = slot_of(warp);
                uint32_t idx_nxt = (warp + 8 < n_occ) ? slot_of(warp + 8) : kEmpty;
                float4 p_cur = point_of(idx_cur);
                for (int k = warp; k < n_occ; k += 8) {
                    const float4 p_nxt = point_of(idx_nxt);
                    const uint32_t idx_nxt2 = (k + 16 < n_occ) ? slot_of(k + 16) : kEmpty;
                    const int xc = s_list[k];
                    const int n = __popc(__ballot_sync(0xffffffffu, idx_cur != kEmpty));   // slots fill from 0
                    const float cx = __fadd_rn(__fmul_rn((float)(x0 + xc), fs.vx), fs.ox);
                    const float2 r = pfn_pillar(wa, wb, p_cur, n, cx, cy, fs.cz, s_stage[warp]);
                    tile[lane * kTileStride + xc] = r.x;
                    tile[(lane + 32) * kTileStride + xc] = r.y;
                    idx_cur = idx_nxt; p_cur = p_nxt; idx_nxt = idx_nxt2;
                }
            }
        }
        __syncthreads();
        // ---- store phase: every canvas byte of the tile exactly once ---------------------------
        {
            const int x = x0 + 4 * lane;
            float *dst = canvas + ((size_t)b * C + c0 + warp) * plane + (size_t)y * nx + x;
            const float4 *src4 = reinterpret_cast<const float4 *>(tile + warp * kTileStride) + lane;
            if (vec_ok && x + 3 < nx) {
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    if (c0 + it * 8 + warp < C) *reinterpret_cast<float4 *>(dst + (size_t)it * 8 * plane) = src4[it * 8 * (kTileStride / 4)];
                }
            } else {
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    if (c0 + it * 8 + warp >= C) continue;
                    const float4 v = src4[it * 8 * (kTileStride / 4)];
                    float *d = dst + (size_t)it * 8 * plane;
                    if (x < nx) d[0] = v.x;
                    if (x + 1 < nx) d[1] = v.y;
                    if (x + 2 < nx) d[2] = v.z;
                    if (x + 3 < nx) d[3] = v.w;
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// 4a'. the same canvas written as channel-last bf16 value + residual planes ([A][ny*nx][64] each): the operand layout of the
// backbone's tensor-core convolutions.  When PointPillar feeds this package's BaseBEVBackbone the fp32 NCHW canvas (1.07 GB
// for 32 agents at 512 x 256) is never written and never converted (k_me_to_nhwc: 1.07 GB read + 1.07 GB written).  Same
// values: the planes are bf16(x) and bf16(x - bf16(x)) of the fp32 feature k_canvas would have stored.
// The tile is kept pixel-major in shared memory; a pixel's 64 channels are 128 contiguous bytes per plane and the 128 pixels
// of the tile are contiguous in global memory, so every store instruction writes 512 contiguous bytes.
// ------------------------------------------------------------------------------------------------
constexpr int kPlaneTileStride = GC_PFN_OUT + 4;   // floats per pixel row of the tile (16-byte aligned, bank-skewed)

// SPARSE: the planes are all-zero on entry (the caller keeps them so: gc_pillar_canvas_planes_sparse + gc_planes_clear_occupied),
// only the occupied cells are written -- 16 % of the cells of a 100 k-point cloud on the 512 x 256 grid -- and a tile without
// a pillar ends after its code load.
template <bool SPARSE>
__global__ void __launch_bounds__(256, 4)
k_canvas_planes(FusedSrc src, int nx, int ny, uint4 *__restrict__ xh, uint4 *__restrict__ xl) {
    __shared__ __align__(16) float tile[kTileX * kPlaneTileStride];
    __shared__ int s_code[kTileX];
    __shared__ int s_list[kTileX];
    __shared__ unsigned s_mask[4];
    __shared__ float4 s_stage[8][32];   // per-warp point exchange of pfn_pillar

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int x0 = blockIdx.x * kTileX, y = blockIdx.y, b = blockIdx.z;
    const int ncell = nx * ny;

    if (t < kTileX) {
        const int x = x0 + t;
        const int code = (x < nx) ? src.code(b, y * nx + x, ncell) : -1;
        const bool occ = (x < nx) && FusedSrc::occupied(code);
        s_code[t] = code;
        const unsigned bal = __ballot_sync(0xffffffffu, occ);
        if (lane == 0) s_mask[warp] = bal;
    }
    // (no zero fill of the tile: an occupied cell's 64 channels are all written by its warp, empty cells are stored as zeros
    // straight from registers -- 84 % of the cells at 100 k points per 512 x 256 grid)
    __syncthreads();
    const unsigned m0 = s_mask[0], m1 = s_mask[1], m2 = s_mask[2], m3 = s_mask[3];
    const int n_occ = __popc(m0) + __popc(m1) + __popc(m2) + __popc(m3);
    if (SPARSE && n_occ == 0) return;   // block-uniform
    if (t < kTileX) {
        const unsigned mine = warp == 0 ? m0 : warp == 1 ? m1 : warp == 2 ? m2 : m3;
        if ((mine >> lane) & 1u) {
            int pos = __popc(mine & ((1u << lane) - 1u));
            pos += (warp > 0 ? __popc(m0) : 0) + (warp > 1 ? __popc(m1) : 0) + (warp > 2 ? __popc(m2) : 0);
            s_list[pos] = t;
        }
    }
    __syncthreads();
    if (warp < n_occ) {   // warp-uniform; one warp per occupied cell, the software pipeline of k_canvas<FusedSrc>
        const FusedSrc &fs = src;
        const PfnLane wa = load_pfn(fs.pfn, lane), wb = load_pfn(fs.pfn, lane + 32);
        const int pbase = __ldg(fs.point_offsets + b);
        const float cy = __fadd_rn(__fmul_rn((float)y, fs.vy), fs.oy);
        auto slot_of = [&](int k) -> uint32_t {
            const unsigned pid = (unsigned)s_code[s_list[k]] & ~kPillarBit;
            return __ldg(fs.slots + ((size_t)b * fs.max_voxels + pid) * 32 + lane);
        };
        auto point_of = [&](uint32_t idx) -> float4 {
            return idx != kEmpty ? __ldg(fs.points + pbase + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        uint32_t idx_cur = slot_of(warp);
        uint32_t idx_nxt = (warp + 8 < n_occ) ? slot_of(warp + 8) : kEmpty;
        float4 p_cur = point_of(idx_cur);
        for (int k = warp; k < n_occ; k += 8) {
            const float4 p_nxt = point_of(idx_nxt);
            const uint32_t idx_nxt2 = (k + 16 < n_occ) ? slot_of(k + 16) : kEmpty;
            const int xc = s_list[k];
            const int n = __popc(__ballot_sync(0xffffffffu, idx_cur != kEmpty));   // slots fill from 0
            const float cx = __fadd_rn(__fmul_rn((float)(x0 + xc), fs.vx), fs.ox);
            const float2 r = pfn_pillar(wa, wb, p_cur, n, cx, cy, fs.cz, s_stage[warp]);
            tile[xc * kPlaneTileStride + lane] = r.x;
            tile[xc * kPlaneTileStride + lane + 32] = r.y;
            idx_cur = idx_nxt; p_cur = p_nxt; idx_nxt = idx_nxt2;
        }
    }
    __syncthreads();
    // ---- store phase: item = (pixel, 8-channel group); eight lanes write one pixel's 128 bytes, a warp four pixels ----
    const size_t row = ((size_t)b * ncell + (size_t)y * nx + x0) * (GC_PFN_OUT / 8);
#pragma unroll
    for (int it = 0; it < kTileX * (GC_PFN_OUT / 8) / 256; ++it) {
        const int i = it * 256 + t, px = i / (GC_PFN_OUT / 8), g = i % (GC_PFN_OUT / 8);
        if (x0 + px >= nx) continue;
        if (!FusedSrc::occupied(s_code[px])) {
            if (!SPARSE) {
                xh[row + (size_t)i] = make_uint4(0u, 0u, 0u, 0u);
                xl[row + (size_t)i] = make_uint4(0u, 0u, 0u, 0u);
            }
            continue;
        }
        const float4 a = *reinterpret_cast<const float4 *>(tile + px * kPlaneTileStride + g * 8);
        const float4 c = *reinterpret_cast<const float4 *>(tile + px * kPlaneTileStride + g * 8 + 4);
        const float v[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const __nv_bfloat162 hh = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
            const __nv_bfloat162 ll = __floats2bfloat162_rn(v[2 * j] - __bfloat162float(hh.x), v[2 * j + 1] - __bfloat162float(hh.y));
            h[j] = *reinterpret_cast<const uint32_t *>(&hh);
            l[j] = *reinterpret_cast<const uint32_t *>(&ll);
        }
        xh[row + (size_t)i] = make_uint4(h[0], h[1], h[2], h[3]);
        xl[row + (size_t)i] = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// Pillar-centric writer of the sparse planes: no tiles, no block barriers.  With the empty cells already zero the canvas
// geometry is irrelevant: warp w of agent a walks the pillars w, w + stride, ... of the agent (creation order = the order of
// their slot rows), software-pipelined like the tile writers (slot row and cell two pillars ahead, points one ahead), and
// stores a pillar's 64 channels as one 128-byte line per plane.  (k_canvas_planes<true> was bound by its per-tile chain
// code load -> barrier -> slot row -> points -> PFN -> barrier -> store at four CTAs per SM: skipping 84 % of the stores
// took only 0.75 -> 0.64 ms off it, profiles/r02bi_step_ab.txt.)
// grid = (blocks per agent, n_agents), 256 threads.
__global__ void __launch_bounds__(256)
k_pillar_planes_sparse(FusedSrc src, const int32_t *__restrict__ pillar_cell, const int32_t *__restrict__ n_pillars, int nx,
                       int ncell, uint32_t *__restrict__ xh, uint32_t *__restrict__ xl) {
    __shared__ float4 s_stage[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, a = blockIdx.y;
    const int np = __ldg(n_pillars + a);
    const int stride = gridDim.x * 8;
    int pid = blockIdx.x * 8 + warp;
    if (pid >= np) return;   // warp-uniform
    const PfnLane wa = load_pfn(src.pfn, lane), wb = load_pfn(src.pfn, lane + 32);
    const int pbase = __ldg(src.point_offsets + a);
    const size_t prow = (size_t)a * src.max_voxels;
    auto slot_of = [&](int q) -> uint32_t { return q < np ? __ldg(src.slots + (prow + q) * 32 + lane) : kEmpty; };
    auto cell_of = [&](int q) -> int { return q < np ? __ldg(pillar_cell + prow + q) : 0; };
    auto point_of = [&](uint32_t idx) -> float4 {
        return idx != kEmpty ? __ldg(src.points + pbase + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    uint32_t idx_cur = slot_of(pid), idx_nxt = slot_of(pid + stride);
    int cell_cur = cell_of(pid), cell_nxt = cell_of(pid + stride);
    float4 p_cur = point_of(idx_cur);
    const int src_lane = 2 * (lane & 15);
    for (; pid < np; pid += stride) {
        const float4 p_nxt = point_of(idx_nxt);
        const uint32_t idx_nxt2 = slot_of(pid + 2 * stride);
        const int cell_nxt2 = cell_of(pid + 2 * stride);
        const int n = __popc(__ballot_sync(0xffffffffu, idx_cur != kEmpty));   // slots fill from 0
        const int y = cell_cur / nx, x = cell_cur - y * nx;
        const float cx = __fadd_rn(__fmul_rn((float)x, src.vx), src.ox);
        const float cy = __fadd_rn(__fmul_rn((float)y, src.vy), src.oy);
        const float2 r = pfn_pillar(wa, wb, p_cur, n, cx, cy, src.cz, s_stage[warp]);
        // lane l holds channels l and l + 32; word j of the pixel's 128-byte line = channels 2j, 2j + 1
        const float a0 = __shfl_sync(0xffffffffu, r.x, src_lane), a1 = __shfl_sync(0xffffffffu, r.x, src_lane + 1);
        const float b0 = __shfl_sync(0xffffffffu, r.y, src_lane), b1 = __shfl_sync(0xffffffffu, r.y, src_lane + 1);
        const float v0 = lane < 16 ? a0 : b0, v1 = lane < 16 ? a1 : b1;
        const __nv_bfloat162 hh = __floats2bfloat162_rn(v0, v1);
        const __nv_bfloat162 ll = __floats2bfloat162_rn(v0 - __bfloat162float(hh.x), v1 - __bfloat162float(hh.y));
        const size_t o = ((size_t)a * ncell + cell_cur) * (GC_PFN_OUT / 2) + lane;
        xh[o] = *reinterpret_cast<const uint32_t *>(&hh);
        xl[o] = *reinterpret_cast<const uint32_t *>(&ll);
        idx_cur = idx_nxt; p_cur = p_nxt; idx_nxt = idx_nxt2;
        cell_cur = cell_nxt; cell_nxt = cell_nxt2;
    }
}

// Zeroes the cells gc_pillar_canvas_planes_sparse wrote (the workspace still holds the pillar list): eight threads per
// pillar, one 16-byte vector per plane each.  grid = (ceil(max_voxels * 8 / 256), n_agents).
__global__ void __launch_bounds__(256)
k_planes_clear(const int32_t *__restrict__ pillar_cell, const int32_t *__restrict__ n_pillars, int max_voxels, int ncell,
               uint4 *__restrict__ xh, uint4 *__restrict__ xl) {
    const int a = blockIdx.y, t = blockIdx.x * 256 + threadIdx.x, pid = t >> 3;
    if (pid >= __ldg(n_pillars + a)) return;
    const int cell = __ldg(pillar_cell + (size_t)a * max_voxels + pid);
    const size_t o = ((size_t)a * ncell + cell) * (GC_PFN_OUT / 8) + (t & 7);
    xh[o] = make_uint4(0u, 0u, 0u, 0u);
    xl[o] = make_uint4(0u, 0u, 0u, 0u);
}

__device__ __forceinline__ float2 dup2(float v) { return make_float2(v, v); }

// ------------------------------------------------------------------------------------------------
// 4b. persistent canvas writer for the fused front end (round-1q; the default for nx % 4 == 0).
//
//     What ncu said about k_canvas<FusedSrc> (profiles/r01l): issue slots 57 % busy, stalls = the three
//     CTA barriers per tile (zero -> PFN -> store) + the serial tail of the most crowded warp; ~220 warp
//     instructions per pillar.  This version removes the block-wide barriers and halves the instructions:
//       * one persistent CTA of 8 PFN warps + 1 store warp; two 64 x 128 tiles in shared memory.
//       * PFN warps never synchronise with each other: warp w owns the cells {4(w+8i)+j} of every tile, takes
//         them from a register-resident list (one 16-byte code load per lane and tile, prefetched a tile ahead)
//         and runs a pillar pipeline that crosses tile boundaries (slot row two pillars ahead, points one ahead).
//         A warp only waits when it is a whole tile ahead of the store warp (mbarrier full/empty pair per tile).
//       * the store warp ships a finished tile with 64 row-wise bulk copies shared -> global
//         (cp.async.bulk, 512 B per channel row, every canvas byte written exactly once), waits for the
//         shared-memory reads only, re-zeroes the tile if a pillar was written into it and hands it back.
//       * the PFN arithmetic is unchanged (bit-exact against oracle/pillar_ref.c) but issued as packed
//         fp32 pairs (FFMA2/FMUL2/FADD2, sm_100): two points per instruction, the pillar's points staged
//         component-wise so one LDS.128 yields two aligned register pairs; padded lanes duplicate point 0
//         (max unchanged), so the loop has no tail; the xor-tree of the mean skips the levels whose
//         partners are all padded zeros (x + 0 is exact).
// ------------------------------------------------------------------------------------------------
constexpr int kCvTileFloats = 64 * kTileX;   // four 128B-swizzled TMA boxes of [64 channels][32 cells]


template <int W, int NB, bool PAIR>
struct CvSmem {
    static constexpr int kCvLists = NB >= 4 ? 8 : 4;   // cell-list ring depth (> NB: lists are built ahead of the tiles)
    float tile[NB][kCvTileFloats];   // must stay first: every box is 1024-byte aligned
    float stage[W][PAIR ? 2 : 1][4][32];   // x, y, z, intensity rows of the pillar(s) being evaluated
    uint2 list[kCvLists][kTileX];    // (slot row, x | y << 16) of the occupied cells of a tile
    int list_n[kCvLists];            // number of entries
    int list_pbase[kCvLists];        // first point of the tile's agent
    int list_take[kCvLists];         // next entry to hand out (atomic)
    float inv_n[36];                 // 1 / n, correctly rounded
    float4 pfn_bd[16][7];            // PAIR: (B0,B1,B2,D0,D1,D2,shift) x channels hl + 16 j of half-lane hl
    unsigned long long full[NB], empty[NB], ready[kCvLists];
    int dirty[NB];
};

struct PfnPacked {
    float a0a, a1a, a2a, a3a;    // channel `lane`      (FFMA2 takes a scalar multiplier for both halves)
    float a0b, a1b, a2b, a3b;    // channel `lane + 32`
    float2 b0, b1, b2, d0, d1, d2, shift;   // (channel lane, channel lane + 32)
};

__device__ __forceinline__ PfnPacked pack_pfn(const PfnLane &wa, const PfnLane &wb) {
    PfnPacked w;
    w.a0a = wa.a0; w.a1a = wa.a1; w.a2a = wa.a2; w.a3a = wa.a3;
    w.a0b = wb.a0; w.a1b = wb.a1; w.a2b = wb.a2; w.a3b = wb.a3;
    w.b0 = make_float2(wa.b0, wb.b0); w.b1 = make_float2(wa.b1, wb.b1); w.b2 = make_float2(wa.b2, wb.b2);
    w.d0 = make_float2(wa.d0, wb.d0); w.d1 = make_float2(wa.d1, wb.d1); w.d2 = make_float2(wa.d2, wb.d2);
    w.shift = make_float2(wa.shift, wb.shift);
    return w;
}


// Same roundings, same order as pfn_pillar().  p = this lane's point for lane < n, a copy of point 0 otherwise.
__device__ __forceinline__ float2 pfn_pillar_packed(const PfnPacked &w, float4 p, int n, float inv_n, float cx,
                                                    float cy, float cz, float *__restrict__ stage, int lane) {
    const float xr = __fsub_rn(p.x, cx), yr = __fsub_rn(p.y, cy), zr = __fsub_rn(p.z, cz);
    __syncwarp();                                   // the previous pillar's stage reads are done
    stage[lane] = xr;
    stage[32 + lane] = yr;
    stage[64 + lane] = zr;
    stage[96 + lane] = p.w;
    const bool valid = lane < n;
    float sx = valid ? xr : 0.0f, sy = valid ? yr : 0.0f, sz = valid ? zr : 0.0f;
    // xor-butterfly over the 32 slots, the oracle's order (skipping the all-zero upper levels of small pillars was
    // measured: the uniform branches + the final broadcast cost more instructions than the levels they save)
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        sx = __fadd_rn(sx, __shfl_xor_sync(0xffffffffu, sx, m));
        sy = __fadd_rn(sy, __shfl_xor_sync(0xffffffffu, sy, m));
        sz = __fadd_rn(sz, __shfl_xor_sync(0xffffffffu, sz, m));
    }
    float2 bias = __ffma2_rn(w.b0, dup2(cx), w.shift);
    bias = __ffma2_rn(w.b1, dup2(cy), bias);
    bias = __ffma2_rn(w.b2, dup2(cz), bias);
    bias = __ffma2_rn(w.d0, dup2(__fmul_rn(sx, inv_n)), bias);
    bias = __ffma2_rn(w.d1, dup2(__fmul_rn(sy, inv_n)), bias);
    bias = __ffma2_rn(w.d2, dup2(__fmul_rn(sz, inv_n)), bias);
    float best_a = -INFINITY, best_b = -INFINITY;
    __syncwarp();                                   // staged points visible to the whole warp
    const float4 *s4 = reinterpret_cast<const float4 *>(stage);
    for (int q = 0; q * 4 < n; ++q) {
        const float4 X = s4[q], Y = s4[8 + q], Z = s4[16 + q], I = s4[24 + q];
        float2 u, v;
        u = __fmul2_rn(dup2(w.a3a), make_float2(I.x, I.y));
        v = __fmul2_rn(dup2(w.a3a), make_float2(I.z, I.w));
        u = __ffma2_rn(dup2(w.a2a), make_float2(Z.x, Z.y), u);
        v = __ffma2_rn(dup2(w.a2a), make_float2(Z.z, Z.w), v);
        u = __ffma2_rn(dup2(w.a1a), make_float2(Y.x, Y.y), u);
        v = __ffma2_rn(dup2(w.a1a), make_float2(Y.z, Y.w), v);
        u = __ffma2_rn(dup2(w.a0a), make_float2(X.x, X.y), u);
        v = __ffma2_rn(dup2(w.a0a), make_float2(X.z, X.w), v);
        best_a = fmaxf(fmaxf(best_a, u.x), u.y);
        best_a = fmaxf(fmaxf(best_a, v.x), v.y);
        u = __fmul2_rn(dup2(w.a3b), make_float2(I.x, I.y));
        v = __fmul2_rn(dup2(w.a3b), make_float2(I.z, I.w));
        u = __ffma2_rn(dup2(w.a2b), make_float2(Z.x, Z.y), u);
        v = __ffma2_rn(dup2(w.a2b), make_float2(Z.z, Z.w), v);
        u = __ffma2_rn(dup2(w.a1b), make_float2(Y.x, Y.y), u);
        v = __ffma2_rn(dup2(w.a1b), make_float2(Y.z, Y.w), v);
        u = __ffma2_rn(dup2(w.a0b), make_float2(X.x, X.y), u);
        v = __ffma2_rn(dup2(w.a0b), make_float2(X.z, X.w), v);
        best_b = fmaxf(fmaxf(best_b, u.x), u.y);
        best_b = fmaxf(fmaxf(best_b, v.x), v.y);
    }
    const float2 o = __fadd2_rn(make_float2(best_a, best_b), bias);
    // relu, and for n < 32 the padded slots' relu(bn(0)) = max(shift, 0):  max(max(o,0), max(shift,0)) = max3(o, 0, shift)
    float oa = fmaxf(o.x, 0.0f), ob = fmaxf(o.y, 0.0f);
    if (n < 32) { oa = fmaxf(oa, w.shift.x); ob = fmaxf(ob, w.shift.y); }
    return make_float2(oa, ob);
}

// tile sequence of one CTA: T_i = blockIdx.x + i * gridDim.x, walked incrementally (no divisions per tile);
// the step gridDim.x is decomposed into (sb, sy, stx) once on the host
struct CvStep { int sb, sy, stx; };
struct CvTile {
    int b, y, tx;
    __device__ __forceinline__ void init(int T, int ny, int tiles_x) {
        tx = T % tiles_x; const int r = T / tiles_x; y = r % ny; b = r / ny;
    }
    __device__ __forceinline__ void advance(const CvStep &s, int ny, int tiles_x) {
        tx += s.stx;
        if (tx >= tiles_x) { tx -= tiles_x; ++y; }
        y += s.sy;
        if (y >= ny) { y -= ny; ++b; }
        b += s.sb;
    }
};

struct CvEnt { int i; int xy; int pbase; };        // i < 0: end of stream
struct CvSlot { CvEnt e; uint32_t idx; float4 p; };   // one pillar in flight

template <int W, int NB, int MINB, bool PAIR, bool PIPE>
__global__ void __launch_bounds__((W + 1) * 32, MINB)
k_canvas_persist(const __grid_constant__ CUtensorMap tmap, const FusedSrc src, const int nx, const int ny,
                 const int n_agents, const CvStep step) {
    using Smem = CvSmem<W, NB, PAIR>;
    constexpr int kCvLists = Smem::kCvLists;
    constexpr int kThreads = (W + 1) * 32;
    static_assert(kCvLists > NB && (kCvLists & (kCvLists - 1)) == 0, "list ring");
    extern __shared__ __align__(1024) unsigned char cv_smem_raw[];   // 1024-byte alignment: swizzled TMA boxes
    Smem &sm = *reinterpret_cast<Smem *>(cv_smem_raw);
    if ((smem_u32(cv_smem_raw) & 1023u) != 0u) __trap();
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int tiles_x = (nx + kTileX - 1) / kTileX;
    const int total_tiles = n_agents * ny * tiles_x;
    const int n_my = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // >= 1 (grid <= tiles)

    {
        float4 *t4 = reinterpret_cast<float4 *>(&sm.tile[0][0]);
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i = t; i < NB * kCvTileFloats / 4; i += kThreads) t4[i] = z;
    }
    if (t < 36) sm.inv_n[t] = __frcp_rn((float)t);
    if (PAIR && t < 16) {
        const PfnLane q0 = load_pfn(src.pfn, t), q1 = load_pfn(src.pfn, t + 16), q2 = load_pfn(src.pfn, t + 32),
                      q3 = load_pfn(src.pfn, t + 48);
        sm.pfn_bd[t][0] = make_float4(q0.b0, q1.b0, q2.b0, q3.b0);
        sm.pfn_bd[t][1] = make_float4(q0.b1, q1.b1, q2.b1, q3.b1);
        sm.pfn_bd[t][2] = make_float4(q0.b2, q1.b2, q2.b2, q3.b2);
        sm.pfn_bd[t][3] = make_float4(q0.d0, q1.d0, q2.d0, q3.d0);
        sm.pfn_bd[t][4] = make_float4(q0.d1, q1.d1, q2.d1, q3.d1);
        sm.pfn_bd[t][5] = make_float4(q0.d2, q1.d2, q2.d2, q3.d2);
        sm.pfn_bd[t][6] = make_float4(q0.shift, q1.shift, q2.shift, q3.shift);
    }
    if (t == 0) {
        for (int s = 0; s < NB; ++s) {
            mbar_init(smem_u32(&sm.full[s]), W);
            mbar_init(smem_u32(&sm.empty[s]), 1);
            sm.dirty[s] = 0;
        }
        for (int s = 0; s < kCvLists; ++s) mbar_init(smem_u32(&sm.ready[s]), 1);
        mbar_init_fence();
    }
    __syncthreads();
    const uint32_t full0 = smem_u32(&sm.full[0]), empty0 = smem_u32(&sm.empty[0]);
    const uint32_t ready0 = smem_u32(&sm.ready[0]), take0 = smem_u32(&sm.list_take[0]);

    if (warp == W) {
        // ------------------------------ control warp ----------------------------------------------
        // builds the occupied-cell list of every tile kCvLists tiles ahead, ships finished tiles
        CvTile lt;           // tile whose list is built next
        lt.init(blockIdx.x, ny, tiles_x);
        int lt_i = 0, lt_b = -1, lt_pbase = 0;
        auto load_codes = [&](const CvTile &q) -> int4 {
            const int x = q.tx * kTileX + 4 * lane;
            if (x >= nx) return make_int4(-1, -1, -1, -1);
            return __ldg(reinterpret_cast<const int4 *>(src.cell_code + ((size_t)q.b * ny + q.y) * nx + x));
        };
        int4 codes = load_codes(lt);
        // L2 warm-up: the slot rows of a tile's pillars are prefetched when its list is built (a few tiles before
        // the PFN warps gather them).  Loading the point indices here as well, to prefetch the points too, was
        // measured and dropped: the loads put a DRAM latency into this warp's per-tile chain.
        auto build_list = [&]() {   // list of tile lt_i into ring slot lt_i % kCvLists; then lt advances
            const int slot = lt_i & (kCvLists - 1);
            const int4 c = codes;
            if (lt.b != lt_b) { lt_b = lt.b; lt_pbase = __ldg(src.point_offsets + lt.b); }
            const uint32_t row0 = (uint32_t)lt.b * (uint32_t)src.max_voxels;
            const int xy0 = (lt.tx * kTileX + 4 * lane) | (lt.y << 16);
            const bool o0 = FusedSrc::occupied(c.x), o1 = FusedSrc::occupied(c.y);
            const bool o2 = FusedSrc::occupied(c.z), o3 = FusedSrc::occupied(c.w);
            const int mine = (int)o0 + (int)o1 + (int)o2 + (int)o3;
            int incl = mine;   // inclusive prefix over the lanes
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += v;
            }
            int pos = incl - mine;
            uint2 *l = &sm.list[slot][0];
            auto put = [&](bool occ, int code, int j) {
                if (occ) {
                    const uint32_t row = row0 + ((unsigned)code & ~kPillarBit);
                    l[pos++] = make_uint2(row, xy0 + j);
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(src.slots + (size_t)row * 32));
                }
            };
            put(o0, c.x, 0);
            put(o1, c.y, 1);
            put(o2, c.z, 2);
            put(o3, c.w, 3);
            if (lane == 31) { sm.list_n[slot] = incl; sm.list_pbase[slot] = lt_pbase; sm.list_take[slot] = 0; }
            __syncwarp();
            if (lane == 0) mbar_arrive(ready0 + 8u * slot);
            ++lt_i;
            if (lt_i < n_my) { lt.advance(step, ny, tiles_x); codes = load_codes(lt); }
        };
        for (int k = 0; k < kCvLists && lt_i < n_my; ++k) build_list();

        CvTile it;
        it.init(blockIdx.x, ny, tiles_x);
        int buf = 0;
        uint32_t parity = 0;
        auto release = [&](int rb) {   // buffer rb has been read by its TMA store: zero it if needed, hand it back
            if (sm.dirty[rb]) {   // warp-uniform
                float4 *t4 = reinterpret_cast<float4 *>(&sm.tile[rb][0]);
                const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
                for (int k = lane; k < kCvTileFloats / 4; k += 32) t4[k] = z;
                __syncwarp();
                if (lane == 0) sm.dirty[rb] = 0;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty0 + 8u * rb);
        };
        int prev = -1;
#pragma unroll 1
        for (int i = 0; i < n_my; ++i) {
            mbar_wait(full0 + 8u * buf, parity);   // every PFN warp is done with tile i and with list i
            fence_async_smem();
            if (lane == 0) {   // four [32 cells][64 channels] boxes; the part of a box beyond nx is clipped by the TMA unit
                const int x0 = it.tx * kTileX;
                const uint32_t s_box = smem_u32(&sm.tile[buf][0]);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (x0 + 32 * k < nx) tma_store_box(&tmap, s_box + 8192u * k, x0 + 32 * k, it.y, it.b * 64);
                bulk_commit();
            }
            if (lt_i < n_my) build_list();            // reuses the ring slot of list i; overlaps the bulk reads
            // the shared-memory reads of tile i overlap the next iteration: only tile i - 1 is reclaimed here
            if (PIPE) {
                if (prev >= 0) {
                    if (lane == 0) bulk_wait_read<1>();
                    __syncwarp();
                    release(prev);
                }
                prev = buf;
            } else {
                if (lane == 0) bulk_wait_read<0>();
                __syncwarp();
                release(buf);
            }
            it.advance(step, ny, tiles_x);
            if (++buf == NB) { buf = 0; parity ^= 1u; }
        }
        if (lane == 0) bulk_wait_read<0>();   // shared memory must outlive the last reads
        __syncwarp();
        return;
    }

    // ---------------------------------- PFN warps -------------------------------------------------
    if constexpr (PAIR) {
        // Two pillars per warp: half-warp h = lane / 16 evaluates list entry k + h; lane hl = lane % 16 owns the
        // output channels hl + 16 j (j < 4) and holds points hl and hl + 16 of its pillar.  The per-pillar
        // bookkeeping (claim, loads, centre, mean, barriers) is issued once for both pillars, which is what bounds
        // the single-pillar variant (ncu r01q: ~280 warp instructions per pillar, 46 of them PFN arithmetic).
        const int half = lane >> 4, hl = lane & 15;
        float a0[4], a1[4], a2[4], a3[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const PfnLane q = load_pfn(src.pfn, hl + 16 * j);
            a0[j] = q.a0; a1[j] = q.a1; a2[j] = q.a2; a3[j] = q.a3;
        }
        const float4 *const bd = &sm.pfn_bd[hl][0];   // the bias constants stay in shared memory (28 registers otherwise)
        float *const stage = &sm.stage[warp][half][0][0];
        // row hl of box 0; rows hl + 16 j are 512 j floats on and share the swizzle phase (16 j % 8 == 0)
        float *const tile_lane = &sm.tile[0][hl * 32];

        struct Slot { int i, xy, pbase; uint32_t idx0, idx1; float4 p0, p1; };   // xy per half (-1: no pillar)
        int g_i = -1, g_n = 0, g_pbase = 0;
        auto next = [&](Slot &s) {
            s.idx0 = s.idx1 = kEmpty;
            s.xy = -1;
#pragma unroll 1
            while (true) {
                if (g_n > 0) {
                    const int slot = g_i & (kCvLists - 1);
                    int k = 0;
                    if (lane == 0)
                        asm volatile("atom.shared.add.u32 %0, [%1], 2;" : "=r"(k) : "r"(take0 + 4u * slot) : "memory");
                    k = __shfl_sync(0xffffffffu, k, 0);
                    if (k < g_n) {
                        s.i = g_i;
                        s.pbase = g_pbase;
                        if (k + half < g_n) {
                            const uint2 v = sm.list[slot][k + half];
                            s.xy = (int)v.y;
                            const uint32_t *row = src.slots + (size_t)v.x * 32 + hl;
                            s.idx0 = __ldg(row);
                            s.idx1 = __ldg(row + 16);
                        }
                        return;
                    }
                    g_n = 0;
                }
                if (g_i >= n_my - 1) { g_i = n_my; s.i = -1; return; }
                const int slot = (g_i + 1) & (kCvLists - 1);
                if (!mbar_test(ready0 + 8u * slot, (uint32_t)((g_i + 1) / kCvLists) & 1u)) { s.i = g_i + 1; return; }
                ++g_i;
                g_n = sm.list_n[slot];
                g_pbase = sm.list_pbase[slot];
            }
        };
        auto load_points = [&](Slot &s) {
            const uint32_t first = __shfl_sync(0xffffffffu, s.idx0, 0, 16);
            const bool more = __any_sync(0xffffffffu, s.idx1 != kEmpty);   // a pillar of the pair has > 16 points
            if (first != kEmpty) {   // per half; padded lanes take a copy of point 0 of their pillar
                s.p0 = __ldg(src.points + s.pbase + (s.idx0 != kEmpty ? s.idx0 : first));
                if (more) s.p1 = __ldg(src.points + s.pbase + (s.idx1 != kEmpty ? s.idx1 : first));
            }
        };
        int cur_i = 0, cur_buf = 0;
        uint32_t cur_par = 1;
        bool wrote = false;
        auto finish_tiles_until = [&](int target) {
#pragma unroll 1
            while (cur_i < target) {
                if (wrote) {
                    if (lane == 0) sm.dirty[cur_buf] = 1;
                    fence_async_smem();
                    wrote = false;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(full0 + 8u * cur_buf);
                ++cur_i;
                if (++cur_buf == NB) { cur_buf = 0; cur_par ^= 1u; }
                if (cur_i < n_my) mbar_wait(empty0 + 8u * cur_buf, cur_par);
            }
        };
        auto pipe = [&](Slot &s0, Slot &s1, Slot &s2) {
            load_points(s1);
            next(s2);
            if (cur_i < s0.i) finish_tiles_until(s0.i);
            const unsigned bal0 = __ballot_sync(0xffffffffu, s0.idx0 != kEmpty);
            const unsigned bal1 = __ballot_sync(0xffffffffu, s0.idx1 != kEmpty);
            if (bal0 == 0u) return;   // bubble
            const int n_lo = __popc(bal0 & 0xFFFFu) + __popc(bal1 & 0xFFFFu);
            const int n_hi = __popc(bal0 >> 16) + __popc(bal1 >> 16);
            const int n = half ? n_hi : n_lo;          // slots fill from 0
            const int nmax = max(n_lo, n_hi);          // warp-uniform
            const int x = s0.xy & 0xFFFF, y = s0.xy >> 16;
            const float cx = __fadd_rn(__fmul_rn((float)x, src.vx), src.ox);
            const float cy = __fadd_rn(__fmul_rn((float)y, src.vy), src.oy);
            const float cz = src.cz;
            const float xr0 = __fsub_rn(s0.p0.x, cx), yr0 = __fsub_rn(s0.p0.y, cy), zr0 = __fsub_rn(s0.p0.z, cz);
            const bool v0 = hl < n;
            float sx = v0 ? xr0 : 0.0f, sy = v0 ? yr0 : 0.0f, sz = v0 ? zr0 : 0.0f;
            __syncwarp();
            stage[hl] = xr0;
            stage[32 + hl] = yr0;
            stage[64 + hl] = zr0;
            stage[96 + hl] = s0.p0.w;
            if (bal1 != 0u) {   // warp-uniform: some pillar of the pair has more than 16 points
                const float xr1 = __fsub_rn(s0.p1.x, cx), yr1 = __fsub_rn(s0.p1.y, cy), zr1 = __fsub_rn(s0.p1.z, cz);
                stage[16 + hl] = xr1;
                stage[48 + hl] = yr1;
                stage[80 + hl] = zr1;
                stage[112 + hl] = s0.p1.w;
                // xor-butterfly of the oracle: level 16 pairs slot s with s + 16 = this lane's two points
                const bool v1 = hl + 16 < n;
                sx = __fadd_rn(sx, v1 ? xr1 : 0.0f);
                sy = __fadd_rn(sy, v1 ? yr1 : 0.0f);
                sz = __fadd_rn(sz, v1 ? zr1 : 0.0f);
            }
#pragma unroll
            for (int m = 8; m >= 1; m >>= 1) {
                sx = __fadd_rn(sx, __shfl_xor_sync(0xffffffffu, sx, m));
                sy = __fadd_rn(sy, __shfl_xor_sync(0xffffffffu, sy, m));
                sz = __fadd_rn(sz, __shfl_xor_sync(0xffffffffu, sz, m));
            }
            const float inv_n = sm.inv_n[n];
            const float mx = __fmul_rn(sx, inv_n), my = __fmul_rn(sy, inv_n), mz = __fmul_rn(sz, inv_n);
            float2 bias[2];
            const float4 sh = bd[6];
            {
                const float4 B0 = bd[0], B1 = bd[1], B2 = bd[2], D0 = bd[3], D1 = bd[4], D2 = bd[5];
                float2 lo = __ffma2_rn(make_float2(B0.x, B0.y), dup2(cx), make_float2(sh.x, sh.y));
                float2 hi = __ffma2_rn(make_float2(B0.z, B0.w), dup2(cx), make_float2(sh.z, sh.w));
                lo = __ffma2_rn(make_float2(B1.x, B1.y), dup2(cy), lo); hi = __ffma2_rn(make_float2(B1.z, B1.w), dup2(cy), hi);
                lo = __ffma2_rn(make_float2(B2.x, B2.y), dup2(cz), lo); hi = __ffma2_rn(make_float2(B2.z, B2.w), dup2(cz), hi);
                lo = __ffma2_rn(make_float2(D0.x, D0.y), dup2(mx), lo); hi = __ffma2_rn(make_float2(D0.z, D0.w), dup2(mx), hi);
                lo = __ffma2_rn(make_float2(D1.x, D1.y), dup2(my), lo); hi = __ffma2_rn(make_float2(D1.z, D1.w), dup2(my), hi);
                bias[0] = __ffma2_rn(make_float2(D2.x, D2.y), dup2(mz), lo);
                bias[1] = __ffma2_rn(make_float2(D2.z, D2.w), dup2(mz), hi);
            }
            float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
            __syncwarp();
            const float4 *s4 = reinterpret_cast<const float4 *>(stage);
#pragma unroll 1
            for (int q = 0; q * 4 < nmax; ++q) {
                const float4 X = s4[q], Y = s4[8 + q], Z = s4[16 + q], I = s4[24 + q];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float2 u = __fmul2_rn(dup2(a3[j]), make_float2(I.x, I.y));
                    float2 v = __fmul2_rn(dup2(a3[j]), make_float2(I.z, I.w));
                    u = __ffma2_rn(dup2(a2[j]), make_float2(Z.x, Z.y), u);
                    v = __ffma2_rn(dup2(a2[j]), make_float2(Z.z, Z.w), v);
                    u = __ffma2_rn(dup2(a1[j]), make_float2(Y.x, Y.y), u);
                    v = __ffma2_rn(dup2(a1[j]), make_float2(Y.z, Y.w), v);
                    u = __ffma2_rn(dup2(a0[j]), make_float2(X.x, X.y), u);
                    v = __ffma2_rn(dup2(a0[j]), make_float2(X.z, X.w), v);
                    best[j] = fmaxf(fmaxf(best[j], u.x), u.y);
                    best[j] = fmaxf(fmaxf(best[j], v.x), v.y);
                }
            }
            if (s0.xy >= 0) {
                const int xc = x & (kTileX - 1);
                float *tl = tile_lane + cur_buf * kCvTileFloats + (xc >> 5) * 2048 + ((((xc >> 2) ^ hl) & 7) << 2) + (xc & 3);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const float2 o = __fadd2_rn(make_float2(best[2 * j], best[2 * j + 1]), bias[j]);
                    float oa = fmaxf(o.x, 0.0f), ob = fmaxf(o.y, 0.0f);
                    if (n < 32) { oa = fmaxf(oa, j ? sh.z : sh.x); ob = fmaxf(ob, j ? sh.w : sh.y); }
                    tl[(2 * j) * 512] = oa;
                    tl[(2 * j + 1) * 512] = ob;
                }
            }
            wrote = true;
        };
        Slot A, B, C;
        A.p0 = A.p1 = B.p0 = B.p1 = C.p0 = C.p1 = make_float4(0.f, 0.f, 0.f, 0.f);
        A.pbase = B.pbase = C.pbase = 0;
        next(A);
        next(B);
        load_points(A);
#pragma unroll 1
        while (true) {
            if (A.i < 0) break;
            pipe(A, B, C);
            if (B.i < 0) break;
            pipe(B, C, A);
            if (C.i < 0) break;
            pipe(C, A, B);
        }
        finish_tiles_until(n_my);
        return;
    }
    const PfnPacked w = pack_pfn(load_pfn(src.pfn, lane), load_pfn(src.pfn, lane + 32));
    float *const stage = &sm.stage[warp][0][0][0];
    float *const tile_lane = &sm.tile[0][lane * 32];   // row `lane` of box 0 (row lane + 32 is 1024 floats on)

    // Generator: takes the next unclaimed occupied cell of the CTA's tile stream (dynamic distribution over the
    // PFN warps, one shared-memory atomic per pillar) and issues the load of its slot row.
    int g_i = -1, g_n = 0, g_pbase = 0;   // list being consumed (g_n = 0: exhausted); g_i == n_my: end of stream
    // Never blocks: when the next list is not built yet (the control warp builds list i + kCvLists only after every
    // PFN warp has handed in tile i) it yields a bubble {i = first tile that may still get cells of this warp,
    // xy = -1}, so the evaluation stage can hand in the tiles below it and the control warp can go on.
    auto next = [&](CvSlot &s) {
        s.idx = kEmpty;
#pragma unroll 1
        while (true) {
            if (g_n > 0) {
                const int slot = g_i & (kCvLists - 1);
                int k = 0;
                if (lane == 0)   // plain atom.shared (nvcc's warp-aggregation prologue is pure overhead for one lane)
                    asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(k) : "r"(take0 + 4u * slot) : "memory");
                k = __shfl_sync(0xffffffffu, k, 0);
                if (k < g_n) {
                    const uint2 v = sm.list[slot][k];
                    s.e = CvEnt{g_i, (int)v.y, g_pbase};
                    s.idx = __ldg(src.slots + (size_t)v.x * 32 + lane);
                    return;
                }
                g_n = 0;
            }
            if (g_i >= n_my - 1) { g_i = n_my; s.e = CvEnt{-1, -1, 0}; return; }
            const int slot = (g_i + 1) & (kCvLists - 1);
            if (!mbar_test(ready0 + 8u * slot, (uint32_t)((g_i + 1) / kCvLists) & 1u)) {
                s.e = CvEnt{g_i + 1, -1, 0};
                return;
            }
            ++g_i;
            g_n = sm.list_n[slot];
            g_pbase = sm.list_pbase[slot];
        }
    };
    auto load_point = [&](CvSlot &s) {
        const uint32_t first = __shfl_sync(0xffffffffu, s.idx, 0);
        if (first != kEmpty)   // false only at the end of the stream (a pillar has >= 1 point)
            s.p = __ldg(src.points + s.e.pbase + (s.idx != kEmpty ? s.idx : first));   // padded lanes: copy of point 0
    };

    int cur_i = 0, cur_buf = 0;   // tile this warp is writing into
    uint32_t cur_par = 1;         // parity to wait for on empty[cur_buf] (fresh barrier: phase "1" is complete)
    bool wrote = false;
    auto finish_tiles_until = [&](int target) {   // hand tiles cur_i .. target-1 to the control warp
#pragma unroll 1
        while (cur_i < target) {
            if (wrote) {
                if (lane == 0) sm.dirty[cur_buf] = 1;
                fence_async_smem();
                wrote = false;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(full0 + 8u * cur_buf);
            ++cur_i;
            if (++cur_buf == NB) { cur_buf = 0; cur_par ^= 1u; }
            if (cur_i < n_my) mbar_wait(empty0 + 8u * cur_buf, cur_par);
        }
    };
    // one pipeline step: s0 is evaluated, s1 gets its points, s2 becomes the pillar after s1
    auto pipe = [&](CvSlot &s0, CvSlot &s1, CvSlot &s2) {
        load_point(s1);
        next(s2);
        if (cur_i < s0.e.i) finish_tiles_until(s0.e.i);
        if (s0.e.xy < 0) return;   // bubble
        const int n = __popc(__ballot_sync(0xffffffffu, s0.idx != kEmpty));   // slots fill from 0
        const int x = s0.e.xy & 0xFFFF, y = s0.e.xy >> 16;
        const float cx = __fadd_rn(__fmul_rn((float)x, src.vx), src.ox);
        const float cy = __fadd_rn(__fmul_rn((float)y, src.vy), src.oy);
        const float2 r = pfn_pillar_packed(w, s0.p, n, sm.inv_n[n], cx, cy, src.cz, stage, lane);
        // cell xc of the tile = box xc / 32, 16-byte chunk (xc % 32) / 4 XOR (row & 7)  (CU_TENSOR_MAP_SWIZZLE_128B)
        const int xc = x & (kTileX - 1);
        float *tl = tile_lane + cur_buf * kCvTileFloats + (xc >> 5) * 2048 + ((((xc >> 2) ^ lane) & 7) << 2) + (xc & 3);
        tl[0] = r.x;
        tl[1024] = r.y;
        wrote = true;
    };

    CvSlot A, B, C;
    A.p = B.p = C.p = make_float4(0.f, 0.f, 0.f, 0.f);
    next(A);
    next(B);
    load_point(A);
#pragma unroll 1
    while (true) {
        if (A.e.i < 0) break;
        pipe(A, B, C);
        if (B.e.i < 0) break;
        pipe(B, C, A);
        if (C.e.i < 0) break;
        pipe(C, A, B);
    }
    finish_tiles_until(n_my);
}

// dense cell -> pillar-row map for the standalone scatter
__global__ void __launch_bounds__(256)
k_build_cell_map(const int4 *__restrict__ coords, int n_pillars, int nx, int ny, int n_batch,
                 int32_t *__restrict__ cell_map) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_pillars) return;
    const int4 c = __ldg(coords + m);   // (b, z, y, x); idx = z + y*nx + x  (point_pillar_scatter.py:58)
    const long long idx = (long long)c.y + (long long)c.z * nx + c.w;
    if (c.x < 0 || c.x >= n_batch || idx < 0 || idx >= (long long)nx * ny) return;
    cell_map[(size_t)c.x * nx * ny + idx] = m;
}

// canvas [A*64][ny][nx] f32 as a 3-D tensor; box = 32 cells x 1 row x 64 channel planes, 128-byte swizzle in shared memory
static bool cv_encode_map(CUtensorMap *map, float *canvas, int nx, int ny, long long planes) {
    const auto encode = tensor_map_encoder();
    if (!encode) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)nx, (cuuint64_t)ny, (cuuint64_t)planes};
    const cuuint64_t gstride[2] = {(cuuint64_t)nx * 4, (cuuint64_t)ny * nx * 4};
    const cuuint32_t box[3] = {32, 1, 64};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, canvas, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int W, int NB, int MINB, bool PAIR, bool PIPE>
static int launch_canvas_persist(const FusedSrc &src, const GeomDev &g, int n_agents, long long tiles, float *canvas,
                                 cudaStream_t st) {
    using Smem = CvSmem<W, NB, PAIR>;
    constexpr size_t kSmemBytes = sizeof(Smem);
    static int sms = 0, per_sm = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaFuncSetAttribute(k_canvas_persist<W, NB, MINB, PAIR, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_canvas_persist<W, NB, MINB, PAIR, PIPE>, (W + 1) * 32, kSmemBytes);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (per_sm < 1) per_sm = 1;
    }
    CUtensorMap map;
    if (!cv_encode_map(&map, canvas, g.grid[0], g.grid[1], (long long)n_agents * 64)) return -1;   // caller falls back
    const int grid = (int)(tiles < (long long)sms * per_sm ? tiles : (long long)sms * per_sm);
    const int tiles_x = (g.grid[0] + kTileX - 1) / kTileX;
    CvStep step;
    step.stx = grid % tiles_x;
    step.sy = (grid / tiles_x) % g.grid[1];
    step.sb = (grid / tiles_x) / g.grid[1];
    k_canvas_persist<W, NB, MINB, PAIR, PIPE><<<grid, (W + 1) * 32, kSmemBytes, st>>>(map, src, g.grid[0], g.grid[1], n_agents, step);
    GC_LAUNCH_CHECK("k_canvas_persist");
    return GC_OK;
}

static int make_geom(const gcVoxelGeom *geom, GeomDev *g) {
    GC_REQUIRE(geom != nullptr, GC_EINVAL, "geom is null");
    GC_REQUIRE(geom->max_points == GC_MAX_POINTS_PER_PILLAR, GC_EUNSUPPORTED,
               "max_points_per_voxel must be 32 (got %d)", geom->max_points);
    GC_REQUIRE(geom->grid[0] > 0 && geom->grid[1] > 0 && geom->grid[2] > 0 && geom->max_voxels > 0, GC_EINVAL,
               "bad voxel grid");
    const long long ncell = (long long)geom->grid[0] * geom->grid[1] * geom->grid[2];
    GC_REQUIRE(ncell < (1ll << 30), GC_EUNSUPPORTED, "voxel grid too large");
    for (int j = 0; j < 3; ++j) {
        g->rmin[j] = geom->range_min[j];
        g->voxel[j] = geom->voxel[j];
        g->grid[j] = geom->grid[j];
    }
    g->max_voxels = geom->max_voxels;
    g->ncell = (int)ncell;
    return GC_OK;
}

static inline int blocks_per_agent(int max_agent_points) { return (max_agent_points + 1023) / 1024 + 1; }

}  // namespace gc

using namespace gc;

extern "C" size_t gc_voxelize_workspace_bytes(const gcVoxelGeom *geom, int n_agents, int total_points) {
    if (!geom || n_agents <= 0 || total_points < 0) return 0;
    return carve_workspace(nullptr, *geom, n_agents, total_points).bytes;
}

static int voxelize_impl(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                           int max_agent_points, const gcVoxelGeom *geom, void *workspace, int32_t *n_pillars,
                           void *stream) {
    GeomDev g;
    if (int rc = make_geom(geom, &g)) return rc;
    GC_REQUIRE(points && point_offsets && workspace && n_pillars, GC_EINVAL, "gc_voxelize: null pointer");
    GC_REQUIRE(n_agents > 0 && n_agents <= 65535 && total_points >= 0, GC_EINVAL, "gc_voxelize: bad sizes");
    if (max_agent_points <= 0 || max_agent_points > total_points) max_agent_points = total_points;
    cudaStream_t st = (cudaStream_t)stream;
    const VoxelWorkspace w = carve_workspace(workspace, *geom, n_agents, total_points);
    const int bpa = blocks_per_agent(max_agent_points);
    cudaMemsetAsync(w.cell_code, 0xFF, (size_t)n_agents * g.ncell * 4, st);
    // GC_VOXELIZE_IMPL=legacy keeps the round-1 four-kernel voxelizer (A/B and parity: tests run both)
    const char *impl = getenv("GC_VOXELIZE_IMPL");
    if (!(impl && strcmp(impl, "legacy") == 0)) {
        const int n_flags = n_agents * (max_agent_points / 128 + 2);
        const int work = total_points > 2 * n_flags ? total_points : 2 * n_flags;
        k_cell_assign2<<<(work + 511) / 512, 256, 0, st>>>((const float4 *)points, point_offsets, n_agents, total_points,
                                                          g, w.cell_code, w.point_cell, (uint32_t *)w.block_counts,
                                                          n_flags);
        GC_LAUNCH_CHECK("k_cell_assign2");
        static int items = 0;
        if (items == 0) {
            const char *e = getenv("GC_VOXELIZE_ITEMS");   // A/B of the points per thread (1, 2, 4); CTAs of 128 threads
            items = e ? atoi(e) : 2;                       // measured the same as 256 (profiles/r02bd_voxelizer_ab.txt)
            if (items != 1 && items != 4) items = 2;
        }
        const int chunks = (max_agent_points + 256 * items - 1) / (256 * items) + 1;
        GC_REQUIRE(chunks <= 65535, GC_EUNSUPPORTED, "gc_voxelize: too many points per agent");
        uint32_t *flags = (uint32_t *)w.block_counts;
#define GC_BUILD(IT_)                                                                                          \
    k_pillar_build<IT_, 256><<<dim3(n_agents, chunks), 256, 0, st>>>(point_offsets, w.point_cell, w.cell_code, \
                                                                     g.ncell, g.max_voxels, chunks, flags,     \
                                                                     w.slots, w.pillar_cell, n_pillars)
        if (items == 1) GC_BUILD(1); else if (items == 4) GC_BUILD(4); else GC_BUILD(2);
#undef GC_BUILD
        GC_LAUNCH_CHECK("k_pillar_build");
        return GC_OK;
    }
    if (total_points > 0) {
        k_cell_assign<<<(total_points + 255) / 256, 256, 0, st>>>((const float4 *)points, point_offsets, n_agents,
                                                                 total_points, g, w.cell_code, w.point_cell);
        GC_LAUNCH_CHECK("k_cell_assign");
    }
    k_pillar_count<<<dim3(bpa, n_agents), 256, 0, st>>>(point_offsets, w.point_cell, w.cell_code, g.ncell, bpa,
                                                        w.block_counts);
    GC_LAUNCH_CHECK("k_pillar_count");
    k_pillar_assign<<<dim3(bpa, n_agents), 256, 0, st>>>(point_offsets, w.point_cell, w.cell_code, g.ncell,
                                                         g.max_voxels, bpa, w.block_counts, w.slots, w.pillar_cell,
                                                         n_pillars);
    GC_LAUNCH_CHECK("k_pillar_assign");
    if (total_points > 0) {
        const int chunks = (max_agent_points + 255) / 256;
        GC_REQUIRE(chunks <= 65535, GC_EUNSUPPORTED, "gc_voxelize: more than 16.7M points per agent");
        k_slot_insert<<<dim3(n_agents, chunks), 256, 0, st>>>(point_offsets, w.point_cell, w.cell_code, g.ncell,
                                                            g.max_voxels, w.slots);
        GC_LAUNCH_CHECK("k_slot_insert");
    }
    return GC_OK;
}

extern "C" int gc_voxelize(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                           int max_agent_points, const gcVoxelGeom *geom, void *workspace, int32_t *n_pillars,
                           void *stream) {
    if (int rc = voxelize_impl(points, point_offsets, n_agents, total_points, max_agent_points, geom, workspace, n_pillars, stream))
        return rc;
    const VoxelWorkspace w = carve_workspace(workspace, *geom, n_agents, total_points);
    cudaMemcpyAsync(w.n_pillars, n_pillars, (size_t)n_agents * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    return GC_OK;
}

extern "C" int gc_voxel_gather(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                               const gcVoxelGeom *geom, const void *workspace, const int32_t *pillar_offsets,
                               int total_pillars, float *voxels, int32_t *coords, int32_t *num_points,
                               void *stream) {
    GeomDev g;
    if (int rc = make_geom(geom, &g)) return rc;
    GC_REQUIRE(points && point_offsets && workspace && pillar_offsets, GC_EINVAL, "gc_voxel_gather: null pointer");
    GC_REQUIRE(n_agents > 0 && total_pillars >= 0, GC_EINVAL, "gc_voxel_gather: bad sizes");
    if (total_pillars == 0) return GC_OK;
    GC_REQUIRE(voxels && coords && num_points, GC_EINVAL, "gc_voxel_gather: null output");
    const VoxelWorkspace w = carve_workspace(const_cast<void *>(workspace), *geom, n_agents, total_points);
    k_voxel_gather<<<(total_pillars + 7) / 8, 256, 0, (cudaStream_t)stream>>>(
        (const float4 *)points, point_offsets, n_agents, g, w.slots, w.pillar_cell, pillar_offsets, total_pillars,
        (float4 *)voxels, (int4 *)coords, num_points);
    GC_LAUNCH_CHECK("k_voxel_gather");
    return GC_OK;
}

extern "C" int gc_pillar_vfe(const float *voxels, const int32_t *num_points, const int32_t *coords, int n_pillars,
                             const float *pfn, const float voxel[3], const float centre_offset[3],
                             float *pillar_features, void *stream) {
    GC_REQUIRE(n_pillars >= 0, GC_EINVAL, "gc_pillar_vfe: negative pillar count");
    if (n_pillars == 0) return GC_OK;
    GC_REQUIRE(voxels && num_points && coords && pfn && voxel && centre_offset && pillar_features, GC_EINVAL,
               "gc_pillar_vfe: null pointer");
    k_pillar_vfe<<<(n_pillars + 7) / 8, 256, 0, (cudaStream_t)stream>>>(
        (const float4 *)voxels, num_points, (const int4 *)coords, n_pillars, pfn, voxel[0], voxel[1], voxel[2],
        centre_offset[0], centre_offset[1], centre_offset[2], pillar_features);
    GC_LAUNCH_CHECK("k_pillar_vfe");
    return GC_OK;
}

extern "C" int gc_scatter_canvas(const float *pillar_features, const int32_t *coords, int n_pillars, int C, int nx,
                                 int ny, int n_batch, int32_t *cell_map, float *canvas, void *stream) {
    GC_REQUIRE(n_pillars >= 0 && C > 0 && nx > 0 && ny > 0 && n_batch >= 0, GC_EINVAL, "gc_scatter_canvas: bad sizes");
    GC_REQUIRE(ny <= 65535 && n_batch <= 65535, GC_EUNSUPPORTED, "gc_scatter_canvas: grid too large");
    if (n_batch == 0) return GC_OK;
    GC_REQUIRE(cell_map && canvas && (n_pillars == 0 || (pillar_features && coords)), GC_EINVAL,
               "gc_scatter_canvas: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(cell_map, 0xFF, (size_t)n_batch * nx * ny * 4, st);
    if (n_pillars > 0) {
        k_build_cell_map<<<(n_pillars + 255) / 256, 256, 0, st>>>((const int4 *)coords, n_pillars, nx, ny, n_batch,
                                                                 cell_map);
        GC_LAUNCH_CHECK("k_build_cell_map");
    }
    FeatSrc src{pillar_features, cell_map, C};
    k_canvas<FeatSrc><<<dim3((nx + kTileX - 1) / kTileX, ny, n_batch), 256, 0, st>>>(src, nx, ny, C, canvas);
    GC_LAUNCH_CHECK("k_canvas<FeatSrc>");
    return GC_OK;
}

extern "C" int gc_pillar_canvas(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                                const gcVoxelGeom *geom, const void *workspace, const float *pfn,
                                const float centre_offset[3], float *canvas, void *stream) {
    GeomDev g;
    if (int rc = make_geom(geom, &g)) return rc;
    GC_REQUIRE(g.grid[2] == 1, GC_EUNSUPPORTED, "PointPillarScatter requires nz == 1 (point_pillar_scatter.py:17)");
    GC_REQUIRE(points && point_offsets && workspace && pfn && centre_offset && canvas, GC_EINVAL,
               "gc_pillar_canvas: null pointer");
    GC_REQUIRE(n_agents > 0 && n_agents <= 65535 && g.grid[1] <= 65535, GC_EINVAL, "gc_pillar_canvas: bad sizes");
    const VoxelWorkspace w = carve_workspace(const_cast<void *>(workspace), *geom, n_agents, total_points);
    FusedSrc src;
    src.points = (const float4 *)points;
    src.point_offsets = point_offsets;
    src.cell_code = w.cell_code;
    src.slots = w.slots;
    src.pfn = pfn;
    src.max_voxels = g.max_voxels;
    src.vx = g.voxel[0];
    src.vy = g.voxel[1];
    src.ox = centre_offset[0];
    src.oy = centre_offset[1];
    src.cz = 0.0f * g.voxel[2] + centre_offset[2];
    // Two writers, same results (bit-exact, tests run both).  The persistent writer wins when the canvas is densely
    // occupied (B200, 8x4 agents x 100k points: 256x256 grid, 27 % of the cells occupied: 0.204 vs 0.249 ms) and loses
    // when it is sparse (512x256 grid, 16 %: 0.49 vs 0.40 ms -- too few pillars per tile to hide its per-tile
    // hand-over latency), so the default is chosen from the mean number of points per cell; GC_CANVAS_IMPL=tile|persist
    // overrides.
    const char *impl = getenv("GC_CANVAS_IMPL");
    const bool dense = (double)total_points >= 1.0 * (double)n_agents * (double)g.ncell;
    bool use_tile = impl ? strcmp(impl, "tile") == 0 : !dense;
    if (impl && strcmp(impl, "persist") == 0) use_tile = false;
    if ((g.grid[0] & 3) != 0) use_tile = true;
    if (!use_tile) {
        const long long tiles = (long long)n_agents * g.grid[1] * ((g.grid[0] + kTileX - 1) / kTileX);
        GC_REQUIRE(tiles < (1ll << 31) && (long long)n_agents * g.max_voxels < (1ll << 32) && g.grid[0] <= 65535 &&
                       g.grid[1] <= 32767,
                   GC_EUNSUPPORTED, "gc_pillar_canvas: grid / agent count too large for the persistent writer");
        static int cfg = -1;
        if (cfg < 0) {
            const char *e = getenv("GC_CANVAS_CFG");   // A/B of the CTA shape; see DESIGN.md section 3
            cfg = e ? atoi(e) : 0;
        }
        int rc;
        cudaStream_t st = (cudaStream_t)stream;
        switch (cfg) {
            case 1: rc = launch_canvas_persist<15, 6, 1, true, false>(src, g, n_agents, tiles, canvas, st); break;
            case 2: rc = launch_canvas_persist<15, 6, 1, true, true>(src, g, n_agents, tiles, canvas, st); break;
            case 3: rc = launch_canvas_persist<9, 3, 2, true, true>(src, g, n_agents, tiles, canvas, st); break;
            case 4: rc = launch_canvas_persist<10, 3, 2, false, false>(src, g, n_agents, tiles, canvas, st); break;
            default: rc = launch_canvas_persist<9, 3, 2, true, false>(src, g, n_agents, tiles, canvas, st); break;
        }
        if (rc != -1) return rc;   // -1: no cuTensorMapEncodeTiled in this driver -> per-tile kernel
    }
    k_canvas<FusedSrc><<<dim3((g.grid[0] + kTileX - 1) / kTileX, g.grid[1], n_agents), 256, 0,
                         (cudaStream_t)stream>>>(src, g.grid[0], g.grid[1], GC_PFN_OUT, canvas);
    GC_LAUNCH_CHECK("k_canvas<FusedSrc>");
    return GC_OK;
}

// The fused front end with the canvas written as the backbone's operand planes (k_canvas_planes); same arguments as
// gc_pillar_canvas, xh / xl: [n_agents][ny*nx][64] bf16 value / residual.
static int pillar_canvas_planes(bool sparse, const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                                const gcVoxelGeom *geom, const void *workspace, const float *pfn,
                                const float centre_offset[3], void *xh, void *xl, void *stream) {
    GeomDev g;
    if (int rc = make_geom(geom, &g)) return rc;
    GC_REQUIRE(g.grid[2] == 1, GC_EUNSUPPORTED, "PointPillarScatter requires nz == 1 (point_pillar_scatter.py:17)");
    GC_REQUIRE(points && point_offsets && workspace && pfn && centre_offset && xh && xl, GC_EINVAL,
               "gc_pillar_canvas_planes: null pointer");
    GC_REQUIRE(n_agents > 0 && n_agents <= 65535 && g.grid[1] <= 65535, GC_EINVAL, "gc_pillar_canvas_planes: bad sizes");
    const VoxelWorkspace w = carve_workspace(const_cast<void *>(workspace), *geom, n_agents, total_points);
    FusedSrc src;
    src.points = (const float4 *)points;
    src.point_offsets = point_offsets;
    src.cell_code = w.cell_code;
    src.slots = w.slots;
    src.pfn = pfn;
    src.max_voxels = g.max_voxels;
    src.vx = g.voxel[0];
    src.vy = g.voxel[1];
    src.ox = centre_offset[0];
    src.oy = centre_offset[1];
    src.cz = 0.0f * g.voxel[2] + centre_offset[2];
    const dim3 grid((g.grid[0] + kTileX - 1) / kTileX, g.grid[1], n_agents);
    if (sparse) {
        static int sms = 0;
        if (sms == 0) {
            int dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        }
        const char *e = getenv("GC_SPARSE_WRITER");   // A/B and tests: "tile" = k_canvas_planes<true>
        if (e && strcmp(e, "tile") == 0) {
            k_canvas_planes<true><<<grid, 256, 0, (cudaStream_t)stream>>>(src, g.grid[0], g.grid[1], (uint4 *)xh, (uint4 *)xl);
        } else {
            // four CTAs of eight warps per SM over all agents; a warp walks its pillars with stride = warps per agent
            int bpa = (4 * sms + n_agents - 1) / n_agents;
            const int cap = (g.max_voxels + 7) / 8;
            bpa = bpa < 1 ? 1 : (bpa > cap ? cap : bpa);
            k_pillar_planes_sparse<<<dim3(bpa, n_agents), 256, 0, (cudaStream_t)stream>>>(
                src, w.pillar_cell, w.n_pillars, g.grid[0], g.ncell, (uint32_t *)xh, (uint32_t *)xl);
        }
    } else
        k_canvas_planes<false><<<grid, 256, 0, (cudaStream_t)stream>>>(src, g.grid[0], g.grid[1], (uint4 *)xh, (uint4 *)xl);
    GC_LAUNCH_CHECK("k_canvas_planes");
    return GC_OK;
}

extern "C" int gc_pillar_canvas_planes(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                                       const gcVoxelGeom *geom, const void *workspace, const float *pfn,
                                       const float centre_offset[3], void *xh, void *xl, void *stream) {
    return pillar_canvas_planes(false, points, point_offsets, n_agents, total_points, geom, workspace, pfn, centre_offset, xh, xl,
                                stream);
}

// Sparse maintenance of the planes: xh / xl are all-zero on entry, only the occupied cells are written; the caller calls
// gc_planes_clear_occupied (same workspace, before the next gc_voxelize) once the planes have been consumed, which zeroes
// exactly those cells again.  330 MB written + 330 MB cleared instead of 2.0 GB written per 60 agents at 512 x 256.
extern "C" int gc_pillar_canvas_planes_sparse(const float *points, const int32_t *point_offsets, int n_agents, int total_points,
                                              const gcVoxelGeom *geom, const void *workspace, const float *pfn,
                                              const float centre_offset[3], void *xh, void *xl, void *stream) {
    return pillar_canvas_planes(true, points, point_offsets, n_agents, total_points, geom, workspace, pfn, centre_offset, xh, xl,
                                stream);
}

extern "C" int gc_planes_clear_occupied(const gcVoxelGeom *geom, int n_agents, int total_points, const void *workspace, void *xh,
                                        void *xl, void *stream) {
    GeomDev g;
    if (int rc = make_geom(geom, &g)) return rc;
    GC_REQUIRE(workspace && xh && xl, GC_EINVAL, "gc_planes_clear_occupied: null pointer");
    GC_REQUIRE(n_agents > 0 && g.grid[2] == 1, GC_EINVAL, "gc_planes_clear_occupied: bad sizes");
    const VoxelWorkspace w = carve_workspace(const_cast<void *>(workspace), *geom, n_agents, total_points);
    GC_REQUIRE(n_agents <= 65535, GC_EUNSUPPORTED, "gc_planes_clear_occupied: too many agents");
    k_planes_clear<<<dim3((g.max_voxels * 8 + 255) / 256, n_agents), 256, 0, (cudaStream_t)stream>>>(
        w.pillar_cell, w.n_pillars, g.max_voxels, g.ncell, (uint4 *)xh, (uint4 *)xl);
    GC_LAUNCH_CHECK("k_planes_clear");
    return GC_OK;
}
