// Every PTX wrapper of the asynchronous sm_100a hardware the kernels use, in one place: mbarriers, TMA tensor and bulk copies
// (global <-> shared, multicast), proxy fences, tensor memory (alloc / ld / st), tcgen05.mma with its shared-memory and
// instruction descriptors and commits, warp election, cluster barriers and DSMEM stores that complete on an mbarrier; plus the
// host-side lookup of cuTensorMapEncodeTiled.  The rules these encode (mbarrier phase parity, expect_tx byte counts, TMEM
// alloc / relinquish / dealloc, wait::ld before reading a tcgen05.ld result) hang or corrupt a kernel when wrong rather than
// fail a test, so they are written once.  PTX that one kernel file uses outside this machinery stays in that file.
//
// Everything here was validated on the B200 by the parity tests of the kernels that use it: K-major SWIZZLE_NONE / SWIZZLE_64B
// shared-memory descriptors (core matrix = 8 rows x 16 bytes; LBO = byte distance between core matrices along K, SBO = along
// M/N), kind::f16 (bf16 operands) and kind::tf32 instruction descriptors with fp32 accumulation, cta_group::1, completion
// through tcgen05.commit -> mbarrier, epilogue through tcgen05.ld.32x32b (lane = accumulator row).
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace gc {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarriers ----
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// after the mbar_init calls, before the barriers are used by other threads, the async proxy or other CTAs of the cluster
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive and add `bytes` to the transaction count the current phase waits for (TMA / bulk copies / st_async4 complete it)
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// spin until the phase with the given parity has completed
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "MBAR_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra MBAR_DONE_%=;\n\t"
        "bra MBAR_WAIT_%=;\n\t"
        "MBAR_DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
// one try_wait: true when that phase has completed
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}

// ---- TMA tensor copies (the map is a __grid_constant__ kernel parameter) ----
__device__ __forceinline__ void tma_load_box(uint32_t dst, const CUtensorMap *map, int x, int y, int plane, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(plane), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap *map, int c, int x, int y, int a, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c), "r"(x), "r"(y), "r"(a), "r"(bar)
        : "memory");
}
// shared -> global, tracked by bulk groups: bulk_commit closes the group, bulk_wait_read<N> waits until at most N groups
// still read their shared-memory source
__device__ __forceinline__ void tma_store_box(const CUtensorMap *map, uint32_t src, int x, int y, int plane) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(plane), "r"(src) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

// ---- 1-D bulk copies global -> shared, completion counted in bytes on an mbarrier; 16-byte aligned, size % 16 == 0 ----
__device__ __forceinline__ void bulk_copy(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
// the same copy delivered to the same shared-memory offset (and mbarrier) of every CTA of the cluster named in cta_mask
__device__ __forceinline__ void bulk_copy_multicast(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(dst),
        "l"(src), "r"(bytes), "r"(bar), "h"(cta_mask)
        : "memory");
}
// a copy that is the only transaction of its barrier phase: arrive + expect its bytes, then issue it
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t bar) {
    mbar_expect_tx(bar, bytes);
    bulk_copy(dst_smem, src, bytes, bar);
}

// ---- fences ----
// generic-proxy shared-memory stores -> async proxy (tensor core, TMA store)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- tensor memory ----
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t *slot) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_free(uint32_t base) {     // the same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}
// tcgen05.ld.32x32b of 8 / 16 consecutive 32-bit columns (lane = accumulator row).  The registers are undefined until
// tmem_wait_ld(): the _nowait forms let several loads fly behind one wait, tmem_ld8 / tmem_ld16 wait before returning.
__device__ __forceinline__ void tmem_ld_raw(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_raw(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
template <bool WAIT, int N>
__device__ __forceinline__ void tmem_ld_f32(uint32_t taddr, float (&v)[N]) {
    uint32_t r[N];
    tmem_ld_raw(taddr, r);
    if constexpr (WAIT) tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, float (&v)[8]) { tmem_ld_f32<false>(taddr, v); }
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float (&v)[16]) { tmem_ld_f32<false>(taddr, v); }
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) { tmem_ld_f32<true>(taddr, v); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) { tmem_ld_f32<true>(taddr, v); }
__device__ __forceinline__ void tmem_st4(uint32_t taddr, float a, float b, float c, float d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(__float_as_uint(a)),
                 "r"(__float_as_uint(b)), "r"(__float_as_uint(c)), "r"(__float_as_uint(d)) : "memory");
}
__device__ __forceinline__ void tmem_zero8(uint32_t taddr) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(taddr), "r"(0u) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- descriptors ----
// K-major, SWIZZLE_NONE shared-memory matrix descriptor
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;
    return d;
}
// K-major SWIZZLE_64B operand: rows of 64 bytes, 8-row groups 512 bytes apart (LBO unused), layout type 4 in bits 61-63
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t saddr) { return make_desc(saddr, 16u, 512u) | (4ull << 61); }
// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, dense
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// kind::tf32 instruction descriptor: D = f32, A = B = tf32, both K-major, dense
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- MMAs and commits ----
// One lane of a converged warp.  MMA issue code belongs inside `if (elect_one())` (or leader_of_warp0()): ptxas then keeps the
// descriptors in uniform registers and emits back-to-back UTCHMMA.  `if (tid == 0)` / `if (lane == 0)` instead wraps every
// tcgen05 instruction in an ELECT / BRA.U.ANY waterfall loop (~100 cycles per MMA, profiles/r02z_mma_issue.txt).
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n\t.reg .pred pe;\n\telect.sync _|pe, 0xffffffff;\n\tselp.u32 %0, 1, 0, pe;\n\t}" : "=r"(p));
    return p != 0;
}
__device__ __forceinline__ bool leader_of_warp0() {   // 1-D blocks; every lane of warp 0 must reach the call
    return __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0) == 0 && elect_one();
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// accumulating bf16 MMA issued by an elect.sync inside the asm: every lane of the warp calls it.  An elect.sync per MMA costs
// 5 R2UR per MMA (~100 cycles measured in the cluster UNet): a run of MMAs belongs in one elect_one() branch instead.
__device__ __forceinline__ void mma_bf16_elect(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe, pa;\n\t"
        "setp.eq.b32 pa, 0, 0;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, pa;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
}
// one arrival on `bar` once every MMA this thread issued before has retired
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void commit_elect(uint32_t bar) {   // the same, from an elect.sync inside the asm
    asm volatile(
        "{\n\t"
        ".reg .pred pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}" ::"r"(bar) : "memory");
}
// the arrival at the same shared-memory offset of every CTA of the cluster named in cta_mask
__device__ __forceinline__ void mma_commit_multicast(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"(cta_mask)
                 : "memory");
}

// ---- clusters ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Remote 16-byte store whose completion is counted (in bytes) on an mbarrier of the destination CTA: the data is visible
// to whoever observes the barrier phase complete -- no cluster-scope fence on the producer.  The hardware cluster
// barrier costs MEMBAR.ALL.GPU + ERRBAR on every arrive.release (measured 1400 cycles per layer, profiles/r02i_trace.txt).
__device__ __forceinline__ void st_async4(uint32_t remote_addr, float4 v, uint32_t remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1,%2,%3,%4}, [%5];"
                 ::"r"(remote_addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(remote_bar) : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);   // .x = lo (low 16 bits), .y = hi
    return *reinterpret_cast<const uint32_t *>(&h);
}

// ---- host: the driver's cuTensorMapEncodeTiled, looked up once; nullptr when the driver does not provide it ----
inline PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
    static const PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                        q == cudaDriverEntryPointSuccess;
        (void)cudaGetLastError();
        return ok ? reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p) : nullptr;
    }();
    return fn;
}

}  // namespace ptx
}  // namespace gc
