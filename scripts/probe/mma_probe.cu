// Timing probe: cycles per tcgen05.mma (kind::f16, M = 128, K = 16) as a function of N and of the shared-memory operand layout.
// Not part of the library; built by scripts/probe/build.sh and run on the GPU box by hand.  Operand contents are irrelevant.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "../../gencomm_b200/csrc/ptx.cuh"
using namespace gc::ptx;

__device__ __forceinline__ uint64_t desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
    return make_desc(saddr, lbo, sbo) | ((uint64_t)layout << 61);
}

// ASTEP / BSTEP: descriptor address increment (16-byte units) between consecutive MMAs, cycling over 8 positions
// ACC: number of distinct accumulators cycled (columns apart N)
template <int N, int LBO_A, int SBO_A, int AOFF, int LAY, int ASTEP, int LBO_B, int SBO_B, int BSTEP, int ACC, int AREP>
__global__ void __launch_bounds__(128, 1) k_probe(long long *out, int slot) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t s_tmem;
    const int warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 200 * 1024 / 4; i += 128) ((uint32_t *)smem)[i] = 0x3c003c00u + i;
    if (warp == 0) tmem_alloc<512>(&s_tmem);
    if (threadIdx.x == 32) { mbar_init(smem_u32(&bar), 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    if (warp == 1) {
        if (elect_one()) {
            const uint32_t base = (smem_u32(smem) + 1023u) & ~1023u;
            const uint64_t a0 = desc(base + AOFF, LBO_A, SBO_A, LAY);
            const uint64_t b0 = desc(base + 128 * 1024, LBO_B, SBO_B, LAY);
            constexpr uint32_t idesc = make_idesc(128, N);
            constexpr int kReps = 16, kInner = 48;
            const long long t0 = clock64();
#pragma unroll 1
            for (int rep = 0; rep < kReps; ++rep) {
#pragma unroll
                for (int i = 0; i < kInner; ++i) {
                    mma_bf16(tmem + (uint32_t)((i / 6 % ACC) * N), a0 + (uint64_t)(((i / AREP) % 8) * ASTEP), b0 + (uint64_t)((i % 8) * BSTEP), idesc, 1u);
                }
            }
            mma_commit(smem_u32(&bar));
            mbar_wait(smem_u32(&bar), 0);
            const long long t1 = clock64();
            out[slot] = (t1 - t0) * 100 / (kReps * kInner);
        }
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free<512>(tmem);
}

static long long *d_out;
static int n_slot = 0;
static const char *names[64];
template <int N, int LBO_A, int SBO_A, int AOFF, int LAY, int ASTEP, int LBO_B, int SBO_B, int BSTEP, int ACC, int AREP>
void run(const char *name, int ctas = 1) {
    auto k = k_probe<N, LBO_A, SBO_A, AOFF, LAY, ASTEP, LBO_B, SBO_B, BSTEP, ACC, AREP>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 201 * 1024);
    k<<<ctas, 128, 201 * 1024>>>(d_out, n_slot);
    k<<<ctas, 128, 201 * 1024>>>(d_out, n_slot);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: %s\n", name, cudaGetErrorString(e)); exit(1); }
    names[n_slot++] = name;
}

int main() {
    cudaMalloc(&d_out, 64 * sizeof(long long));
    cudaMemset(d_out, 0, 64 * sizeof(long long));
    constexpr int G = 6 * 130 * 16 + 16;   // conv_rows<64,4>: channel-group stride
    //   N   LBO_A SBO_A AOFF LAY ASTEP  LBO_B      SBO_B BSTEP ACC AREP
    run<64, G, 128, 0, 0, 130, 64 * 16, 128, 0, 4, 1>("N64 conv_rows layout, A row step, aligned");
    run<64, G, 128, 16, 0, 130, 64 * 16, 128, 0, 4, 1>("N64 conv_rows layout, A +16 B (kx shift)");
    run<64, G, 128, 0, 0, 0, 64 * 16, 128, 0, 4, 1>("N64 conv_rows layout, same A every MMA");
    run<64, 128, 256, 0, 0, 256, 128, 256, 0, 4, 1>("N64 dense no-swizzle (K-adjacent core matrices contiguous)");
    run<64, 2048, 128, 0, 0, 256, 1024, 128, 0, 4, 1>("N64 no-swizzle, LBO 2048 (M-contiguous, aligned)");
    run<64, 16, 1024, 0, 2, 512, 16, 1024, 0, 4, 1>("N64 SWIZZLE_128B");
    run<64, 16, 256, 0, 6, 256, 16, 256, 0, 4, 1>("N64 SWIZZLE_32B");
    run<64, 16, 512, 0, 4, 256, 16, 512, 0, 4, 1>("N64 SWIZZLE_64B");
    run<128, G, 128, 0, 0, 130, 128 * 16, 128, 0, 2, 1>("N128 conv_rows layout");
    run<128, 16, 1024, 0, 2, 512, 16, 1024, 0, 2, 1>("N128 SWIZZLE_128B");
    run<256, G, 128, 0, 0, 130, 256 * 16, 128, 0, 1, 1>("N256 conv_rows layout");
    run<256, 16, 1024, 0, 2, 512, 16, 1024, 0, 1, 1>("N256 SWIZZLE_128B");
    run<32, G, 128, 0, 0, 130, 32 * 16, 128, 0, 4, 1>("N32 conv_rows layout");
    run<32, 16, 1024, 0, 2, 512, 16, 1024, 0, 4, 1>("N32 SWIZZLE_128B");
    run<16, 16, 1024, 0, 2, 512, 16, 1024, 0, 4, 1>("N16 SWIZZLE_128B");
    run<64, G, 128, 0, 0, 130, 64 * 16, 128, 0, 4, 1>("N64 conv_rows layout, 148 CTAs", 148);
    long long h[64];
    cudaMemcpy(h, d_out, sizeof(h), cudaMemcpyDeviceToHost);
    for (int i = 0; i < n_slot; ++i) printf("%-62s %7.2f cycles/MMA\n", names[i], h[i] / 100.0);
    return 0;
}
