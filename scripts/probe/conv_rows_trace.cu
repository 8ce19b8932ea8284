// where the roles of one CTA of k_conv_rows wait at the backbone's level-1 / level-2 shapes (arbitrary operand contents).
#define CR_TRACE 1
#include <cstdarg>
#include <cstdio>
#include <vector>
#include "../../gencomm_b200/csrc/conv_rows.cu"
namespace gc { void set_error(const char *fmt, ...) { va_list ap; va_start(ap, fmt); vprintf(fmt, ap); va_end(ap); printf("\n"); } }

static void run(int A, int C, int NOUT, int H, int W) {
    const size_t plane = (size_t)A * H * W * C * 2, wbytes = (size_t)9 * C * NOUT * 4 + 65536, obytes = (size_t)A * H * W * NOUT * 2;
    void *xh, *xl, *w, *oh, *ol; float *bias;
    cudaMalloc(&xh, plane); cudaMalloc(&xl, plane); cudaMalloc(&w, wbytes); cudaMalloc(&oh, obytes); cudaMalloc(&ol, obytes);
    cudaMalloc(&bias, 4096);
    cudaMemset(xh, 0x3c, plane); cudaMemset(xl, 0x30, plane); cudaMemset(w, 0x38, wbytes); cudaMemset(bias, 0, 4096);
    gc::ConvLayer L;
    L.xh = (const uint4 *)xh; L.xl = (const uint4 *)xl; L.A = A; L.C = L.c_in = C; L.H_in = H; L.W_in = W;
    L.w = (const uint4 *)w; L.n_pad = L.n_out = L.out_ch_total = NOUT; L.bias = bias; L.epi = 5; L.oh = (uint4 *)oh; L.ol = (uint4 *)ol;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int it = 0; it < 3; ++it) {
        cudaEventRecord(e0);
        int rc = gc::conv_rows(0, L);
        cudaEventRecord(e1);
        cudaError_t e = cudaDeviceSynchronize();
        if (rc || e != cudaSuccess) { printf("failed rc=%d %s\n", rc, cudaGetErrorString(e)); exit(1); }
    }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    long long t[16];
    cudaMemcpyFromSymbol(t, gc::cr::g_trace, sizeof(t));
    printf("A=%d C=%d NOUT=%d %dx%d: %.1f us | CTA 8 (last launch; counters accumulate over 3): %lld cycles; feeder waits: operand rows %lld, "
           "accumulator %lld, weights %lld, weight slot %lld; stagers wait for a free operand buffer %lld\n", A, C, NOUT, H, W, ms * 1e3f, t[5],
           t[0] / 3, t[1] / 3, t[2] / 3, t[3] / 3, t[4] / 3);
    { long long z[16] = {0}; cudaMemcpyToSymbol(gc::cr::g_trace, z, sizeof(z)); }
    cudaFree(xh); cudaFree(xl); cudaFree(w); cudaFree(oh); cudaFree(ol); cudaFree(bias);
}
int main() {
    run(32, 64, 64, 128, 256);
    cudaMemset(nullptr, 0, 0);
    run(32, 128, 128, 64, 128);
    return 0;
}
