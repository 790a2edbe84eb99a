// microbench_casc.cu -- the k_chain3 section step (skewed cascade of CH sections in registers) in isolation:
// does it matter where the coefficients come from?  MODE 0: 5*CH coefficient registers per lane (what k_chain3 does: the
// chain of a warp is only known at run time -- but see MODE 2: with a block-uniform address ptxas keeps them in UNIFORM registers);
// MODE 2: 5*CH coefficient VECTOR registers (lane-dependent address), k_chain3's real situation; MODE 1: constant-bank operands with compile-time offsets (c[bank][imm]
// operands: two register sources per IMAD.WIDE instead of three).  W warps per sub-partition, one CTA per SM.
// MODE 3: the unit-gain form of kernel_chain3.cu (unitStep: z += a1 d1 + a2 d2, y = x + (z >> 28), two sticky records), vector-register
// coefficients as in MODE 2.  Rates count 5 MACs per section in every mode, so cycles per MAC compare the cost of a section.
#include <cstdio>
#include <cuda_runtime.h>

__device__ __forceinline__ int opaque(int v) { asm volatile("" : "+r"(v)); return v; }
__device__ __forceinline__ long long mac32(long long acc, int a, int b) { return acc + (long long)opaque(a) * (long long)opaque(b); }
__device__ __forceinline__ long long mac32c(long long acc, int a, int b) { return acc + (long long)opaque(a) * (long long)b; }
__device__ __forceinline__ int lo32(long long v) { int l, h; asm("mov.b64 {%0,%1}, %2;" : "=r"(l), "=r"(h) : "l"(v)); (void)h; return l; }
__device__ __forceinline__ int hi32(long long v) { int l, h; asm("mov.b64 {%0,%1}, %2;" : "=r"(l), "=r"(h) : "l"(v)); (void)l; return h; }
__device__ __forceinline__ int q59(long long a) { return (int)__funnelshift_r((unsigned)lo32(a), (unsigned)hi32(a), 28); }

__constant__ int cCoef[40];

template <int CH, int MODE>
__global__ void __launch_bounds__(512) k(long long* out, const int* __restrict__ coefG, int iters) {
    long long acc[CH];
    int y1[CH], y2[CH], y3[CH], X1 = threadIdx.x, X2 = 3;
    int b0[CH], b1[CH], b2[CH], a1[CH], a2[CH];
#pragma unroll
    for (int c = 0; c < CH; c++) {
        acc[c] = (long long)(threadIdx.x + c) * 0x100001ll; y1[c] = c; y2[c] = c + 1; y3[c] = c + 2;
        // MODE 2: the address depends on the lane, so ptxas cannot keep the coefficients in uniform registers (what k_chain3 gets:
        // its chain is a function of the warp id); MODE 0: block-uniform address -> ptxas promotes them to uniform registers
        const int* cf = coefG + 5 * c + (MODE == 2 ? (int)(threadIdx.x & 1) : (int)(blockIdx.x & 1));
        b0[c] = cf[0]; b1[c] = cf[1]; b2[c] = cf[2]; a1[c] = cf[3]; a2[c] = cf[4];
    }
    unsigned w0 = 0, w1 = 0, wx = 0;
    int xin = threadIdx.x * 77;
    long long z[CH]; int d1[CH], d2[CH];
#pragma unroll
    for (int c = 0; c < CH; c++) { z[c] = acc[c]; d1[c] = c; d2[c] = c + 1; }
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            long long a[CH];
            if (MODE == 3) {
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32(z[c], d1[c], a1[c]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32(a[c], d2[c], a2[c]);
                int y[CH];
#pragma unroll
                for (int c = 0; c < CH; c++) {
                    const int s = q59(a[c]);
                    if (c & 1) w1 = max(w1, (unsigned)hi32(a[c]) + 0x100000u); else w0 = max(w0, (unsigned)hi32(a[c]) + 0x100000u);
                    y[c] = (c ? y1[c - 1] : xin) + s;
                    z[c] = a[c]; d2[c] = d1[c]; d1[c] = s;
                }
                wx = max(wx, (unsigned)xin + 0x78000000u);
#pragma unroll
                for (int c = 0; c < CH; c++) { y3[c] = y2[c]; y2[c] = y1[c]; y1[c] = y[c]; }
                X2 = X1; X1 = xin; xin = xin * 5 + 1;
                continue;
            }
            if (MODE == 0 || MODE == 2) {
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32(acc[c], c ? y2[c - 1] : X1, b1[c]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32(a[c], c ? y3[c - 1] : X2, b2[c]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32(a[c], y1[c], a1[c]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32(a[c], y2[c], a2[c]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32(a[c], c ? y1[c - 1] : xin, b0[c]);
            } else {
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32c(acc[c], c ? y2[c - 1] : X1, cCoef[5 * c + 1]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32c(a[c], c ? y3[c - 1] : X2, cCoef[5 * c + 2]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32c(a[c], y1[c], cCoef[5 * c + 3]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32c(a[c], y2[c], cCoef[5 * c + 4]);
#pragma unroll
                for (int c = 0; c < CH; c++) a[c] = mac32c(a[c], c ? y1[c - 1] : xin, cCoef[5 * c]);
            }
#pragma unroll
            for (int c = 0; c < CH; c++) {
                if (c & 1) w1 = max(w1, (unsigned)hi32(a[c]) + 0x7fffffeu); else w0 = max(w0, (unsigned)hi32(a[c]) + 0x7fffffeu);
                acc[c] = a[c]; y3[c] = y2[c]; y2[c] = y1[c]; y1[c] = q59(a[c]);
            }
            X2 = X1; X1 = xin; xin = xin * 5 + 1;
        }
    }
    long long s = w0 ^ w1 ^ wx;
#pragma unroll
    for (int c = 0; c < CH; c++) s ^= acc[c] + z[c] + y1[c] + y3[c];
    if (s == 0x123456789abcdefll) out[0] = s;
}

template <int CH, int MODE> void run(int W, int iters, const int* dCoef) {
    int dev; cudaGetDevice(&dev); cudaDeviceProp p; cudaGetDeviceProperties(&p, dev);
    long long* d; cudaMalloc(&d, 8);
    const int blocks = p.multiProcessorCount, threads = 128 * W;
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    k<CH, MODE><<<blocks, threads>>>(d, dCoef, iters / 8 + 1);
    double best = 0;
    for (int rep = 0; rep < 3; rep++) {
        cudaEventRecord(a); k<CH, MODE><<<blocks, threads>>>(d, dCoef, iters); cudaEventRecord(b); cudaEventSynchronize(b);
        float ms; cudaEventElapsedTime(&ms, a, b);
        const double rate = (double)blocks * threads * CH * 5.0 * 4.0 * iters / (ms * 1e-3);
        if (rate > best) best = rate;
    }
    int clk; cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, dev);
    const double perClkSM = best / (p.multiProcessorCount * (double)clk * 1e3);
    printf("{\"sections\": %d, \"coefficients\": \"%s\", \"warps_per_subpartition\": %d, \"T_mac_per_s\": %.3f, \"mac_per_clk_per_SM\": %.2f, "
           "\"cycles_per_warp_mac_per_subpartition\": %.2f}\n", CH, MODE == 1 ? "constant bank" : MODE == 2 ? "vector registers" : MODE == 3 ? "vector registers, unit-gain form" : "uniform registers", W, best / 1e12, perClkSM, 128.0 / perClkSM);
    cudaFree(d);
}

int main(int argc, char**) {
    int h[48]; for (int i = 0; i < 48; i++) h[i] = 0x0123457 * (i + 3);
    int* dCoef; cudaMalloc(&dCoef, sizeof h); cudaMemcpy(dCoef, h, sizeof h, cudaMemcpyHostToDevice);
    cudaMemcpyToSymbol(cCoef, h, 40 * sizeof(int));
    if (argc > 1) {          // "unitgain": the general and the unit-gain part side by side, parts of 3 and 4 sections
        for (int W : {2, 3}) { run<4, 2>(W, 2048, dCoef); run<4, 3>(W, 2048, dCoef); run<3, 2>(W, 2048, dCoef); run<3, 3>(W, 2048, dCoef); }
        return 0;
    }
    for (int W : {1, 2, 3, 4}) run<8, 0>(W, 2048, dCoef);
    for (int W : {1, 2, 3, 4}) run<8, 1>(W, 2048, dCoef);
    for (int W : {1, 2, 3, 4}) run<4, 0>(W, 2048, dCoef);
    for (int W : {1, 2, 3, 4}) run<4, 1>(W, 2048, dCoef);
    for (int W : {2, 3, 4}) run<3, 0>(W, 2048, dCoef);
    for (int W : {2, 3, 4}) run<3, 1>(W, 2048, dCoef);
    for (int W : {1, 2, 3, 4}) run<8, 2>(W, 2048, dCoef);
    for (int W : {1, 2, 3, 4}) run<4, 2>(W, 2048, dCoef);
    for (int W : {2, 3, 4}) run<3, 2>(W, 2048, dCoef);
    return 0;
}
