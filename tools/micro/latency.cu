// Dependent-issue latencies on the box (one warp, one CTA): what a serial per-sample recurrence pays per operation.
// nvcc -O3 -gencode arch=compute_100a,code=sm_100a tools/micro/latency.cu -o tools/micro/latency && tools/micro/latency
#include <cstdio>
#include <cuda_runtime.h>
#define N 4096
__global__ void k(double* out, long long* cyc, double a, double b, float fa, float fb) {
    double x = a; float f = fa; long long t0, t1;
    t0 = clock64();
    #pragma unroll 16
    for (int i = 0; i < N; ++i) x = fma(x, b, a);
    t1 = clock64(); cyc[0] = t1 - t0;
    t0 = clock64();
    #pragma unroll 16
    for (int i = 0; i < N; ++i) x = x + b;
    t1 = clock64(); cyc[1] = t1 - t0;
    t0 = clock64();
    #pragma unroll 16
    for (int i = 0; i < N; ++i) f = fmaf(f, fb, fa);
    t1 = clock64(); cyc[2] = t1 - t0;
    t0 = clock64();
    #pragma unroll 16
    for (int i = 0; i < N; ++i) f = __shfl_sync(0xffffffffu, f, (threadIdx.x + 1) & 31);
    t1 = clock64(); cyc[3] = t1 - t0;
    t0 = clock64();
    #pragma unroll 16
    for (int i = 0; i < N; ++i) x = (double) ((float) x) + b;       // f64 -> f32 -> f64 round trip + add
    t1 = clock64(); cyc[4] = t1 - t0;
    __shared__ float sm[64];
    if (threadIdx.x < 32) { sm[threadIdx.x] = f; sm[threadIdx.x + 32] = f; }
    __syncthreads();
    t0 = clock64();
    int idx = threadIdx.x & 31;
    #pragma unroll 16
    for (int i = 0; i < N; ++i) idx = (int) sm[idx & 63] & 31;        // dependent shared-memory loads
    t1 = clock64(); cyc[5] = t1 - t0;
    t0 = clock64();
    #pragma unroll 16
    for (int i = 0; i < N; ++i) x = x / (b + x);                       // dependent IEEE double division
    t1 = clock64(); cyc[6] = t1 - t0;
    out[threadIdx.x] = x + f + idx;
}
// Dependent global-load chase (one lane): the round trip a warp pays for each global load it must wait on before it can issue the
// next one.  LDG.E.STRONG.GPU (ld.global.cg) skips L1, so a hop is an L2 hit or an L2 miss served from HBM.
#define HOPS 2048
__device__ unsigned long long g_chase_sink;
__global__ void chase(const unsigned* __restrict__ next, unsigned start, int hops, long long* cyc, long long* ns) {
    unsigned i = start;
    long long t0, t1, g0, g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0));
    t0 = clock64();
    for (int h = 0; h < hops; ++h) i = __ldcg(next + i);
    t1 = clock64();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    g_chase_sink = i;
    cyc[0] = t1 - t0; ns[0] = g1 - g0;
}
// A random cycle of HOPS hops over `span` bytes, one hop per distinct 128-byte line.
static void make_chain(unsigned* h, size_t span) {
    const size_t lines = span / 128, stride = lines / HOPS;
    unsigned long long s = 0x9E3779B97F4A7C15ull;
    unsigned order[HOPS];
    for (int j = 0; j < HOPS; ++j) order[j] = j;
    for (int j = HOPS - 1; j > 0; --j) { s = s * 6364136223846793005ull + 1442695040888963407ull; const int r = (int) ((s >> 33) % (j + 1)); const unsigned t = order[j]; order[j] = order[r]; order[r] = t; }
    for (int j = 0; j < HOPS; ++j) h[(size_t) order[j] * stride * 32] = (unsigned) ((size_t) order[(j + 1) % HOPS] * stride * 32);
}
int main() {
    double* o; long long* c; cudaMalloc(&o, 32 * 16 * 8); cudaMalloc(&c, 64);
    for (int warps = 1; warps <= 16; warps *= 4) {
        k<<<1, 32 * warps>>>(o, c, 1.0000001, 0.9999999, 1.0001f, 0.9999f);
        k<<<1, 32 * warps>>>(o, c, 1.0000001, 0.9999999, 1.0001f, 0.9999f);
        long long h[8];
        const cudaError_t e = cudaMemcpy(h, c, 56, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(e)); return 1; }
        printf("warps/CTA %2d  cycles per dependent op: DFMA %.1f  DADD %.1f  FFMA %.1f  SHFL %.1f  F64->F32->F64+DADD %.1f  LDS(dependent) %.1f  DDIV %.1f\n", warps,
               h[0] / (double) N, h[1] / (double) N, h[2] / (double) N, h[3] / (double) N, h[4] / (double) N, h[5] / (double) N, h[6] / (double) N);
    }
    // global round trips: spans of 8 MiB (inside the 126 MB L2) and 1 GiB; "flushed" = a 512 MiB memset right before the timed chase,
    // "resident" = the same chase run once before (so every line of it is in L2)
    const size_t flushBytes = (size_t) 512 << 20;
    void* flush; cudaMalloc(&flush, flushBytes);
    long long* ns; cudaMalloc(&ns, 8);
    const size_t spans[2] = {(size_t) 8 << 20, (size_t) 1 << 30};
    for (size_t span : spans) {
        unsigned* h = (unsigned*) calloc(span / 4, 4); make_chain(h, span);
        unsigned* d; cudaMalloc(&d, span); cudaMemcpy(d, h, span, cudaMemcpyHostToDevice); free(h);
        for (int rep = 0; rep < 3; ++rep) {
            long long cy[2], t[2];
            cudaMemset(flush, rep, flushBytes);
            chase<<<1, 1>>>(d, 0, HOPS, c, ns); cudaMemcpy(&cy[0], c, 8, cudaMemcpyDeviceToHost); cudaMemcpy(&t[0], ns, 8, cudaMemcpyDeviceToHost);
            chase<<<1, 1>>>(d, 0, HOPS, c, ns); cudaMemcpy(&cy[1], c, 8, cudaMemcpyDeviceToHost);
            const cudaError_t e = cudaMemcpy(&t[1], ns, 8, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(e)); return 1; }
            printf("dependent global load, span %5zu MiB, %d hops: L2 flushed %.0f cycles (%.0f ns) per hop, L2 resident %.0f cycles (%.0f ns) per hop\n",
                   span >> 20, HOPS, cy[0] / (double) HOPS, t[0] / (double) HOPS, cy[1] / (double) HOPS, t[1] / (double) HOPS);
        }
        cudaFree(d);
    }
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(e)); return 1; }
    return 0;
}
