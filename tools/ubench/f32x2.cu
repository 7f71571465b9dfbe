// Microbenchmark: issue throughput and dependent latency of scalar vs packed fp32 (FFMA vs FFMA2,
// FADD vs FADD2), predicated FADD2, MUFU.EX2, FMNMX3 and mixes, per SM sub-partition on sm_100a.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o /tmp/ubench_f32x2 tools/ubench/f32x2.cu
#include <cstdio>
#include <cuda_runtime.h>

constexpr int ITERS = 4096;

template <int MODE, int ILP>
__global__ void k(float* out, unsigned long long* cyc, float seed) {
    float2 a[ILP];
    float s[ILP];
#pragma unroll
    for (int i = 0; i < ILP; ++i) { a[i] = make_float2(seed + i, seed * 0.5f + i); s[i] = seed + i; }
    const float2 m = make_float2(1.0001f, 0.9999f), c = make_float2(0.001f, -0.001f);
    __syncthreads();
    const unsigned long long t0 = clock64();
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it) {
#pragma unroll
        for (int i = 0; i < ILP; ++i) {
            if (MODE == 0) s[i] = fmaf(s[i], m.x, c.x);                       // FFMA
            if (MODE == 1) a[i] = __ffma2_rn(a[i], m, c);                      // FFMA2
            if (MODE == 2) s[i] = s[i] + c.x;                                 // FADD
            if (MODE == 3) a[i] = __fadd2_rn(a[i], c);                         // FADD2
            if (MODE == 4) { asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(s[i])); }   // MUFU
            if (MODE == 5) { s[i] = fmaf(s[i], m.x, c.x); a[i] = __ffma2_rn(a[i], m, c); }   // mix 1:1
            if (MODE == 6) { a[i] = __fadd2_rn(a[i], c); s[i] = fmaxf(s[i], a[i].x); }      // FADD2 + FMNMX (alu)
            if (MODE == 7) { asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(s[i])); a[i] = __ffma2_rn(a[i], m, c); }
        }
    }
    const unsigned long long t1 = clock64();
    float r = 0.f;
#pragma unroll
    for (int i = 0; i < ILP; ++i) r += a[i].x + a[i].y + s[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = r;
    if (threadIdx.x == 0 && blockIdx.x == 0) *cyc = t1 - t0;
}

template <int MODE, int ILP>
void run(const char* name, int warps_per_smsp, float* out, unsigned long long* cyc) {
    const int threads = warps_per_smsp * 4 * 32;
    k<MODE, ILP><<<148, threads>>>(out, cyc, 1.0f);
    cudaDeviceSynchronize();
    k<MODE, ILP><<<148, threads>>>(out, cyc, 1.0f);
    cudaDeviceSynchronize();
    unsigned long long h;
    cudaMemcpy(&h, cyc, 8, cudaMemcpyDeviceToHost);
    const double per = (double)h / ((double)ITERS * ILP * warps_per_smsp);
    printf("%-28s ILP %2d warps/SMSP %d : %.2f cycles per warp-instruction-slot per SMSP (latency-ish if 1 warp ILP 1: %.2f)\n", name, ILP,
           warps_per_smsp, per, (double)h / ((double)ITERS * ILP));
}

int main() {
    float* out; unsigned long long* cyc;
    cudaMalloc(&out, 148 * 1024 * 4); cudaMalloc(&cyc, 8);
    run<0, 1>("FFMA  chain", 1, out, cyc);
    run<1, 1>("FFMA2 chain", 1, out, cyc);
    run<2, 1>("FADD  chain", 1, out, cyc);
    run<3, 1>("FADD2 chain", 1, out, cyc);
    run<4, 1>("EX2   chain", 1, out, cyc);
    run<0, 8>("FFMA", 1, out, cyc);  run<0, 8>("FFMA", 4, out, cyc);
    run<1, 8>("FFMA2", 1, out, cyc); run<1, 8>("FFMA2", 4, out, cyc);
    run<2, 8>("FADD", 4, out, cyc);
    run<3, 8>("FADD2", 1, out, cyc); run<3, 8>("FADD2", 4, out, cyc);
    run<4, 8>("EX2", 1, out, cyc);   run<4, 8>("EX2", 4, out, cyc);
    run<5, 8>("FFMA+FFMA2 (per pair)", 4, out, cyc);
    run<6, 8>("FADD2+FMNMX (per pair)", 4, out, cyc);
    run<7, 8>("EX2+FFMA2 (per pair)", 4, out, cyc);
    return 0;
}
