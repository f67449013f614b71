// fp32_pipes.cu -- how many FP32 operations per clock per SM the B200 sustains for scalar FFMA / FADD and for the
// packed FFMA2 / FADD2 (fma.rn.f32x2, add.rn.f32x2: sm_100 only).  Decides whether the Linearizer term of the fused
// kernel (~200 scalar FP32 instructions per accepted correspondence) should be written with packed operations; it is
// (term_add_e in corr_lin.cuh).  Build: nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o fp32_pipes fp32_pipes.cu
#include <cstdio>
#include <cuda_runtime.h>

template <int MODE>
__global__ void __launch_bounds__(256) k(float *out, int iters, float a, float b) {
  // 8 independent chains per thread (FFMA latency 4, so 8 chains keep the pipe full at 8 warps / SMSP)
  float x[8];
  unsigned long long p[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    x[i] = threadIdx.x * 0.001f + i;
    p[i] = ((unsigned long long)__float_as_uint(x[i]) << 32) | __float_as_uint(x[i] + 0.5f);
  }
  const unsigned long long pa = ((unsigned long long)__float_as_uint(a) << 32) | __float_as_uint(a);
  const unsigned long long pb = ((unsigned long long)__float_as_uint(b) << 32) | __float_as_uint(b);
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      if (MODE == 0) x[i] = fmaf(x[i], a, b);
      if (MODE == 1) x[i] = __fadd_rn(x[i], b);
      if (MODE == 2) asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(p[i]) : "l"(pa), "l"(pb));
      if (MODE == 3) asm volatile("add.rn.f32x2 %0, %0, %1;" : "+l"(p[i]) : "l"(pb));
      if (MODE == 4) asm volatile("mul.rn.f32x2 %0, %0, %1;" : "+l"(p[i]) : "l"(pa));
      if (MODE == 5) { x[i] = fmaf(x[i], a, b); asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(p[i]) : "l"(pa), "l"(pb)); }
    }
  }
  float s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += x[i] + __uint_as_float((unsigned)p[i]) + __uint_as_float((unsigned)(p[i] >> 32));
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <int MODE>
static void run(const char *name, int opsPerInstr, int instrPerIter) {
  int dev = 0, sms = 0, khz = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev);
  const int blocks = sms * 8, iters = 1 << 14;
  float *out;
  cudaMalloc(&out, blocks * 256 * sizeof(float));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  k<MODE><<<blocks, 256>>>(out, 64, 1.0001f, 0.001f);
  float best = 1e30f;
  for (int r = 0; r < 5; r++) {
    cudaEventRecord(e0);
    k<MODE><<<blocks, 256>>>(out, iters, 1.0001f, 0.001f);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  const double warpInstr = (double)blocks * 8 * iters * 8 * instrPerIter;
  const double perSmPerUs = warpInstr / sms / (best * 1e3);
  printf("%-28s %8.3f ms  %7.1f warp-instr/us/SM  = %.2f warp-instr/clk/SM at %d MHz nominal, %.1f TFLOP-equivalent lanes/s\n", name,
         best, perSmPerUs, perSmPerUs / (khz / 1e3), khz / 1000, warpInstr * 32 * opsPerInstr / (best * 1e-3) / 1e12);
  cudaFree(out);
}

// dependent-issue latency: one warp, one chain
template <int MODE>
__global__ void klat(float *out, int iters, float a, float b, long long *cycles) {
  float x = threadIdx.x * 0.001f;
  unsigned long long p = ((unsigned long long)__float_as_uint(x) << 32) | __float_as_uint(x + 0.5f);
  const unsigned long long pa = ((unsigned long long)__float_as_uint(a) << 32) | __float_as_uint(a);
  const unsigned long long pb = ((unsigned long long)__float_as_uint(b) << 32) | __float_as_uint(b);
  long long t0 = clock64();
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 16; i++) {
      if (MODE == 0) x = fmaf(x, a, b);
      if (MODE == 1) asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(p) : "l"(pa), "l"(pb));
      if (MODE == 2) asm volatile("add.rn.f32x2 %0, %0, %1;" : "+l"(p) : "l"(pb));
    }
  }
  long long t1 = clock64();
  out[threadIdx.x] = x + __uint_as_float((unsigned)p) + __uint_as_float((unsigned)(p >> 32));
  if (threadIdx.x == 0) *cycles = t1 - t0;
}
template <int MODE>
static void lat(const char *name) {
  float *out;
  long long *cyc, h = 0;
  cudaMalloc(&out, 32 * sizeof(float));
  cudaMalloc(&cyc, sizeof(long long));
  const int iters = 4096;
  klat<MODE><<<1, 32>>>(out, iters, 1.0001f, 0.001f, cyc);
  klat<MODE><<<1, 32>>>(out, iters, 1.0001f, 0.001f, cyc);
  cudaMemcpy(&h, cyc, sizeof h, cudaMemcpyDeviceToHost);
  printf("%-28s dependent-chain latency %.2f cycles\n", name, (double)h / (iters * 16.0));
  cudaFree(out);
  cudaFree(cyc);
}

int main() {
  lat<0>("FFMA");
  lat<1>("FFMA2");
  lat<2>("FADD2");
  run<0>("FFMA (scalar, 3-reg)", 1, 1);
  run<1>("FADD (scalar)", 1, 1);
  run<2>("FFMA2 (fma.rn.f32x2)", 2, 1);
  run<3>("FADD2 (add.rn.f32x2)", 2, 1);
  run<4>("FMUL2 (mul.rn.f32x2)", 2, 1);
  run<5>("FFMA + FFMA2 interleaved", 3, 2);
  return 0;
}
