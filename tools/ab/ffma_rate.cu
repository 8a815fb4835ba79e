// Microbenchmark: FP32 FMA issue rates on sm_100a by operand form, to bound the depthwise kernel (csrc/dwconv.cu).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/ab/ffma_rate tools/ab/ffma_rate.cu && tools/ab/ffma_rate
// One CTA of 512 threads per SM (4 warps per scheduler); every variant runs ITERS x 16 independent FMA(2)s per thread
// and reports FMA lanes per clock per SM from clock64().
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>

constexpr int ITERS = 4096;
__constant__ float cw[64];

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

template <int V>
__global__ void __launch_bounds__(512, 1) rate(const float* __restrict__ in, float* __restrict__ out, long long* cyc) {
  float x[16], w[16], acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    x[i] = in[threadIdx.x + 512 * i];
    w[i] = in[threadIdx.x + 512 * (16 + i)];
    acc[i] = 0.f;
  }
  __syncthreads();
  const long long t0 = clock64();
  if (V == 0) {  // FFMA, three distinct registers
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(x[i], w[i], acc[i]);
  } else if (V == 1) {  // FFMA, one operand shared by consecutive instructions (reuse cache)
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(x[it & 1], w[i], acc[i]);
  } else if (V == 2) {  // FFMA2, distinct register pairs
    float2* a2 = reinterpret_cast<float2*>(acc);
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int i = 0; i < 8; ++i)
          a2[i] = ffma2(make_float2(x[2 * i], x[2 * i + 1]), make_float2(w[2 * i], w[2 * i + 1]), a2[i]);
  } else if (V == 3) {  // FFMA2, shared multiplicand (the depthwise kernel's pattern)
    float2* a2 = reinterpret_cast<float2*>(acc);
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int i = 0; i < 8; ++i) a2[i] = ffma2(make_float2(x[r], x[r + 2]), make_float2(w[2 * i], w[2 * i + 1]), a2[i]);
  } else if (V == 4) {  // FFMA with a constant-bank multiplier
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(x[i], cw[i], acc[i]);
  } else if (V == 5) {  // FFMA with a constant-bank multiplier and shared x
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(x[it & 1], cw[i], acc[i]);
  } else if (V == 6) {  // FFMA2 with a constant-bank pair
    float2* a2 = reinterpret_cast<float2*>(acc);
    const float2* c2 = reinterpret_cast<const float2*>(cw);
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int i = 0; i < 8; ++i) a2[i] = ffma2(make_float2(x[2 * i], x[2 * i + 1]), c2[i + 8 * r], a2[i]);
  } else if (V == 7) {  // FFMA with an immediate multiplier
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(x[i], 1.0009765625f, acc[i]);
  } else if (V == 8) {  // FFMA with a warp-uniform (shared-memory broadcast -> uniform register?) multiplier
    __shared__ float sw[16];
    if (threadIdx.x < 16) sw[threadIdx.x] = in[threadIdx.x];
    __syncthreads();
    float u[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) u[i] = __shfl_sync(0xffffffffu, sw[i], 0);
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(x[i], u[i], acc[i]);
  }
  const long long t1 = clock64();
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i];
  out[blockIdx.x * 512 + threadIdx.x] = s;
  if (threadIdx.x == 0) cyc[blockIdx.x] = t1 - t0;
}

template <int V>
void run(const char* name, const float* in, float* out, long long* cyc, int sms) {
  rate<V><<<sms, 512>>>(in, out, cyc);
  rate<V><<<sms, 512>>>(in, out, cyc);
  cudaDeviceSynchronize();
  long long h[256];
  cudaMemcpy(h, cyc, sizeof(long long) * sms, cudaMemcpyDeviceToHost);
  double mean = 0;
  for (int i = 0; i < sms; ++i) mean += h[i];
  mean /= sms;
  printf("%-48s %8.0f cycles  %6.1f FMA lanes/clk/SM\n", name, mean, 512.0 * 16 * ITERS / mean);
}

int main() {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  float *in, *out;
  long long* cyc;
  cudaMalloc(&in, 512 * 32 * 4);
  cudaMalloc(&out, 512 * 256 * 4);
  cudaMalloc(&cyc, 256 * 8);
  float h[512 * 32];
  for (int i = 0; i < 512 * 32; ++i) h[i] = 1.0f + (rand() % 1000) * 1e-6f;
  cudaMemcpy(in, h, sizeof(h), cudaMemcpyHostToDevice);
  cudaMemcpyToSymbol(cw, h, 64 * 4);
  run<0>("FFMA  r,r,r distinct", in, out, cyc, sms);
  run<1>("FFMA  shared multiplicand (reuse)", in, out, cyc, sms);
  run<2>("FFMA2 distinct pairs", in, out, cyc, sms);
  run<3>("FFMA2 shared multiplicand (dw pattern)", in, out, cyc, sms);
  run<4>("FFMA  constant-bank multiplier", in, out, cyc, sms);
  run<5>("FFMA  constant-bank multiplier, shared x", in, out, cyc, sms);
  run<6>("FFMA2 constant-bank pair", in, out, cyc, sms);
  run<7>("FFMA  immediate multiplier", in, out, cyc, sms);
  run<8>("FFMA  warp-uniform multiplier", in, out, cyc, sms);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("error %s\n", cudaGetErrorString(e)); return 1; }
  return 0;
}
