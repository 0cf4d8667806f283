// Microbenchmark: the bf16 logit reads of the paste at stride 32 (64^3 windows, 32^3 cores).  A core row is the 64
// bytes [32, 96) of a 128-byte window row, so it straddles both 64-byte halves of the line; this times the read of
// every core of 2.1 GB of bf16 logits (far above L2) with each L2 prefetch-size qualifier, CUDA events, median of 20.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o bf16_core_read bf16_core_read.cu
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <vector>

template <int MODE>
__device__ __forceinline__ float ld(const __nv_bfloat16* p) {
  unsigned short h;
  if (MODE == 0) asm volatile("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(h) : "l"(p));
  if (MODE == 1) asm volatile("ld.global.nc.L1::no_allocate.L2::64B.b16 %0, [%1];" : "=h"(h) : "l"(p));
  if (MODE == 2) asm volatile("ld.global.nc.L1::no_allocate.L2::128B.b16 %0, [%1];" : "=h"(h) : "l"(p));
  if (MODE == 3) asm volatile("ld.global.nc.L1::no_allocate.L2::256B.b16 %0, [%1];" : "=h"(h) : "l"(p));
  return __uint_as_float((unsigned)h << 16);
}

// grid = (32 core planes, cubes * channels), block 256: the 32 x 32 core of one plane of one channel
template <int MODE>
__global__ void core_read(const __nv_bfloat16* __restrict__ in, float* __restrict__ out) {
  const __nv_bfloat16* plane = in + (size_t)blockIdx.y * 262144 + (size_t)(blockIdx.x + 16) * 4096;
  float acc = 0.f;
  for (int e = threadIdx.x; e < 1024; e += 256) acc += ld<MODE>(plane + ((e >> 5) + 16) * 64 + 16 + (e & 31));
  if (acc == 123.456f) out[0] = acc;
}

template <int MODE>
float run(const __nv_bfloat16* in, float* out, int n) {
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  std::vector<float> ts;
  for (int r = 0; r < 23; ++r) {
    cudaEventRecord(a);
    core_read<MODE><<<dim3(32, n), 256>>>(in, out);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    float ms;
    cudaEventElapsedTime(&ms, a, b);
    if (r >= 3) ts.push_back(ms);
  }
  std::sort(ts.begin(), ts.end());
  return ts[ts.size() / 2];
}

int main() {
  const int n = 4096;  // cube channels of 64^3 bf16: 2.1 GB
  __nv_bfloat16* in;
  float* out;
  if (cudaMalloc(&in, (size_t)n * 262144 * 2) != cudaSuccess || cudaMalloc(&out, 4) != cudaSuccess) return 1;
  cudaMemset(in, 0, (size_t)n * 262144 * 2);
  const double core_bytes = (double)n * 32 * 32 * 32 * 2;
  const char* names[4] = {"none", "L2::64B", "L2::128B", "L2::256B"};
  float t[4] = {run<0>(in, out, n), run<1>(in, out, n), run<2>(in, out, n), run<3>(in, out, n)};
  for (int m = 0; m < 4; ++m)
    printf("{\"qualifier\": \"%s\", \"ms\": %.4f, \"core_GBps\": %.1f}\n", names[m], t[m], core_bytes / (t[m] * 1e-3) / 1e9);
  cudaFree(in);
  cudaFree(out);
  return cudaGetLastError() != cudaSuccess;
}
