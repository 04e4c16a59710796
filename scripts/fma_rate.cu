// FP32 FMA issue rate of the card: every thread runs 8 independent fmaf chains; prints FMAs per second (CUDA events).
// Built and run by scripts/umap_bench.py, which states the kNN rate against it.
#include <cstdio>
#include <cuda_runtime.h>

__global__ void k_fma(float* out, int iters, float a, float b) {
  float x[8];
  for (int c = 0; c < 8; ++c) x[c] = threadIdx.x * 1e-3f + c;
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int c = 0; c < 8; ++c) x[c] = fmaf(x[c], a, b);
  float s = 0;
  for (int c = 0; c < 8; ++c) s += x[c];
  if (s == 1234.5f) out[0] = s;
}

int main() {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  float* out;
  cudaMalloc(&out, 4);
  const int blocks = sms * 8, threads = 256, iters = 1 << 16;
  k_fma<<<blocks, threads>>>(out, 1024, 0.999f, 1e-3f);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  cudaEventRecord(a);
  for (int r = 0; r < 5; ++r) k_fma<<<blocks, threads>>>(out, iters, 0.999f, 1e-3f);
  cudaEventRecord(b);
  cudaEventSynchronize(b);
  float ms = 0;
  cudaEventElapsedTime(&ms, a, b);
  const double fmas = 5.0 * blocks * threads * (double)iters * 8;
  printf("%.6e\n", fmas / (ms * 1e-3));
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}
