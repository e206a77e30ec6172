// micro-benchmark: throughput of fp64 count accumulation patterns on one B200 (round 2 design input)
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o profiles/micro/red_bench profiles/micro/red_bench.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
__device__ __forceinline__ uint32_t rng(uint32_t& s) { s = s * 1664525u + 1013904223u; return s >> 8; }
// mode 0: RED.F64 to random cell of n cells (x copies by block)   mode 1: RED.F32   mode 2: smem CAS double (per CTA table), flush at end
// mode 3: match_any aggregation then RED   mode 4: RED.F64 with zipf-ish skew (square of uniform)
template <int MODE>
__global__ void k(double* tab, float* tabf, uint32_t n, uint32_t copies, int iters, int skew) {
  extern __shared__ double sh[];
  uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u + 12345u;
  if (MODE == 2) { for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) sh[i] = 0; __syncthreads(); }
  double* t = tab + (size_t)(blockIdx.x % copies) * n;
  float* tf = tabf + (size_t)(blockIdx.x % copies) * n;
  for (int it = 0; it < iters; ++it) {
    uint32_t r = rng(s);
    uint32_t c;
    if (skew) { float u = (r & 0xffff) / 65536.f; c = (uint32_t)(u * u * u * n); } else c = r % n;
    if (c >= n) c = n - 1;
    double v = 1e-3 * (r & 7);
    if (MODE == 0) atomicAdd(&t[c], v);
    if (MODE == 1) atomicAdd(&tf[c], (float)v);
    if (MODE == 2) atomicAdd(&sh[c], v);
    if (MODE == 3) {
      unsigned m = __match_any_sync(0xffffffffu, c);
      int leader = __ffs(m) - 1;
      double sum = 0;
      for (unsigned mm = m; mm; mm &= mm - 1) sum += __shfl_sync(m, v, __ffs(mm) - 1);
      if ((threadIdx.x & 31) == leader) atomicAdd(&t[c], sum);
    }
  }
  if (MODE == 2) { __syncthreads(); for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) atomicAdd(&t[i], sh[i]); }
}
int main() {
  double* tab; float* tabf;
  const size_t cap = 64u << 20;
  cudaMalloc(&tab, cap * 8); cudaMalloc(&tabf, cap * 4);
  cudaMemset(tab, 0, cap * 8); cudaMemset(tabf, 0, cap * 4);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int grid = 148 * 3, block = 256, iters = 2000;
  auto run = [&](const char* name, int mode, uint32_t n, uint32_t copies, int skew) {
    float best = 1e9;
    for (int rep = 0; rep < 3; ++rep) {
      cudaEventRecord(e0);
      size_t sm = mode == 2 ? n * 8 : 0;
      switch (mode) {
        case 0: k<0><<<grid, block, sm>>>(tab, tabf, n, copies, iters, skew); break;
        case 1: k<1><<<grid, block, sm>>>(tab, tabf, n, copies, iters, skew); break;
        case 2: k<2><<<grid, block, sm>>>(tab, tabf, n, copies, iters, skew); break;
        case 3: k<3><<<grid, block, sm>>>(tab, tabf, n, copies, iters, skew); break;
      }
      cudaEventRecord(e1); cudaEventSynchronize(e1);
      float ms; cudaEventElapsedTime(&ms, e0, e1); if (ms < best) best = ms;
    }
    double ops = (double)grid * block * iters;
    printf("%-28s n=%8u copies=%3u skew=%d  %.3f ms  %.1f Gupd/s  err=%s\n", name, n, copies, skew, best, ops / best / 1e6, cudaGetErrorString(cudaGetLastError()));
  };
  for (int skew = 0; skew < 2; ++skew) {
    for (uint32_t n : {1024u, 16384u, 1u << 20}) for (uint32_t copies : {1u, 8u, 64u}) { if ((size_t)n * copies > cap) continue; run("RED.F64 global", 0, n, copies, skew); }
    run("RED.F32 global", 1, 1024, 64, skew);
    run("RED.F32 global", 1, 1u << 20, 1, skew);
    run("smem CAS f64 per CTA", 2, 1024, 64, skew);
    run("smem CAS f64 per CTA", 2, 4096, 64, skew);
    run("match_any + RED.F64", 3, 1024, 64, skew);
    run("match_any + RED.F64", 3, 1u << 20, 1, skew);
  }
  return 0;
}
