// cml_common.cuh -- shared declarations of the carmel_b200 device library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/carmel_b200.h"

#define CML_SM_COUNT_FALLBACK 148

#define CML_CUDA(call)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (call);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(_e);                       \
      return CML_ERR_CUDA;                                                                 \
    }                                                                                      \
  } while (0)

// Per-example descriptor of the layered-CSR layout (32-byte aligned, read once per example).
struct __align__(16) CmlExDesc {
  uint64_t arc_base;    // first arc of this example in in_arc / out_arc
  uint64_t row_base;    // first row-offset entry (n_states+1 entries) in in_off / out_off
  uint64_t lvl_base;    // first entry (n_levels+1 entries) in lvl_off
  uint64_t scratch_base;  // first state slot in the global alpha/beta scratch (GLOBAL class only)
  uint32_t n_states;
  uint32_t n_levels;
  uint32_t fin;         // layered index of the goal state (start is layered index 0)
  uint32_t ex_index;    // index of the example within its batch (for ex_lnp)
  double weight;        // example weight
  double ln_weight;     // ln(weight)
};

// splitmix64 finaliser: the mixing step of every counter-based uniform (Gibbs samplers, cml_sample)
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// sample_uniform(seed, key, r, t) of include/carmel_b200.h (cml_sample, cml_forests_sample), with
// h0 = mix64(seed ^ mix64(key)) computed once per lattice or forest
__host__ __device__ __forceinline__ double sample_uniform(uint64_t h0, uint32_t r, uint32_t t) {
  const uint64_t h = mix64(h0 + (((uint64_t)r << 32) | t));
  return (double)(h >> 11) * (1.0 / 9007199254740992.0);
}

// Two CUDA events that bracket a call's kernels (its kernel time), destroyed on every return path
struct EventPair {
  cudaEvent_t a = nullptr, b = nullptr;
  cudaError_t create() {
    const cudaError_t e = cudaEventCreate(&a);
    return e != cudaSuccess ? e : cudaEventCreate(&b);
  }
  ~EventPair() {
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
  }
  EventPair() {}
  EventPair(EventPair const&) = delete;
  EventPair& operator=(EventPair const&) = delete;
};

template <typename T>
struct DevArray {
  T* p = nullptr;
  size_t n = 0;
  cudaError_t alloc(size_t count) {
    release();
    n = count;
    if (!count) return cudaSuccess;
    return cudaMalloc((void**)&p, count * sizeof(T));
  }
  // always allocates at least one element so kernels never see a null table
  cudaError_t upload(const T* h, size_t count, cudaStream_t s) {
    cudaError_t e = alloc(count ? count : 1);
    if (e != cudaSuccess) return e;
    if (!count || !h) return cudaMemsetAsync(p, 0, sizeof(T), s);  // (kernels that walk `n` elements see a defined value)
    return cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s);
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  ~DevArray() { release(); }
  DevArray() {}
  DevArray(DevArray const&) = delete;
  DevArray& operator=(DevArray const&) = delete;
};
