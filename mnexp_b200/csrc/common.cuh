// Shared device helpers for the LSTUR sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/lstur_b200.h"

namespace lstur {

void set_error(const char* fmt, ...);
extern unsigned long long g_launch_count;   // kernels launched through this library (bench.py: gpu_launches)

#define LSTUR_CHECK_LAUNCH(name)                                              \
  do {                                                                        \
    ++lstur::g_launch_count;                                                  \
    cudaError_t e__ = cudaGetLastError();                                     \
    if (e__ != cudaSuccess) {                                                 \
      lstur::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
      return LSTUR_ERR_CUDA;                                                  \
    }                                                                         \
  } while (0)

#define LSTUR_REQUIRE(cond, name)                                             \
  do {                                                                        \
    if (!(cond)) {                                                            \
      lstur::set_error("%s: invalid argument: %s", name, #cond);              \
      return LSTUR_ERR_ARG;                                                   \
    }                                                                         \
  } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// Widest CTA a kernel can be launched with on the current device (its register count included); 0 if the query fails.
static inline int kernel_max_threads(const void* fn) {
  cudaFuncAttributes a{};
  return cudaFuncGetAttributes(&a, fn) == cudaSuccess ? a.maxThreadsPerBlock : 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ int warp_or(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v |= __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Counter-based RNG for dropout: lowbias32 of (index, seed).  The same
// function is replicated in numpy by mnexp_b200/rng.py so that tests can hand
// the exact mask to the oracle.
__device__ __host__ __forceinline__ uint32_t lowbias32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du;
  x ^= x >> 15; x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}

__device__ __host__ __forceinline__ uint32_t rng_u32(uint32_t seed, uint64_t idx) {
  uint32_t lo = (uint32_t)idx, hi = (uint32_t)(idx >> 32);
  return lowbias32(lo ^ lowbias32(hi + 0x9e3779b9u * (seed + 1u)));
}

// ---- tensor-core path dropout stream ("quad stream"): one hash per FOUR consecutive elements.
// quad index q = element >> 2;  a = lo32(q) ^ key(hi32(q), seed);  b = fold(a * M1);  u0 = fold((b ^ C0) * M2),
// u1 = fold((b ^ C1) * M3)  with fold(x*y) = lo32 ^ hi32 of the 64-bit product.  Element k of the quad keeps iff the
// 15-bit field (u[k>>1] >> 16*(k&1)) & 0x7fff >= thr15 = floor(p * 32768).  ~3.75 integer ops per element (hash +
// mask) against ~10 for lowbias32 per pair with 16-bit compares; replicated in mnexp_b200/rng.py (quad_keep).
__device__ __host__ __forceinline__ uint32_t quad_key(uint32_t hi, uint32_t seed) {
  return lowbias32(hi + 0x9e3779b9u * (seed + 1u));
}
__device__ __host__ __forceinline__ uint32_t mulfold(uint32_t a, uint32_t m) {
  const unsigned long long p = (unsigned long long)a * (unsigned long long)m;
  return (uint32_t)p ^ (uint32_t)(p >> 32);
}
__device__ __host__ __forceinline__ void quad_hash(uint32_t a, uint32_t& u0, uint32_t& u1) {
  const uint32_t b = mulfold(a, 0x9E3779B1u);
  u0 = mulfold(b ^ 0x85EBCA6Bu, 0xC2B2AE35u);
  u1 = mulfold(b ^ 0x27D4EB2Fu, 0x165667B1u);
}
__device__ __host__ __forceinline__ uint32_t quad_thr15(float p) { return (uint32_t)(p * 32768.0f); }
// addend that moves "field >= thr15" into bit 15 of each 16-bit half (no carry between the halves)
__device__ __host__ __forceinline__ uint32_t quad_addend(uint32_t thr15) { return (0x8000u - thr15) * 0x10001u; }
#ifdef __CUDACC__
// 0xffff in each half whose 15-bit field is >= thr15 (addend = quad_addend(thr15)): AND, ADD, one byte-permute that
// replicates the sign bits of bytes 1 and 3
__device__ __forceinline__ uint32_t quad_mask(uint32_t u, uint32_t addend) {
  const uint32_t t = (u & 0x7fff7fffu) + addend;
  uint32_t m;
  asm("prmt.b32 %0, %1, %1, 0xBB99;" : "=r"(m) : "r"(t));
  return m;
}
#endif

// keep-probability threshold on the top 24 bits: keep iff (u >> 8) >= thr.
__device__ __host__ __forceinline__ uint32_t dropout_threshold(float p) {
  return (uint32_t)(p * 16777216.0f);
}

__device__ __forceinline__ float hard_sigmoid_f(float x) { return fminf(fmaxf(0.2f * x + 0.5f, 0.f), 1.f); }

}  // namespace lstur
