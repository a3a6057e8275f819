// Shared helpers for libmelissa_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/melissa_b200.h"

void mls_set_error(const char* fmt, ...);
void mls_count_launch(int n = 1);
extern "C" int mls_get_option(const char* key);
// grid of a persistent kernel (a CTA loops over tiles blockIdx.x, blockIdx.x + gridDim.x, ...) under option "max_ctas"
int mls_cap_grid(int grid);

#define MLS_CHECK_ARG(cond, ...)          \
  do {                                    \
    if (!(cond)) {                        \
      mls_set_error(__VA_ARGS__);         \
      return MLS_ERR_INVALID;             \
    }                                     \
  } while (0)

#define MLS_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      mls_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return MLS_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define MLS_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    cudaError_t e_ = cudaGetLastError();                                                 \
    if (e_ != cudaSuccess) {                                                             \
      mls_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
      return MLS_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

// Philox4x32-10 (Salmon et al.), counter-based: same (key, counter) -> same 4 words on
// every launch geometry.  Used for movement offsets and epsilon-greedy draws.
struct Philox4 {
  uint32_t v[4];
};
__host__ __device__ inline Philox4 philox4x32_10(uint64_t key, uint64_t ctr_lo, uint64_t ctr_hi) {
  uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
  uint32_t c0 = (uint32_t)ctr_lo, c1 = (uint32_t)(ctr_lo >> 32), c2 = (uint32_t)ctr_hi, c3 = (uint32_t)(ctr_hi >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  Philox4 o;
  o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
  return o;
}
// 53-bit uniform in [0,1) from two 32-bit words (same construction numpy uses for doubles).
__host__ __device__ inline double u01_from_u32x2(uint32_t a, uint32_t b) {
  return (double)(((uint64_t)(a >> 5) << 26) | (uint64_t)(b >> 6)) * (1.0 / 9007199254740992.0);
}
