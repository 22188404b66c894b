// Shared helpers for libgccvae: status/error plumbing, launch counting, Philox4x32-10, math.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "gccvae.h"
#include "gccvae_debug.h"

namespace gccvae {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define GCC_REQUIRE(cond, ...)          \
  do {                                  \
    if (!(cond)) {                      \
      ::gccvae::set_error(__VA_ARGS__); \
      return GCCVAE_EINVAL;             \
    }                                   \
  } while (0)

#define GCC_CHECK_LAUNCH(name)                                                          \
  do {                                                                                  \
    cudaError_t e__ = cudaGetLastError();                                               \
    if (e__ != cudaSuccess) {                                                           \
      ::gccvae::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));     \
      return GCCVAE_ECUDA;                                                              \
    }                                                                                   \
    ::gccvae::count_launch();                                                           \
  } while (0)

#define GCC_CUDA(call)                                                                  \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      ::gccvae::set_error("%s failed: %s", #call, cudaGetErrorString(e__));            \
      return GCCVAE_ECUDA;                                                              \
    }                                                                                   \
  } while (0)

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based generator (Salmon et al. 2011).  ctr = (index_lo, index_hi,
// stream id, per-step offset); key = seed.  Forward and backward kernels regenerate identical
// noise from identical counters, so no noise tensor ever touches HBM in RNG mode.
// ---------------------------------------------------------------------------------------------
enum PhiloxStream : uint32_t { PH_EPS = 0, PH_EPS_K = 1, PH_UY = 2, PH_GATE = 3, PH_IW_EPS = 4, PH_IW_UY = 5 };

__host__ __device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#ifdef __CUDA_ARCH__
  uint32_t hi0 = __umulhi(M0, c[0]), hi1 = __umulhi(M1, c[2]);
#else
  uint32_t hi0 = (uint32_t)(((uint64_t)M0 * c[0]) >> 32), hi1 = (uint32_t)(((uint64_t)M1 * c[2]) >> 32);
#endif
  uint32_t lo0 = M0 * c[0], lo1 = M1 * c[2];
  uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}

__host__ __device__ __forceinline__ void philox4x32(uint64_t seed, uint64_t offset, uint32_t stream,
                                                    uint64_t index, uint32_t (&out)[4]) {
  uint32_t c[4] = {(uint32_t)index, (uint32_t)(index >> 32), stream ^ (uint32_t)(offset >> 32) * 0x9E3779B9u,
                   (uint32_t)offset};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}

// uniform in [0,1): 24 random bits
__host__ __device__ __forceinline__ float u32_to_unit(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
// uniform in (0,1]
__host__ __device__ __forceinline__ float u32_to_unit_open0(uint32_t x) {
  return ((float)(x >> 8) + 1.0f) * (1.0f / 16777216.0f);
}

#ifdef __CUDACC__
// Launch of the prologue-less auxiliary kernels, WITHOUT the programmatic-stream-serialization attribute.
// Measured on B200: programmatic dependent launch pays for the tensor-core kernels (long prologues: 2.30 -> 2.10 ms
// per step) but NOT for these (2.10 -> 2.17 ms: their early-scheduled CTAs only occupy SM slots).
template <class... KArgs, class... Args>
static inline cudaError_t launch_aux(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
__device__ __forceinline__ void pdl_prologue() {   // let the successor start, then wait for the predecessor
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// four N(0,1) from one Philox block (Box-Muller on two pairs)
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint64_t offset, uint32_t stream, uint64_t index,
                                               float (&n)[4]) {
  uint32_t r[4];
  philox4x32(seed, offset, stream, index, r);
  float u0 = u32_to_unit_open0(r[0]), u1 = u32_to_unit(r[1]);
  float u2 = u32_to_unit_open0(r[2]), u3 = u32_to_unit(r[3]);
  float m0 = sqrtf(-2.0f * __logf(u0)), m1 = sqrtf(-2.0f * __logf(u2));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  n[0] = m0 * c0; n[1] = m0 * s0; n[2] = m1 * c1; n[3] = m1 * s1;
}

__device__ __forceinline__ float softplus_f(float x) { return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float clip_f(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
#endif

}  // namespace gccvae
