// Reconstruction log-likelihood (+ its gradient), Keras-semantics Adam, column sums, and the
// library's status plumbing.
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace gccvae {

static thread_local char g_err[512] = "";
static thread_local long long g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches += n; }

// ---------------------------------------------------------------------------------------------
// utils.py:101-105: log p(x|z) = sum_{h,w,c} Laplace(xhat,1).log_prob(x) = -|x-xhat|_1 - n ln2.
// One CTA per image (deterministic reduction order); optional fused gradient w.r.t. the
// decoder's pre-sigmoid logits:  dL/dlogit = coef[b] * sign(x - xhat) * xhat (1 - xhat).
// Algorithmic bytes per image: read x + xhat (2*49152 B), write dlogit (49152 B).
// ---------------------------------------------------------------------------------------------
template <bool GRAD>
__global__ void __launch_bounds__(256) recon_kernel(const float4* __restrict__ x, const float4* __restrict__ xh,
                                                    int vec_per_image, const float* __restrict__ coef,
                                                    float* __restrict__ log_pxz, float4* __restrict__ dlogit,
                                                    float n_ln2) {
  __shared__ float red[8];
  const int b = blockIdx.x;
  const size_t base = (size_t)b * vec_per_image;
  const float cb = GRAD ? coef[b] : 0.0f;
  float acc = 0.0f;
  for (int t = threadIdx.x; t < vec_per_image; t += 256) {
    const float4 a = __ldg(x + base + t), r = __ldg(xh + base + t);
    const float d0 = a.x - r.x, d1 = a.y - r.y, d2 = a.z - r.z, d3 = a.w - r.w;
    acc += (fabsf(d0) + fabsf(d1)) + (fabsf(d2) + fabsf(d3));
    if (GRAD) {
      float4 g;
      g.x = cb * ((d0 > 0.f) - (d0 < 0.f)) * r.x * (1.0f - r.x);
      g.y = cb * ((d1 > 0.f) - (d1 < 0.f)) * r.y * (1.0f - r.y);
      g.z = cb * ((d2 > 0.f) - (d2 < 0.f)) * r.z * (1.0f - r.z);
      g.w = cb * ((d3 > 0.f) - (d3 < 0.f)) * r.w * (1.0f - r.w);
      dlogit[base + t] = g;
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.0f;
#pragma unroll
    for (int q = 0; q < 8; ++q) tot += red[q];
    log_pxz[b] = -tot - n_ln2;
  }
}

// Keras 2.8 Adam.  `step_dev` (optional) holds t on the device so that a captured CUDA graph of the
// whole step can be replayed: bump_kernel increments it before every update.
// debug marker: records %globaltimer (ns) into slot idx; launched WITHOUT the PDL attribute, so it runs after
// everything before it on the stream has finished -> segment times of a captured graph
__global__ void mark_kernel(long long* buf, int idx) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  buf[idx] = (long long)t;
}

__global__ void bump_kernel(int* p) {
  pdl_prologue();
 *p += 1; }

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v, long long n,
                                                   float lr, float b1, float b2, float eps, int step,
                                                   const int* __restrict__ step_dev) {
  pdl_prologue();
  const int t = step_dev ? *step_dev : step;
  const float lr_t = (float)((double)lr * sqrt(1.0 - pow((double)b2, (double)t)) / (1.0 - pow((double)b1, (double)t)));
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float gi = g[i];
    const float mi = m[i] + (gi - m[i]) * (1.0f - b1);
    const float vi = v[i] + (gi * gi - v[i]) * (1.0f - b2);
    m[i] = mi;
    v[i] = vi;
    p[i] -= lr_t * mi / (sqrtf(vi) + eps);
  }
}

// The same update with the step bookkeeping inside: t = state[0] + 1 is used, the gradient buffer is cleared behind
// the read (the next backward accumulates into it: no separate memset on the step's critical path), and - when
// `publish` is set - the last block to finish publishes state[0] = t (state[1] is the ticket counter, left at 0).
// The element range [i0, n) lets the step run the update in two parts: everything but the first layer's parameters
// as soon as their gradients are complete (concurrently with the last dgrad), the rest at the very end (publishing).
__global__ void __launch_bounds__(256) adam_fused_kernel(float* __restrict__ p, float* __restrict__ g,
                                                         float* __restrict__ m, float* __restrict__ v, long long i0,
                                                         long long n, long long n_zero, float lr, float b1, float b2,
                                                         float eps, int* __restrict__ state, int publish,
                                                         const float* __restrict__ res_loss,
                                                         const float* __restrict__ res_c, float* __restrict__ ring,
                                                         int ring_slots) {
  pdl_prologue();
  const int t = state[0] + 1;
  // the step's results (loss, gate sample c) are copied into slot (t - 1) % ring_slots of a caller-owned ring by the
  // publishing launch: what train_step returns stays valid for ring_slots further steps although the step itself
  // (a replayed graph) always writes the same addresses
  if (publish && ring != nullptr && blockIdx.x == 0) {
    float* dst = ring + (size_t)((t - 1) % ring_slots) * GCCVAE_RESULT_SLOT_FLOATS;
    for (int i = threadIdx.x; i < 1 + GCCVAE_ZC * GCCVAE_Y; i += 256) dst[i] = i == 0 ? res_loss[0] : res_c[i - 1];
  }
  const float lr_t = (float)((double)lr * sqrt(1.0 - pow((double)b2, (double)t)) / (1.0 - pow((double)b1, (double)t)));
  for (long long i = i0 + blockIdx.x * 256LL + threadIdx.x; i < n_zero; i += (long long)gridDim.x * 256) {
    if (i < n) {
      const float gi = g[i];
      const float mi = m[i] + (gi - m[i]) * (1.0f - b1);
      const float vi = v[i] + (gi * gi - v[i]) * (1.0f - b2);
      m[i] = mi;
      v[i] = vi;
      p[i] -= lr_t * mi / (sqrtf(vi) + eps);
    }
    g[i] = 0.0f;
  }
  if (!publish) return;
  __syncthreads();                      // every thread of this block has read state[0]
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int ticket = atomicAdd(reinterpret_cast<unsigned int*>(state + 1), 1u);
    if (ticket == gridDim.x - 1) {      // all blocks have read t: publish the new step count, reset the ticket
      state[0] = t;
      state[1] = 0;
    }
  }
}

// out[c] = sum_r in[r, c].  Two deterministic stages: grid (col-blocks, row-splits) writes partial
// rows into the workspace, a second launch adds the splits in fixed order.
__global__ void __launch_bounds__(256) colsum_stage1(const float* __restrict__ in, long long rows, int cols,
                                                     int rows_per_split, float* __restrict__ part) {
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r0 = threadIdx.x >> 5;
  const long long rbeg = (long long)blockIdx.y * rows_per_split;
  long long rend = rbeg + rows_per_split;
  if (rend > rows) rend = rows;
  float acc = 0.0f;
  if (c < cols)
    for (long long r = rbeg + r0; r < rend; r += 8) acc += in[r * cols + c];
  red[r0][threadIdx.x & 31] = acc;
  __syncthreads();
  if (r0 == 0 && c < cols) {
    float tot = 0.0f;
#pragma unroll
    for (int q = 0; q < 8; ++q) tot += red[q][threadIdx.x];
    part[(size_t)blockIdx.y * cols + c] = tot;
  }
}
__global__ void colsum_stage2(const float* __restrict__ part, int splits, int cols, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float tot = 0.0f;
  for (int s = 0; s < splits; ++s) tot += part[(size_t)s * cols + c];
  out[c] = tot;
}

static int colsum_splits(long long rows, int cols) {
  const int colblocks = (cols + 31) / 32;
  long long want = (148LL * 4 + colblocks - 1) / colblocks;
  long long maxs = (rows + 63) / 64;
  if (want > maxs) want = maxs;
  if (want < 1) want = 1;
  return (int)want;
}

// forward-only loss value from the per-image terms (one CTA, fixed order)
__global__ void __launch_bounds__(256) elbo_loss_kernel(const float* __restrict__ terms,
                                                        const float* __restrict__ log_pxz, int B, int Bg, int sup,
                                                        const float* __restrict__ mu, float reg,
                                                        float* __restrict__ loss) {
  __shared__ float red[8];
  float acc = 0.0f;
  for (int b = threadIdx.x; b < B; b += 256) {
    const float kl = terms[b], lq = terms[(size_t)B + b], lqx = terms[2 * (size_t)B + b], w = terms[3 * (size_t)B + b],
                lpy = terms[4 * (size_t)B + b], lpx = log_pxz[b];
    acc += sup ? -(w * (lpx - kl - lq) + lpy + lqx) : -(lpx + lpy - kl - lq);
  }
  acc /= (float)Bg;
  if (mu != nullptr)
    for (int p = threadIdx.x; p < 324; p += 256) acc += reg * fabsf(mu[p]) / 324.0f;
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.0f;
    for (int q = 0; q < 8; ++q) t += red[q];
    loss[0] = t;
  }
}

}  // namespace gccvae

using namespace gccvae;

extern "C" int gccvae_elbo_loss_f32(const float* terms, const float* log_pxz, int batch, int batch_global,
                                    int supervised, const float* mu, float gating_reg, float* loss, void* stream) {
  GCC_REQUIRE(terms && log_pxz && loss && batch > 0 && batch_global >= batch, "elbo_loss: bad args");
  elbo_loss_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(terms, log_pxz, batch, batch_global, supervised, mu,
                                                        gating_reg, loss);
  GCC_CHECK_LAUNCH("elbo_loss");
  return GCCVAE_OK;
}

extern "C" int gccvae_abi_version(void) { return GCCVAE_ABI_VERSION; }
extern "C" const char* gccvae_last_error(void) { return g_err; }
extern "C" long long gccvae_launch_count(void) { return g_launches; }
extern "C" void gccvae_reset_launch_count(void) { g_launches = 0; }
extern "C" void gccvae_add_launch_count(long long n) { g_launches += n; }

extern "C" int gccvae_arch_check(int device) {
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    set_error("arch_check: cudaGetDeviceProperties(%d): %s", device, cudaGetErrorString(e));
    return GCCVAE_ECUDA;
  }
  if (prop.major != 10) {
    set_error("arch_check: device %d is sm_%d%d, this library is built for sm_100a only", device, prop.major,
              prop.minor);
    return GCCVAE_EARCH;
  }
  return GCCVAE_OK;
}

extern "C" int gccvae_recon_f32(const float* x, const float* xhat, int batch, int per_image, const float* coef,
                                float* log_pxz, float* dlogit, void* stream) {
  GCC_REQUIRE(x && xhat && log_pxz && batch > 0, "recon: null pointer / empty batch");
  GCC_REQUIRE(per_image > 0 && per_image % 4 == 0, "recon: per_image (%d) must be a multiple of 4", per_image);
  GCC_REQUIRE((dlogit == nullptr) == (coef == nullptr), "recon: coef and dlogit go together");
  GCC_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)xhat % 16 == 0) && ((uintptr_t)dlogit % 16 == 0),
              "recon: pointers must be 16-byte aligned");
  const float n_ln2 = (float)((double)per_image * 0.6931471805599453);
  if (dlogit)
    recon_kernel<true><<<batch, 256, 0, (cudaStream_t)stream>>>((const float4*)x, (const float4*)xhat, per_image / 4,
                                                                coef, log_pxz, (float4*)dlogit, n_ln2);
  else
    recon_kernel<false><<<batch, 256, 0, (cudaStream_t)stream>>>((const float4*)x, (const float4*)xhat, per_image / 4,
                                                                 nullptr, log_pxz, nullptr, n_ln2);
  GCC_CHECK_LAUNCH("recon");
  return GCCVAE_OK;
}

extern "C" int gccvae_adam_f32(float* param, const float* grad, float* m, float* v, long long n, float lr, float beta1,
                               float beta2, float eps, int step, int* step_dev, void* stream) {
  GCC_REQUIRE(param && grad && m && v && n > 0 && (step >= 1 || step_dev), "adam: bad args");
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (step_dev) {
    GCC_CUDA(launch_aux(bump_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, step_dev));
    GCC_CHECK_LAUNCH("adam_bump");
  }
  GCC_CUDA(launch_aux(adam_kernel, dim3((int)blocks), dim3(256), 0, (cudaStream_t)stream, param, grad, m, v, n, lr,
                      beta1, beta2, eps, step, (const int*)step_dev));
  GCC_CHECK_LAUNCH("adam");
  return GCCVAE_OK;
}

extern "C" int gccvae_adam_fused_f32(float* param, float* grad, float* m, float* v, long long i0, long long n,
                                     long long n_zero, float lr, float beta1, float beta2, float eps, int* step_state,
                                     int publish, const float* result_loss, const float* result_c, float* result_ring,
                                     int ring_slots, void* stream) {
  GCC_REQUIRE(param && grad && m && v && i0 >= 0 && n > i0 && n_zero >= n && step_state, "adam_fused: bad args");
  GCC_REQUIRE(result_ring == nullptr || (result_loss && result_c && ring_slots > 0), "adam_fused: bad result ring");
  long long blocks = (n_zero - i0 + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  GCC_CUDA(launch_aux(adam_fused_kernel, dim3((int)blocks), dim3(256), 0, (cudaStream_t)stream, param, grad, m, v, i0,
                      n, n_zero, lr, beta1, beta2, eps, step_state, publish, result_loss, result_c, result_ring,
                      ring_slots));
  GCC_CHECK_LAUNCH("adam_fused");
  return GCCVAE_OK;
}

extern "C" int gccvae_debug_mark(long long* buf, int idx, void* stream) {
  GCC_REQUIRE(buf && idx >= 0, "debug_mark: bad args");
  mark_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(buf, idx);
  GCC_CHECK_LAUNCH("debug_mark");
  return GCCVAE_OK;
}

extern "C" size_t gccvae_colsum_f32_workspace_bytes(long long rows, int cols) {
  return (size_t)colsum_splits(rows, cols) * cols * sizeof(float);
}

extern "C" int gccvae_colsum_f32(const float* in, long long rows, int cols, float* out, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  GCC_REQUIRE(in && out && rows > 0 && cols > 0 && workspace, "colsum: bad args");
  const int splits = colsum_splits(rows, cols);
  if (workspace_bytes < (size_t)splits * cols * sizeof(float)) {
    set_error("colsum: workspace %zu < %zu bytes", workspace_bytes, (size_t)splits * cols * sizeof(float));
    return GCCVAE_ENOMEM;
  }
  const int rps = (int)((rows + splits - 1) / splits);
  dim3 grid((cols + 31) / 32, splits);
  colsum_stage1<<<grid, 256, 0, (cudaStream_t)stream>>>(in, rows, cols, rps, (float*)workspace);
  GCC_CHECK_LAUNCH("colsum_stage1");
  colsum_stage2<<<(cols + 127) / 128, 128, 0, (cudaStream_t)stream>>>((const float*)workspace, splits, cols, out);
  GCC_CHECK_LAUNCH("colsum_stage2");
  return GCCVAE_OK;
}
