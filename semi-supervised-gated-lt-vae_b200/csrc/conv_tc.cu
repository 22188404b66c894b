// bf16 tensor-core path of the encoder / decoder convolutions (networks.py:11-15,45-49):
// implicit GEMM on tcgen05 (accumulators in TMEM), operands staged in shared memory by TMA.
//
// "tap-GEMM" (this file): for a tile of 128 output pixels,
//     D[128, N] = sum_{tap t} sum_{chunk c}  A_t[128, KC] * B_t[N, KC]^T
// where A_t is ONE 4-D TMA box of the NHWC activation tensor, shifted by the tap's (dh, dw) and (for
// stride-2 convolutions) traversed with elementStrides (1,2,2,1); out-of-image coordinates are
// zero-filled by TMA, which implements the padding.  B_t is a 2-D TMA box of the pre-packed bf16
// weight matrix.  Both land in the canonical K-major swizzled layout the UMMA descriptors expect
// (swizzle width = KC*2 bytes).  The same kernel runs
//   * L->S  (Conv2D forward / Conv2DTranspose dgrad): 16 taps, stride-2 box,
//   * S->L  (Conv2DTranspose forward / Conv2D dgrad): 4 output-parity phases x 4 taps,
//   * dense (conv5 as [B,2048]x[2048,256], ...): 1 tap, many chunks.
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2-5 = epilogue
// (TMEM -> registers -> bias/activation/mask -> bf16 -> global).  Persistent: one CTA per SM walks a
// contiguous range of (tile, N-slab, phase) work items; the accumulator is double-buffered in TMEM so
// the epilogue of item i overlaps the TMA/MMA main loop of item i+1.
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <type_traits>

#include "common.cuh"
#include "tc_common.cuh"

namespace gccvae {
using namespace tc;

// Space-to-depth ("s2d") storage of an H x W x C plane: (H/2+1) x (W/2+1) blocks of 2x2 pixels, block (i, j) holding
// pixels (2i-1+dy, 2j-1+dx) in slot dy*2+dx (zero slots outside the plane).  s2d_slot() = index of pixel (y, x) of
// image n in units of C channels.  A stride-2 k4/p1 gather over the plane is then a 2x2-tap stride-1 gather over the
// blocks with 4C channels per tap: TMA rows of 4C*2 bytes instead of 16 taps of C*2 bytes with element stride 2.
__device__ __forceinline__ size_t s2d_slot(int n, int y, int x, int H, int W) {
  const int HB = (H >> 1) + 1, WB = (W >> 1) + 1;
  return (((size_t)n * HB + ((y + 1) >> 1)) * WB + ((x + 1) >> 1)) * 4 + (((y + 1) & 1) * 2 + ((x + 1) & 1));
}

struct alignas(64) TapGemmParams {
  CUtensorMap tmA, tmB;
  int num_taps, chunks, KC, swz;
  int a_scale;
  int BW, BH, BN;
  int tiles_w, tiles_h;
  int N, n_store;
  int b_tap_stride;
  short a_dw[4][16], a_dh[4][16];
  int b_row0[4];
  void* out;
  const void* mask;
  const float* bias;
  int bias_mod;  // bias index = channel % bias_mod (dense S->L: channel = (kh,kw,cl))
  int act;
  int out_f32;
  int OH, OW, OC, oys, oxs;
  int oy0[4], ox0[4];
  int batch;
  int stages;
  int tps;      // k-blocks (tap, chunk) per pipeline stage: one barrier round trip feeds tps * KC/16 MMAs
  int n_slabs;  // slabs of N output channels (B rows / output channels offset by slab*N)
  int phases;
  int total_items;  // tiles * n_slabs * phases, spread contiguously over the persistent CTAs
  int bias_n;       // number of valid bias entries (channels >= bias_n get no bias)
  long long* timeline;  // debug: block 0 records clock64() at pipeline events [item][8] (NULL = off)
  int out_s2d, mask_s2d;   // the output / the mask tensor is stored in s2d block form (bf16 only)
  int rows_valid;          // rows of the 128-row tile that carry work (TMA box rows); the rest is never stored
  int pad_;                // keeps halo2 / a_box_rows 8-byte aligned: the kernel reads the pair with one 64-bit load
  // "halo2" (4-tap L -> S over s2d blocks, full-width tiles of one image): instead of four shifted boxes of BH x BW block
  // rows, TWO column-shifted boxes (b = 0, 1) of (BH + 1) x BW rows are loaded per chunk and the row tap a = 0, 1 is a
  // start-address offset of BW rows (a multiple of the 1 KB swizzle atom) in the A descriptor: (BH + 1) / (2 BH) of the
  // L2 -> shared-memory traffic the four-box form needs.  A k-block then carries the B tiles of both row taps.
  int halo2;
  int a_box_rows;     // rows of one A box (128, or (BH + 1) * BW in halo2 mode)
};

// Pipeline timeline (scripts/timeline_probe.py).  Compiled in only with -DGCCVAE_TIMELINE (libgccvae_tl.so): even with
// a NULL buffer the hooks cost a constant-bank load, a special-register read and a predicate chain per event, which
// the ncu source view showed as ~25 % of the stall samples of the (epilogue-bound) c3conv epilogue.
#ifdef GCCVAE_TIMELINE
#define TL_ON(p) ((p).timeline != nullptr)
#define TL(item_local, slot)                                                              \
  do {                                                                                    \
    if (p.timeline != nullptr && blockIdx.x == 0 && (item_local) < 32)                    \
      p.timeline[(item_local) * 8 + (slot)] = clock64();                                  \
  } while (0)
#else
#define TL_ON(p) false
#define TL(item_local, slot) \
  do {                       \
  } while (0)
#endif

constexpr int TG_THREADS = 192;

__global__ void __launch_bounds__(TG_THREADS) tapgemm_kernel(const __grid_constant__ TapGemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const int a_bytes = p.a_box_rows * p.KC * 2, b_tile = p.N * p.KC * 2, b_bytes = (p.halo2 ? 2 : 1) * b_tile;
  const int a_stride = (a_bytes + 1023) & ~1023, b_stride = (b_bytes + 1023) & ~1023;
  const int stage_stride = p.tps * (a_stride + b_stride);   // [tps A blocks][tps B blocks]
  uint8_t* sA = smem;
  uint8_t* sB = smem + p.tps * a_stride;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.stages * stage_stride);
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;   // [2] accumulator stage ready for the epilogue
  uint64_t* tempty = tfull + 2;         // [2] accumulator stage drained by the epilogue
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* s_bias = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 15) & ~(uintptr_t)15);   // [256] bias (zero beyond bias_n)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  // persistent: this CTA owns a contiguous range of work items; item = (tile, slab, phase), phase fastest,
  // so the 4 output-parity phases that re-read one input tile run back to back on the same SM.
  const int per_cta = (p.total_items + (int)gridDim.x - 1) / (int)gridDim.x;
  const int item_beg = blockIdx.x * per_cta;
  const int item_end = min(item_beg + per_cta, p.total_items);
  const int tiles_per_group = p.tiles_w * p.tiles_h;
  uint32_t acc_cols = 32;
  while ((int)acc_cols < p.N) acc_cols <<= 1;
  const uint32_t tmem_cols = acc_cols * 2;   // two accumulator stages

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above overlapped the predecessor's tail; its outputs are needed from here on
  if (TL_ON(p) && threadIdx.x == 0 && blockIdx.x < 1024) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    p.timeline[40 * 8 + 2 * blockIdx.x] = (long long)gt;
  }

  const int k_iters = p.num_taps * p.chunks;
  if (warp == 0) {
    // ===== TMA producer: one stage = tps consecutive k-blocks (tap, chunk) =====
    if (elect_one()) {
      int stage = 0;
      uint32_t ph = 0;
      long long prod_wait = 0;
      const long long tp0 = clock64();
      const uint32_t stage_tx =
          (uint32_t)(p.tps * ((p.halo2 ? p.a_box_rows : p.rows_valid) * p.KC * 2 + b_bytes));
      for (int item = item_beg; item < item_end; ++item) {
        const int phase_id = item % p.phases, slab = (item / p.phases) % p.n_slabs, tile = item / (p.phases * p.n_slabs);
        const int grp = tile / tiles_per_group, tin = tile % tiles_per_group;
        const int w0 = (tin % p.tiles_w) * p.BW, h0 = (tin / p.tiles_w) * p.BH, n0 = grp * p.BN;
        const int aw = p.a_scale * w0, ah = p.a_scale * h0, brow = p.b_row0[phase_id] + slab * p.N;
        int t = 0, c = 0;
        for (int it = 0; it < k_iters; it += p.tps) {
          const long long tw0 = TL_ON(p) ? clock64() : 0;
          mbar_wait(&empty[stage], ph ^ 1);
          if (TL_ON(p)) prod_wait += clock64() - tw0;
          if (it == 0) TL(item - item_beg, 0);
          mbar_expect_tx(&full[stage], stage_tx);
          uint8_t* a_dst = sA + stage * stage_stride;
          uint8_t* b_dst = sB + stage * stage_stride;
          for (int j = 0; j < p.tps; ++j) {
            tma_load_4d(a_dst, &p.tmA, &full[stage], c * p.KC, aw + p.a_dw[phase_id][t], ah + p.a_dh[phase_id][t], n0);
            if (p.halo2) {   // t = column tap b; the B tiles of row taps a = 0, 1 (tap index a * 2 + b)
              tma_load_2d(b_dst, &p.tmB, &full[stage], t * p.b_tap_stride + c * p.KC, brow);
              tma_load_2d(b_dst + b_tile, &p.tmB, &full[stage], (2 + t) * p.b_tap_stride + c * p.KC, brow);
            } else {
              tma_load_2d(b_dst, &p.tmB, &full[stage], t * p.b_tap_stride + c * p.KC, brow);
            }
            a_dst += a_stride;
            b_dst += b_stride;
            if (++c == p.chunks) { c = 0; ++t; }
          }
          if (it + p.tps >= k_iters) TL(item - item_beg, 1);
          if (++stage == p.stages) { stage = 0; ph ^= 1; }
        }
      }
      if (TL_ON(p) && blockIdx.x == 0) {
        p.timeline[32 * 8 + 0] = prod_wait;
        p.timeline[32 * 8 + 1] = clock64() - tp0;
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: ONE thread runs the whole loop.  Descriptors are built once; per MMA only the 14-bit
    // start-address field advances (a 64-bit add), so the issue cost is a handful of instructions =====
    if (lane == 0) {
      const uint32_t idesc = instr_desc_bf16(128, p.N, 0, 0);
      const uint32_t sbo = 8u * (uint32_t)p.KC * 2u;  // 8 rows of the swizzle atom
      const uint64_t dproto = smem_desc(0, 16, sbo, (uint32_t)p.swz);
      const uint64_t adesc0 = dproto + (uint64_t)(smem_u32(sA) >> 4), bdesc0 = dproto + (uint64_t)(smem_u32(sB) >> 4);
      const uint32_t a_step = (uint32_t)a_stride >> 4, b_step = (uint32_t)b_stride >> 4;
      const uint32_t st_step = (uint32_t)stage_stride >> 4;
      const int kk_n = p.KC / 16;
      int stage = 0;
      uint32_t ph = 0;
      long long mma_wait = 0, acc_wait = 0;
      const long long tm0 = clock64();
      // the whole issue loop is instantiated per KC / 16 (1, 2 or 4 MMAs per k-block): with a run-time trip count every
      // UTCHMMA drags ~100 cycles of uniform-register moves and convergence code along (scripts/microbench/mma_rate.cu)
      auto run = [&](auto kk_c) {
      constexpr int KK = decltype(kk_c)::value;
      for (int item = item_beg; item < item_end; ++item) {
        const int li = item - item_beg, as = li & 1;
        const long long ta0 = TL_ON(p) ? clock64() : 0;
        mbar_wait(&tempty[as], ((uint32_t)(li >> 1) & 1u) ^ 1u);
        if (TL_ON(p)) acc_wait += clock64() - ta0;
        tc_fence_after();
        TL(li, 2);
        const uint32_t tacc = tmem_base + (uint32_t)as * acc_cols;
        for (int it = 0; it < k_iters; it += p.tps) {
          const long long tw0 = TL_ON(p) ? clock64() : 0;
          mbar_wait(&full[stage], ph);
          if (TL_ON(p)) mma_wait += clock64() - tw0;
          tc_fence_after();
          if (it + p.tps >= k_iters) TL(li, 3);
          uint64_t ad = adesc0 + (uint64_t)((uint32_t)stage * st_step);
          uint64_t bd = bdesc0 + (uint64_t)((uint32_t)stage * st_step);
          if (p.halo2) {
            // per k-block (column tap, chunk): row tap a = 0, 1 -> A shifted by BW rows, B tile a
            const uint32_t a_shift = (uint32_t)(p.BW * p.KC * 2) >> 4, b_shift = (uint32_t)b_tile >> 4;
            for (int j = 0; j < p.tps; ++j) {
              for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int kk = 0; kk < KK; ++kk)
                  umma_bf16(tacc, ad + (uint64_t)(a * a_shift + 2u * kk), bd + (uint64_t)(a * b_shift + 2u * kk), idesc,
                            (it > 0 || j > 0 || a > 0 || kk > 0) ? 1u : 0u);
              ad += a_step;
              bd += b_step;
            }
          } else {
          umma_bf16(tacc, ad, bd, idesc, it > 0 ? 1u : 0u);
#pragma unroll
          for (int kk = 1; kk < KK; ++kk) umma_bf16(tacc, ad + 2u * kk, bd + 2u * kk, idesc, 1u);
          for (int j = 1; j < p.tps; ++j) {
            ad += a_step;
            bd += b_step;
#pragma unroll
            for (int kk = 0; kk < KK; ++kk) umma_bf16(tacc, ad + 2u * kk, bd + 2u * kk, idesc, 1u);
          }
          }
          umma_commit(&empty[stage]);
          if (it + p.tps >= k_iters) umma_commit(&tfull[as]);
          if (++stage == p.stages) { stage = 0; ph ^= 1; }
        }
      }
      };
      if (kk_n == 4) run(std::integral_constant<int, 4>{});
      else if (kk_n == 2) run(std::integral_constant<int, 2>{});
      else run(std::integral_constant<int, 1>{});
      if (TL_ON(p) && blockIdx.x == 0) {
        p.timeline[32 * 8 + 2] = mma_wait;
        p.timeline[32 * 8 + 3] = acc_wait;
        p.timeline[32 * 8 + 4] = clock64() - tm0;
        p.timeline[32 * 8 + 5] = (long long)(item_end - item_beg) * (k_iters / p.tps);
        p.timeline[32 * 8 + 6] = p.stages;
        p.timeline[32 * 8 + 7] = gridDim.x;
      }
    }
  } else {
    // ===== epilogue: warps 2..5 own TMEM lanes 32*(warp%4) .. +31 =====
    const int q = warp & 3;
    const int m = q * 32 + lane;
    const int dx = m % p.BW, dy = (m / p.BW) % p.BH, dn = m / (p.BW * p.BH);
    // bias -> shared memory once per CTA (a global load per item would sit on the epilogue's critical path)
    {
      const int nb = p.bias == nullptr ? 0 : (p.bias_mod < p.bias_n ? p.bias_mod : p.bias_n);
      for (int i = threadIdx.x - 64; i < 256; i += 128) s_bias[i] = i < nb ? p.bias[i] : 0.0f;
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    for (int item = item_beg; item < item_end; ++item) {
      const int li = item - item_beg, as = li & 1;
      const int phase_id = item % p.phases, slab = (item / p.phases) % p.n_slabs, tile = item / (p.phases * p.n_slabs);
      const int grp = tile / tiles_per_group, tin = tile % tiles_per_group;
      const int w0 = (tin % p.tiles_w) * p.BW, h0 = (tin / p.tiles_w) * p.BH, n0 = grp * p.BN;
      const int slab0 = slab * p.N;
      const int n = n0 + dn, y = h0 + dy, x = w0 + dx;
      const bool valid = n < p.batch && m < p.rows_valid;
      const int oyy = y * p.oys + p.oy0[phase_id], oxx = x * p.oxs + p.ox0[phase_id];
      const size_t opix_lin = ((size_t)n * p.OH + (size_t)oyy) * p.OW + oxx;
      const size_t opix_s2d = (p.out_s2d | p.mask_s2d) ? s2d_slot(n, oyy, oxx, p.OH, p.OW) : 0;
      const size_t opix = p.out_s2d ? opix_s2d : opix_lin;
      const size_t mpix = p.mask_s2d ? opix_s2d : opix_lin;
      const uint32_t tacc = tmem_base + (uint32_t)as * acc_cols + ((uint32_t)(q * 32) << 16);
      // the mask (ReLU derivative of the consumer) does not depend on the accumulator: fetch the first
      // 64 channels of it BEFORE waiting for the MMAs so its latency hides behind the main loop
      uint32_t mpre[4][8];
      const bool use_mask = p.mask != nullptr && valid;
      if (use_mask) {
        const __nv_bfloat16* mk = reinterpret_cast<const __nv_bfloat16*>(p.mask) + mpix * p.OC + slab0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (i * 16 < p.N && slab0 + i * 16 < p.n_store) ld_global_nc_256(mk + i * 16, mpre[i]);
      }
      mbar_wait(&tfull[as], (uint32_t)(li >> 1) & 1u);
      tc_fence_after();
      if (threadIdx.x == 64) TL(li, 4);
      // bias index of this slab's first channel: host guarantees bias_mod % N == 0 or bias_mod >= n_store,
      // so no per-element modulo is needed
      const int bias_base = slab0 % p.bias_mod;
      const uint32_t s_bias_u32 = smem_u32(s_bias);
      for (int c0 = 0; c0 < p.N; c0 += 16) {
        const int cg = slab0 + c0;  // global output channel of this chunk
        // bias_base + c0 + i < 256 always: bias_mod <= 256 wraps it, otherwise n_store <= 256
        const uint32_t bsrc = s_bias_u32 + (uint32_t)(((bias_base + c0) & 255) * 4);
        uint32_t r[16];
        tmem_ld16(tacc + (uint32_t)c0, r);
        tmem_ld_wait();
        if (c0 + 16 >= p.N) {  // accumulator fully read: hand the TMEM stage back to the MMA warp
          tc_fence_before();
          if (lane == 0) mbar_arrive(&tempty[as]);
          if (threadIdx.x == 64) TL(li, 5);
        }
        if (!valid || cg >= p.n_store) continue;
        float v[16];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 t = lds_f4(bsrc + 16u * i);
          v[4 * i] = __uint_as_float(r[4 * i]) + t.x;
          v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + t.y;
          v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + t.z;
          v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + t.w;
        }
        if (p.act == GCCVAE_ACT_RELU) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.0f);
        } else if (p.act == GCCVAE_ACT_SIGMOID) {
          if (p.out_f32 == 2) {   // 3-channel image: only the real channels
#pragma unroll
            for (int i = 0; i < 3; ++i) v[i] = __fdividef(1.0f, 1.0f + __expf(-v[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __fdividef(1.0f, 1.0f + __expf(-v[i]));
          }
        }
        const size_t o = opix * p.OC + cg;
        if (use_mask) {
          uint32_t mw[8];
          if (c0 < 64) {
            // static indexing keeps mpre[] in registers
            switch (c0 >> 4) {
              case 0:
#pragma unroll
                for (int i = 0; i < 8; ++i) mw[i] = mpre[0][i];
                break;
              case 1:
#pragma unroll
                for (int i = 0; i < 8; ++i) mw[i] = mpre[1][i];
                break;
              case 2:
#pragma unroll
                for (int i = 0; i < 8; ++i) mw[i] = mpre[2][i];
                break;
              default:
#pragma unroll
                for (int i = 0; i < 8; ++i) mw[i] = mpre[3][i];
                break;
            }
          } else {
            ld_global_nc_256(reinterpret_cast<const __nv_bfloat16*>(p.mask) + mpix * p.OC + cg, mw);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            // bf16 > 0  <=>  sign bit clear and magnitude non-zero
            const uint32_t lo = mw[i] & 0xffffu, hi = mw[i] >> 16;
            if (!(lo != 0 && lo < 0x8000u)) v[2 * i] = 0.0f;
            if (!(hi != 0 && hi < 0x8000u)) v[2 * i + 1] = 0.0f;
          }
        }
        if (p.out_f32 == 2) {
          // 3-channel image padded to 4 (decoder output): one float4 per pixel, pad channel = 0
          if (c0 == 0) reinterpret_cast<float4*>(p.out)[opix] = make_float4(v[0], v[1], v[2], 0.0f);
        } else if (p.out_f32) {
          float* dst = reinterpret_cast<float*>(p.out) + o;
          uint32_t w0[8], w1[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) { w0[i] = __float_as_uint(v[i]); w1[i] = __float_as_uint(v[8 + i]); }
          st_global_256(dst, w0);
          st_global_256(dst + 8, w1);
        } else {
          uint32_t w[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) w[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
          st_global_256(reinterpret_cast<__nv_bfloat16*>(p.out) + o, w);   // one full 32-byte sector per lane
        }
      }
      if (threadIdx.x == 64) TL(li, 6);
    }
    tc_fence_before();
  }
  __syncthreads();
  if (TL_ON(p) && threadIdx.x == 0 && blockIdx.x < 1024) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    p.timeline[40 * 8 + 2 * blockIdx.x + 1] = (long long)gt;
  }
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------------
// S -> L "halo" kernel (Conv2DTranspose forward / Conv2D dgrad for 16x16 and 32x32 S planes).
// The generic tap-GEMM above reads every input tile 16 times from L2 (4 output-parity phases x 4 taps)
// and is L2-bandwidth bound.  Here one CTA computes ALL FOUR phases of a tile of BH full-width rows:
//   * the input rows h0-1 .. h0+BH (one halo row above and below) are loaded ONCE per column shift
//     dw in {-1,0,+1} (3 TMA boxes, zero-filled outside the image);
//   * the row shift dh in {-1,0,+1} of a tap is a descriptor start-address offset of BW rows (a multiple
//     of the swizzle pattern), so the 16 (phase, tap) MMAs all read those three buffers;
//   * the 16 weight blocks [N x C] stay resident in shared memory for the whole (persistent) kernel;
//   * 4 phases x 2 stages of fp32 accumulators live in TMEM; 8 epilogue warps drain them.
// L2->SM traffic per tile: 3*(BH+2)/BH tile-equivalents instead of 16.
// ---------------------------------------------------------------------------------------------------
struct alignas(64) SlHaloParams {
  CUtensorMap tmA, tmB;
  int C, BW, BH, tiles_h;
  int N, n_store, swz;
  void* out;
  const void* mask;
  const float* bias;
  int bias_n, act, out_f32;
  int OH, OW, OC, batch, total_tiles, stages;
  long long* timeline;  // debug: block 0 records clock64() at pipeline events [tile][8] (NULL = off)
  int mask_s2d;         // the mask tensor is stored in s2d block form
};
constexpr int HALO_THREADS = 320;

__global__ void __launch_bounds__(HALO_THREADS) sl_halo_kernel(const __grid_constant__ SlHaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const int rowb = p.C * 2;                       // bytes per pixel row (64 or 128)
  const int avb = (p.BH + 2) * p.BW * rowb;       // one column-shift variant
  const int a_stage = 3 * avb;
  const int bblk = 4 * p.N * rowb;                // one view's weight block: [4 phases x N rows][C]
  uint8_t* sB = smem;
  uint8_t* sA = smem + ((9 * bblk + 1023) & ~1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(sA + p.stages * a_stage);
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;
  uint64_t* tempty = tfull + 2;
  uint64_t* bfull = tempty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);
  float* s_bias = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 15) & ~(uintptr_t)15);   // [256], 16-byte aligned (ld.shared.v4)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  const int per_cta = (p.total_tiles + (int)gridDim.x - 1) / (int)gridDim.x;
  const int tile_beg = blockIdx.x * per_cta;
  const int tile_end = min(tile_beg + per_cta, p.total_tiles);
  uint32_t tmem_cols = 32;                        // 2 stages x 4 phases x N columns, power of two
  while ((int)tmem_cols < 8 * p.N) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 8);
    }
    mbar_init(bfull, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, tmem_cols);
  for (int i = threadIdx.x; i < 256; i += HALO_THREADS)
    s_bias[i] = (p.bias != nullptr && i < p.bias_n) ? p.bias[i] : 0.0f;   // parameters: not written by the predecessor
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  if (warp == 0) {
    // ===== TMA producer =====
    if (elect_one() && tile_beg < tile_end) {
      mbar_expect_tx(bfull, (uint32_t)(9 * bblk));
      for (int view = 0; view < 9; ++view)   // packed weights "sl9": [view][phase][N rows][C]
        tma_load_2d(sB + view * bblk, &p.tmB, bfull, 0, view * 4 * p.N);
      int stage = 0;
      uint32_t ph = 0;
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        const int n = tile / p.tiles_h, h0 = (tile % p.tiles_h) * p.BH;
        mbar_wait(&empty[stage], ph ^ 1);
        TL(tile - tile_beg, 0);
        mbar_expect_tx(&full[stage], (uint32_t)a_stage);
        for (int v = 0; v < 3; ++v)
          tma_load_4d(sA + stage * a_stage + v * avb, &p.tmA, &full[stage], 0, v - 1, h0 - 1, n);
        TL(tile - tile_beg, 1);
        if (++stage == p.stages) { stage = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    // One MMA covers all four output-parity phases: N = 4*N_phase, the B block of a view holds each phase's
    // weights for the tap that reads this view (zeros where a phase does not use it).  9 views x C/16 MMAs
    // instead of 16 (phase,tap) x C/16.  Descriptors are built once; per MMA only the address field advances.
    if (lane == 0 && tile_beg < tile_end) {
      const uint32_t idesc = instr_desc_bf16(128, 4 * p.N, 0, 0);
      const uint32_t sbo = 8u * (uint32_t)rowb;
      const uint64_t dproto = smem_desc(0, 16, sbo, (uint32_t)p.swz);
      const uint64_t bdesc0 = dproto + (uint64_t)(smem_u32(sB) >> 4);
      const uint64_t adesc0 = dproto + (uint64_t)(smem_u32(sA) >> 4);
      const uint32_t a_stage16 = (uint32_t)a_stage >> 4, avb16 = (uint32_t)avb >> 4, row16 = (uint32_t)(p.BW * rowb) >> 4;
      const uint32_t bblk16 = (uint32_t)bblk >> 4;
      const int kk_n = p.C / 16;
      int stage = 0;
      uint32_t ph = 0;
      mbar_wait(bfull, 0);
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        const int li = tile - tile_beg, as = li & 1;
        mbar_wait(&tempty[as], ((uint32_t)(li >> 1) & 1u) ^ 1u);
        TL(li, 2);
        mbar_wait(&full[stage], ph);
        tc_fence_after();
        TL(li, 3);
        const uint64_t a_st = adesc0 + (uint64_t)((uint32_t)stage * a_stage16);
        const uint32_t tacc = tmem_base + (uint32_t)as * 4u * (uint32_t)p.N;
        // fully unrolled for both channel counts: from a loop with a run-time trip count every UTCHMMA drags ~100 cycles of
        // uniform-register moves and convergence code along (scripts/microbench/mma_rate.cu)
        if (kk_n == 2) {
#pragma unroll
          for (int view = 0; view < 9; ++view) {
            const uint64_t ad = a_st + (uint64_t)((uint32_t)(view % 3) * avb16 + (uint32_t)(view / 3) * row16);
            const uint64_t bd = bdesc0 + (uint64_t)((uint32_t)view * bblk16);
#pragma unroll
            for (int kk = 0; kk < 2; ++kk)
              umma_bf16(tacc, ad + 2u * kk, bd + 2u * kk, idesc, (view > 0 || kk > 0) ? 1u : 0u);
          }
        } else {
#pragma unroll
          for (int view = 0; view < 9; ++view) {
            const uint64_t ad = a_st + (uint64_t)((uint32_t)(view % 3) * avb16 + (uint32_t)(view / 3) * row16);
            const uint64_t bd = bdesc0 + (uint64_t)((uint32_t)view * bblk16);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16(tacc, ad + 2u * kk, bd + 2u * kk, idesc, (view > 0 || kk > 0) ? 1u : 0u);
          }
        }
        umma_commit(&empty[stage]);
        umma_commit(&tfull[as]);
        TL(li, 7);
        if (++stage == p.stages) { stage = 0; ph ^= 1; }
      }
    }
  } else {
    // ===== epilogue: 8 warps; warp pair (q, q+4) shares TMEM lane quadrant q, each takes 2 phases =====
    const int ew = warp - 2, q = warp & 3, half = ew >> 2;
    const uint32_t s_bias_u32 = smem_u32(s_bias);
    const int m = q * 32 + lane;
    const int dy = m / p.BW, dx = m % p.BW;
    for (int tile = tile_beg; tile < tile_end; ++tile) {
      const int li = tile - tile_beg, as = li & 1;
      const int n = tile / p.tiles_h, h0 = (tile % p.tiles_h) * p.BH;
      const int y = h0 + dy;
      size_t opix[2], mpix[2];
      uint32_t mpre[2][2][8];
      const bool use_mask = p.mask != nullptr;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int phase = half * 2 + j;
        opix[j] = ((size_t)n * p.OH + (size_t)(2 * y + (phase >> 1))) * p.OW + (2 * dx + (phase & 1));
        mpix[j] = p.mask_s2d ? s2d_slot(n, 2 * y + (phase >> 1), 2 * dx + (phase & 1), p.OH, p.OW) : opix[j];
        if (use_mask) {   // first 32 channels of the ReLU mask, fetched before the accumulator is ready
          const __nv_bfloat16* mk = reinterpret_cast<const __nv_bfloat16*>(p.mask) + mpix[j] * p.OC;
#pragma unroll
          for (int i = 0; i < 2; ++i)
            if (i * 16 < p.n_store) ld_global_nc_256(mk + i * 16, mpre[j][i]);
        }
      }
      mbar_wait(&tfull[as], (uint32_t)(li >> 1) & 1u);
      tc_fence_after();
      if (threadIdx.x == 64) TL(li, 4);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int phase = half * 2 + j;
        const uint32_t tacc = tmem_base + (uint32_t)(as * 4 + phase) * (uint32_t)p.N + ((uint32_t)(q * 32) << 16);
        for (int c0 = 0; c0 < p.N; c0 += 16) {
          uint32_t r[16];
          tmem_ld16(tacc + (uint32_t)c0, r);
          tmem_ld_wait();
          if (j == 1 && c0 + 16 >= p.N) {  // this warp has read both of its accumulators
            tc_fence_before();
            if (lane == 0) mbar_arrive(&tempty[as]);
            if (threadIdx.x == 64) TL(li, 5);
          }
          if (c0 >= p.n_store) continue;
          float v[16];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 t = lds_f4(s_bias_u32 + (uint32_t)(c0 + 4 * i) * 4u);
            v[4 * i] = __uint_as_float(r[4 * i]) + t.x;
            v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + t.y;
            v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + t.z;
            v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + t.w;
          }
          if (p.act == GCCVAE_ACT_RELU) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.0f);
          } else if (p.act == GCCVAE_ACT_SIGMOID) {
            if (p.out_f32 == 2) {
#pragma unroll
              for (int i = 0; i < 3; ++i) v[i] = __fdividef(1.0f, 1.0f + __expf(-v[i]));
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = __fdividef(1.0f, 1.0f + __expf(-v[i]));
            }
          }
          const size_t o = opix[j] * p.OC + c0;
          if (use_mask) {
            uint32_t mw[8];
            if (c0 == 0) {
#pragma unroll
              for (int i = 0; i < 8; ++i) mw[i] = mpre[j][0][i];
            } else if (c0 == 16) {
#pragma unroll
              for (int i = 0; i < 8; ++i) mw[i] = mpre[j][1][i];
            } else {
              ld_global_nc_256(reinterpret_cast<const __nv_bfloat16*>(p.mask) + mpix[j] * p.OC + c0, mw);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint32_t lo = mw[i] & 0xffffu, hi = mw[i] >> 16;
              if (!(lo != 0 && lo < 0x8000u)) v[2 * i] = 0.0f;
              if (!(hi != 0 && hi < 0x8000u)) v[2 * i + 1] = 0.0f;
            }
          }
          if (p.out_f32 == 2) {
            if (c0 == 0) reinterpret_cast<float4*>(p.out)[opix[j]] = make_float4(v[0], v[1], v[2], 0.0f);
          } else if (p.out_f32) {
            float* dst = reinterpret_cast<float*>(p.out) + o;
            uint32_t w0[8], w1[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { w0[i] = __float_as_uint(v[i]); w1[i] = __float_as_uint(v[8 + i]); }
            st_global_256(dst, w0);
            st_global_256(dst + 8, w1);
          } else {
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
            st_global_256(reinterpret_cast<__nv_bfloat16*>(p.out) + o, w);
          }
        }
      }
      if (threadIdx.x == 64) TL(li, 6);
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------------
// weight-gradient kernel: dW[(tap,cl), cs] += sum_pix gather(L)[pix,(tap,cl)] * S[pix, cs]
// The reduction axis of this GEMM is the PIXEL axis, so both operands are MN-major: a TMA box
// [128 pixels x channels] is, as it lands, the canonical MN-major swizzled layout (channels
// contiguous, 8-pixel groups at SBO, further 64/32-channel blocks - here: further taps - at LBO).
// One CTA owns one 128-row slice of dW (128/CL taps) and a range of pixel tiles (split-K);
// the fp32 TMEM accumulator is added to dW with red.global at the end.
// ---------------------------------------------------------------------------------------------------
struct alignas(64) WgParams {
  CUtensorMap tmA, tmB;
  int blocks_per_mtile, blocks_per_tap, taps, kcA, b_loads, kcB, swzA, swzB;
  int c4_rows;  // 0: dW rows as computed; 2: x2 rows, 3: s2d rows, scattered to Keras (kh, kw, c) order (see the epilogue)
  int a_scale, BW, BH, BN, tiles_w, tiles_h;
  short a_dw[16], a_dh[16];
  int N;
  int tiles_total, tiles_per_cta;
  gccvae_wg_out out;   // destination segments (columns -> tensors); out.m_valid rows are stored
  int stages;
  // x2 mode: the A operand (128 pixels x 64 (a,b,dy,dx,c4) values, 128-byte rows) is built by warps 2-5 with cp.async
  // from the [B,33,33,16] block tensor instead of 8 TMA boxes of 32-byte rows (TMA is row-rate bound)
  const uint4* in2;
  int s2d_cl;   // c4_rows == 3: channels per pixel of the s2d L operand
  float* ones_db;   // c4_rows == 2: row 15 = (tap (0,0), slot (1,1), pad channel) is all ones in prep_x2's blocks: += column sums of S
  long long* timeline;   // instrumented build only (scripts/timeline_wgrad.py)
};

__global__ void __launch_bounds__(TG_THREADS) wgrad_kernel(const __grid_constant__ WgParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const int a_slab = 128 * p.kcA * 2, b_slab = 128 * p.kcB * 2;
  const int a_bytes = p.blocks_per_mtile * a_slab, b_bytes = p.b_loads * b_slab;
  uint8_t* sA = smem;
  uint8_t* sB = smem + p.stages * a_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(sB + p.stages * b_bytes);
  uint64_t* empty = full + p.stages;
  uint64_t* tmem_full = empty + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  const int mtile = blockIdx.y;
  const int tile_beg = blockIdx.x * p.tiles_per_cta;
  int tile_end = tile_beg + p.tiles_per_cta;
  if (tile_end > p.tiles_total) tile_end = p.tiles_total;
  const int n_tiles = tile_end - tile_beg;  // may be <= 0 for trailing CTAs
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < p.N) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], p.in2 != nullptr ? 129 : 1);   // TMA transaction (+ one cp.async arrival per A-builder thread)
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  if (n_tiles > 0) {
    const int tiles_per_group = p.tiles_w * p.tiles_h;
    if (warp == 0) {
      if (elect_one()) {
        int stage = 0;
        uint32_t ph = 0;
        // everything that does not change from tile to tile is computed once, and the tile coordinates advance
        // incrementally: the divisions by run-time values cost ~0.2 us of the ~0.35 us this thread needed per tile
        // (scripts/timeline_wgrad.py), on the round trip of a pipeline that is two stages deep
        const int n_bl = p.in2 != nullptr ? 0 : p.blocks_per_mtile;
        int bl_c[8], bl_dw[8], bl_dh[8];
        bool bl_real[8];
#pragma unroll
        for (int bl = 0; bl < 8; ++bl) {
          const int bg = mtile * p.blocks_per_mtile + bl;
          const int t = bg / p.blocks_per_tap;
          // blocks past the last tap are loaded from out-of-range images: TMA zero-fills them
          bl_real[bl] = t < p.taps;
          bl_c[bl] = (bg - t * p.blocks_per_tap) * p.kcA;
          bl_dw[bl] = bl_real[bl] ? p.a_dw[t] : 0;
          bl_dh[bl] = bl_real[bl] ? p.a_dh[t] : 0;
        }
        const uint32_t tx = (uint32_t)((p.in2 != nullptr ? 0 : a_bytes) + b_bytes);
        int grp = tile_beg / tiles_per_group, tin = tile_beg - grp * tiles_per_group;
        int tw = tin % p.tiles_w, th = tin / p.tiles_w;
        for (int it = 0; it < n_tiles; ++it) {
          const int w0 = tw * p.BW, h0 = th * p.BH, n0 = grp * p.BN;
          mbar_wait(&empty[stage], ph ^ 1);
          if (blockIdx.y == 0) TL(it, 0);
          mbar_expect_tx(&full[stage], tx);
#pragma unroll
          for (int bl = 0; bl < 8; ++bl)
            if (bl < n_bl)
              tma_load_4d(sA + stage * a_bytes + bl * a_slab, &p.tmA, &full[stage], bl_c[bl], p.a_scale * w0 + bl_dw[bl],
                          p.a_scale * h0 + bl_dh[bl], bl_real[bl] ? n0 : 0x3fffff00);
          for (int h = 0; h < p.b_loads; ++h)
            tma_load_4d(sB + stage * b_bytes + h * b_slab, &p.tmB, &full[stage], h * p.kcB, w0, h0, n0);
          if (blockIdx.y == 0) TL(it, 1);
          if (++stage == p.stages) { stage = 0; ph ^= 1; }
          if (++tw == p.tiles_w) {
            tw = 0;
            if (++th == p.tiles_h) { th = 0; ++grp; }
          }
        }
      }
    } else if (warp == 1) {
      if (lane == 0) {   // one thread issues; descriptors built once, only the address field advances
        const uint32_t idesc = instr_desc_bf16(128, p.N, 1, 1);
        const uint32_t rowA = (uint32_t)p.kcA * 2u, rowB = (uint32_t)p.kcB * 2u;
        const uint64_t ad0 = smem_desc(smem_u32(sA), (uint32_t)a_slab, 8 * rowA, (uint32_t)p.swzA);
        const uint64_t bd0 = smem_desc(smem_u32(sB), (uint32_t)b_slab, 8 * rowB, (uint32_t)p.swzB);
        const uint32_t a16 = (uint32_t)a_bytes >> 4, b16 = (uint32_t)b_bytes >> 4;
        int stage = 0;
        uint32_t ph = 0;
        for (int it = 0; it < n_tiles; ++it) {
          if (blockIdx.y == 0) TL(it, 2);
          mbar_wait(&full[stage], ph);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // cp.async-built A tile -> async proxy
          tc_fence_after();
          if (blockIdx.y == 0) TL(it, 3);
          const uint64_t ad = ad0 + (uint64_t)((uint32_t)stage * a16), bd = bd0 + (uint64_t)((uint32_t)stage * b16);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)   // 16 pixels per MMA
            umma_bf16(tmem_base, ad + (uint64_t)(kk * rowA), bd + (uint64_t)(kk * rowB), idesc,
                      (it > 0 || kk > 0) ? 1u : 0u);
          umma_commit(&empty[stage]);
          if (it == n_tiles - 1) umma_commit(tmem_full);
          if (blockIdx.y == 0) TL(it, 7);
          if (++stage == p.stages) { stage = 0; ph ^= 1; }
        }
      }
    } else {
      if (p.in2 != nullptr) {
        // ---- x2 mode: thread m builds row m (one pixel, 128 bytes = four 32-byte blocks) of the A tile ----
        const int m = threadIdx.x - 64;
        const int dy = m >> 5, dx = m & 31;
        const uint32_t row_off = (uint32_t)m * 128u, sw = (uint32_t)(m & 7);
        int stage = 0;
        uint32_t ph = 0;
        for (int it = 0; it < n_tiles; ++it) {
          const int tile = tile_beg + it;
          const int n = tile >> 3, h0 = (tile & 7) * 4;
          const uint4* src = p.in2 + (((size_t)n * 33 + (h0 + dy)) * 33 + dx) * 2;
          mbar_wait_relaxed(&empty[stage], ph ^ 1);
          const uint32_t dst = smem_u32(sA + stage * a_bytes) + row_off;
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const uint4* sp = src + ((t >> 1) * 33 + (t & 1)) * 2;
#pragma unroll
            for (int h = 0; h < 2; ++h)
              asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + ((((uint32_t)(2 * t + h)) ^ sw) << 4)),
                           "l"(sp + h)
                           : "memory");
          }
          asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&full[stage])) : "memory");
          if (++stage == p.stages) { stage = 0; ph ^= 1; }
        }
      }
      const int q = warp & 3;
      const int m = mtile * 128 + q * 32 + lane;
      mbar_wait(tmem_full, 0);
      tc_fence_after();
      if (blockIdx.y == 0 && threadIdx.x == 64) TL(n_tiles < 31 ? n_tiles : 31, 4);
      for (int c0 = 0; c0 < p.N; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
        tmem_ld_wait();
        // c4_rows 2: x2 rows (a, b, dy, dx, c4) -> ((2a+dy)*4 + 2b+dx, c3)
        //         3: s2d rows (a, b, dy, dx, c < CL) -> ((2a+dy)*4 + 2b+dx, c)   [CL = p.kcB_unused / out.cl]
        int mrow;
        if (p.c4_rows == 3) {
          const int CL = p.s2d_cl, t = m / (4 * CL), r = m - t * 4 * CL, sub = r / CL, c = r - sub * CL;
          mrow = ((2 * (t >> 1) + (sub >> 1)) * 4 + 2 * (t & 1) + (sub & 1)) * CL + c;
        } else {
          mrow = p.c4_rows == 2
                     ? ((2 * (m >> 5) + ((m >> 3) & 1)) * 4 + 2 * ((m >> 4) & 1) + ((m >> 2) & 1)) * 3 + (m & 3)
                     : m;
        }
        if (p.ones_db != nullptr && m == 15) {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (c0 + i < p.N) atomicAdd(p.ones_db + c0 + i, __uint_as_float(r[i]));
        }
        if (m < p.out.m_valid && !(p.c4_rows == 2 && (m & 3) == 3)) {
#pragma unroll
          for (int sg = 0; sg < 2; ++sg) {
            if (sg >= p.out.n_seg) break;
            const int col0 = p.out.seg[sg].col0, ncols = p.out.seg[sg].ncols, ld = p.out.seg[sg].ld;
            if (c0 + 16 <= col0 || c0 >= col0 + ncols) continue;
            float* drow = p.out.seg[sg].dst + (size_t)mrow * ld - col0;   // drow[c] = element of column c
            if ((ld & 3) == 0 && (col0 & 3) == 0 && c0 >= col0 && c0 + 16 <= col0 + ncols) {
#pragma unroll
              for (int i = 0; i < 16; i += 4)
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(drow + c0 + i),
                             "f"(__uint_as_float(r[i])), "f"(__uint_as_float(r[i + 1])), "f"(__uint_as_float(r[i + 2])),
                             "f"(__uint_as_float(r[i + 3]))
                             : "memory");
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (c0 + i >= col0 && c0 + i < col0 + ncols) atomicAdd(drow + c0 + i, __uint_as_float(r[i]));
            }
          }
        }
      }
      tc_fence_before();
      if (blockIdx.y == 0 && threadIdx.x == 64) TL(n_tiles < 31 ? n_tiles : 31, 6);
    }
  }
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// bias gradient from a bf16 [rows, cols] tensor: out[c] += sum_r in[r,c]  (fp32 atomics; out pre-zeroed)
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const __nv_bfloat16* __restrict__ in, long long rows, int cols,
                                                          int rows_per_cta, int n_valid, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  // thread handles column pair (2 bf16) ; cols even, cols/2 <= 128 -> 256 threads cover (cols/2) x (256/(cols/2)) rows
  const int cp = cols >> 1;
  const int tc = threadIdx.x % cp, tr = threadIdx.x / cp, nr = 256 / cp;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta;
  if (r1 > rows) r1 = rows;
  float a0 = 0.0f, a1 = 0.0f;
  if (tr < nr)
    for (long long r = r0 + tr; r < r1; r += nr) {
      const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(in + r * cols + 2 * tc);
      a0 += __low2float(v);
      a1 += __high2float(v);
    }
  __shared__ float red[256][2];
  red[threadIdx.x][0] = a0;
  red[threadIdx.x][1] = a1;
  __syncthreads();
  if (tr == 0) {
    for (int q = 1; q < nr; ++q) {
      a0 += red[q * cp + tc][0];
      a1 += red[q * cp + tc][1];
    }
    if (2 * tc < n_valid) atomicAdd(out + 2 * tc, a0);
    if (2 * tc + 1 < n_valid) atomicAdd(out + 2 * tc + 1, a1);
  }
}

// the same with 16-byte loads (8 columns per thread, 4 rows in flight): cols % 8 == 0, 256 % (cols / 8) == 0.  The 4-byte
// loads of the kernel above reach ~3 TB/s on the two big tensors (75.8 MB: 25 us each); this one is HBM-bound.
__global__ void __launch_bounds__(256) colsum_bf16_v8_kernel(const __nv_bfloat16* __restrict__ in, long long rows, int cols,
                                                             int rows_per_cta, int n_valid, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  const int cp = cols >> 3;
  const int tc = threadIdx.x % cp, tr = threadIdx.x / cp, nr = 256 / cp;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta;
  if (r1 > rows) r1 = rows;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.0f;
  const uint4* base = reinterpret_cast<const uint4*>(in) + tc;
  long long r = r0 + tr;
  for (; r + 3LL * nr < r1; r += 4LL * nr) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldg(base + (r + (long long)u * nr) * cp);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[2 * i] += __uint_as_float(w[i] << 16);
        acc[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
      }
    }
  }
  for (; r < r1; r += nr) {
    const uint4 v = __ldg(base + r * cp);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      acc[2 * i] += __uint_as_float(w[i] << 16);
      acc[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __shared__ float red[256][9];
#pragma unroll
  for (int i = 0; i < 8; ++i) red[threadIdx.x][i] = acc[i];
  __syncthreads();
  // thread t < cols sums column t over the nr row groups
  if ((int)threadIdx.x < cols && (int)threadIdx.x < n_valid) {
    const int c8 = threadIdx.x >> 3, ci = threadIdx.x & 7;
    float tot = 0.0f;
    for (int q = 0; q < nr; ++q) tot += red[q * cp + c8][ci];
    atomicAdd(out + threadIdx.x, tot);
  }
}

__global__ void fill_kernel(float* __restrict__ p, int n, float v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// all weight repacking of one step in ONE launch: blockIdx.y = job
struct PackJobs {
  gccvae_pack_job j[48];
};
__global__ void __launch_bounds__(256) pack_jobs_kernel(const __grid_constant__ PackJobs jobs) {
  pdl_launch_dependents();
  pdl_wait();
  const gccvae_pack_job& jb = jobs.j[blockIdx.y];
  const float* __restrict__ W = jb.W;
  __nv_bfloat16* __restrict__ out = reinterpret_cast<__nv_bfloat16*>(jb.out);
  const int CL = jb.CL, CS = jb.CS, taps = jb.taps;
  const long long stride = (long long)gridDim.x * 256;
  const long long i0 = blockIdx.x * 256LL + threadIdx.x;
  if (jb.kind == 0) {          // ls: out[cs][(tap,cl)]
    const int K = taps * CL, rows_pad = (CS + 15) / 16 * 16;
    const long long n = (long long)rows_pad * K;
    for (long long i = i0; i < n; i += stride) {
      const int cs = (int)(i / K), k = (int)(i % K);
      out[i] = __float2bfloat16(cs < CS ? W[(size_t)k * CS + cs] : 0.0f);
    }
  } else if (jb.kind == 1) {   // sl, k4/s2/p1: out[phase][cl][(th,tw,cs)]
    const int K = 4 * CS, rows_pad = (CL + 15) / 16 * 16;
    const long long n = 4LL * rows_pad * K;
    for (long long i = i0; i < n; i += stride) {
      const int k = (int)(i % K);
      const int cl = (int)((i / K) % rows_pad), phase = (int)(i / ((long long)K * rows_pad));
      const int ph = phase >> 1, pw = phase & 1, t = k / CS, cs = k % CS;
      const int kh = ((ph + 1) & 1) + 2 * (t >> 1), kw = ((pw + 1) & 1) + 2 * (t & 1);
      out[i] = __float2bfloat16(cl < CL ? W[((size_t)(kh * 4 + kw) * CL + cl) * CS + cs] : 0.0f);
    }
  } else if (jb.kind == 2) {   // plain cast
    const long long n = (long long)taps * CL * CS;
    for (long long i = i0; i < n; i += stride) out[i] = __float2bfloat16(W[i]);
  } else if (jb.kind == 6) {   // "sl9" (halo kernel): out[view][phase][cl (padded)][cs]; view = (dh+1)*3 + (dw+1)
    const int rows_pad = (CL + 15) / 16 * 16;
    const long long n = 9LL * 4 * rows_pad * CS;
    for (long long i = i0; i < n; i += stride) {
      const int cs = (int)(i % CS);
      const int cl = (int)((i / CS) % rows_pad);
      const int phase = (int)((i / ((long long)CS * rows_pad)) % 4), view = (int)(i / ((long long)CS * rows_pad * 4));
      const int dh = view / 3 - 1, dw = view % 3 - 1, ph = phase >> 1, pw = phase & 1;
      const int th = ph - dh, tw = pw - dw;   // the tap of this phase that reads input shifted by (dh, dw)
      float v = 0.0f;
      if (cl < CL && th >= 0 && th <= 1 && tw >= 0 && tw <= 1) {
        const int kh = ((ph + 1) & 1) + 2 * th, kw = ((pw + 1) & 1) + 2 * tw;
        v = W[((size_t)(kh * 4 + kw) * CL + cl) * CS + cs];
      }
      out[i] = __float2bfloat16(v);
    }
  } else if (jb.kind == 9) {
    // s2d packing of a k4/s2/p1 kernel W[kh,kw,CL,CS]: out[cs][(a,b)][(dy,dx,cl)], kh = 2a+dy, kw = 2b+dx
    // (B operand of the 4-tap L->S GEMM over s2d blocks: gccvae_tap4_ls_bf16 with CB = 4 CL)
    const int K = 16 * CL, rows_pad = (CS + 15) / 16 * 16;
    const long long n = (long long)rows_pad * K;
    for (long long i = i0; i < n; i += stride) {
      const int cs = (int)(i / K), k = (int)(i % K);
      const int t = k / (4 * CL), r = k % (4 * CL), sub = r / CL, c = r % CL;
      const int kh = 2 * (t >> 1) + (sub >> 1), kw = 2 * (t & 1) + (sub & 1);
      out[i] = __float2bfloat16(cs < CS ? W[((size_t)(kh * 4 + kw) * CL + c) * CS + cs] : 0.0f);
    }
  } else if (jb.kind == 7 || jb.kind == 8) {
    // x2 (space-to-depth) packing of a 3-channel k4/s2/p1 kernel W[kh,kw,3,CS]:
    //  kind 7: out[cs][(a,b)][(dy,dx,c4)]   (B operand of the 4-tap L->S GEMM: conv1 forward, conv5t dgrad)
    //  kind 8: out[(dy,dx,c4)][(a,b)][cs]   (B operand of the fused conv5t forward), kh = 2a+dy, kw = 2b+dx
    const long long n = (long long)CS * 64;
    for (long long i = i0; i < n; i += stride) {
      int cs, a, b, dy, dx, c;
      if (jb.kind == 7) {
        cs = (int)(i / 64);
        const int k = (int)(i % 64);
        a = k >> 5; b = (k >> 4) & 1; dy = (k >> 3) & 1; dx = (k >> 2) & 1; c = k & 3;
      } else {
        const int row = (int)(i / (4 * CS)), k = (int)(i % (4 * CS));
        dy = row >> 3; dx = (row >> 2) & 1; c = row & 3;
        a = k / (2 * CS); b = (k / CS) & 1; cs = k % CS;
      }
      const int kh = 2 * a + dy, kw = 2 * b + dx;
      out[i] = __float2bfloat16(c < 3 ? W[(size_t)((kh * 4 + kw) * 3 + c) * CS + cs] : 0.0f);
    }
  } else if (jb.kind == 4 || jb.kind == 5) {
    // strided copy into a zero-padded operand: out[(row_off + r) * ld_out + col_off + k] = W[r*sr + k*sk]
    // (kind 4: bf16 destination, kind 5: fp32 destination); taps = R, CL = K, CS unused
    const int R = jb.taps, K = jb.CL;
    const long long n = (long long)R * K;
    for (long long i = i0; i < n; i += stride) {
      const int r = (int)(i / K), k = (int)(i % K);
      const float v = W[(size_t)r * jb.sr + (size_t)k * jb.sk];
      const size_t o = (size_t)(jb.row_off + r) * jb.ld_out + jb.col_off + k;
      if (jb.kind == 4) out[o] = __float2bfloat16(v);
      else reinterpret_cast<float*>(jb.out)[o] = v;
    }
  } else {                     // c4: out[cs][(tap, c4)], W = [16][3][CS]
    const long long n = (long long)CS * 64;
    for (long long i = i0; i < n; i += stride) {
      const int cs = (int)(i / 64), k = (int)(i % 64), t = k >> 2, c = k & 3;
      out[i] = __float2bfloat16(c < 3 ? W[(size_t)(t * 3 + c) * CS + cs] : 0.0f);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Space-to-depth ("x2") form of the two 3-channel end layers.  A 64x64x3 image is stored as 33x33 blocks of
// 2x2 pixels x 4 channels (3 + 1 zero), shifted by one pixel so that block (i, j) holds pixels
// (2i-1+dy, 2j-1+dx):   X2[n, i, j, (dy, dx, c4)]  (bf16, 32-byte rows, zero outside the image).
// Then Conv2D(k4, s2, p1) over the image is a 2x2-tap stride-1 convolution over the blocks,
//     out[oh, ow] = sum_{a,b in {0,1}} X2[oh + a, ow + b, :] . W[(2a+dy, 2b+dx, c)],
// i.e. a 4-tap tap-GEMM with K = 16 per tap (conv1 forward, conv5t dgrad) and a 64-row MN-major wgrad, and
// Conv2DTranspose(k4, s2, p1) PRODUCES its output in the same block form from 2x2 taps of its input,
//     out2[i, j, (dy,dx,c)] = sum_{a,b} S[i - a, j - b, :] . W[(2a+dy, 2b+dx, c)].
// 36 MB per 1024 images instead of the 134 MB K=64 im2col matrix, and no separate im2col / reconstruction pass.
// ---------------------------------------------------------------------------------------------------
// uint8 pixels are normalised through a 256-entry table of float(u) / 255.0f computed ONCE on the host with IEEE
// division (utils_data.py:57-59: np.float32(img) / 255.0, bit-exact); an in-kernel __fdiv_rn costs ~10 instructions
// and a slow-path branch per pixel, which serialised the epilogue's independent chains (83 vs 58 us).
__device__ float g_u8lut[256];
static int ensure_u8lut() {
  static bool done = false;
  if (!done) {
    float h[256];
    for (int i = 0; i < 256; ++i) h[i] = (float)i / 255.0f;
    GCC_CUDA(cudaMemcpyToSymbol(g_u8lut, h, sizeof(h)));
    done = true;
  }
  return GCCVAE_OK;
}
template <typename XT>
__device__ __forceinline__ float load_px(const XT* p, const float* lut);
template <>
__device__ __forceinline__ float load_px<float>(const float* p, const float*) { return __ldg(p); }
template <>
__device__ __forceinline__ float load_px<uint8_t>(const uint8_t* p, const float* lut) { return lut[__ldg(p)]; }

template <typename XT>
__device__ __forceinline__ float px_value(XT raw, const float* lut);
template <>
__device__ __forceinline__ float px_value<float>(float raw, const float*) { return raw; }
template <>
__device__ __forceinline__ float px_value<uint8_t>(uint8_t raw, const float* lut) { return lut[raw]; }

// one thread per block (n, i, j): 4 pixels x 3 channels in, 32 bytes out
// The pad channel of the block's LAST pixel slot (element 15) is the constant 1.0 instead of 0: the layers that read X2
// have zero weights for the pad channels, and in conv1's weight gradient (gccvae_tap4_wg_bf16) the operand row of tap
// (0, 0), slot (1, 1), pad channel is then a row of ones over all 32 x 32 output pixels - its product with the S operand
// is the BIAS gradient, computed by MMAs that run anyway (a separate column-sum pass over the 67 MB of conv2's dgrad
// output was the last launch of the step).
// XB (uint8 images only, optional): the RAW bytes of the block, [B,33,33,16] uint8 = 4 pixels x 3 channels + 4 zero bytes
// (zero outside the image) - what the fused likelihood kernel reads back with one 16-byte load per block.
template <typename XT>
__device__ __forceinline__ uint32_t raw_byte(XT) { return 0u; }
template <>
__device__ __forceinline__ uint32_t raw_byte<uint8_t>(uint8_t v) { return (uint32_t)v; }

template <typename XT>
__global__ void __launch_bounds__(256) prep_x2_kernel(const XT* __restrict__ x, long long total, uint4* __restrict__ X2,
                                                      uint4* __restrict__ XB) {
  pdl_launch_dependents();
  __shared__ float s_lut[256];
  s_lut[threadIdx.x] = g_u8lut[threadIdx.x];   // written once at library initialisation, never by a kernel
  __syncthreads();
  pdl_wait();
  for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total; idx += (long long)gridDim.x * 256) {
    const int j = (int)(idx % 33), i = (int)((idx / 33) % 33);
    const long long n = idx / (33 * 33);
    uint32_t w[8];
    uint32_t rb[3] = {0u, 0u, 0u};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int Y = 2 * i - 1 + (q >> 1), X = 2 * j - 1 + (q & 1);
      float v0 = 0.f, v1 = 0.f, v2 = 0.f;
      if ((unsigned)Y < 64u && (unsigned)X < 64u) {
        const XT* px = x + ((n * 64 + Y) * 64 + X) * 3;
        v0 = load_px<XT>(px, s_lut); v1 = load_px<XT>(px + 1, s_lut); v2 = load_px<XT>(px + 2, s_lut);
#pragma unroll
        for (int c = 0; c < 3; ++c) rb[(3 * q + c) >> 2] |= raw_byte<XT>(__ldg(px + c)) << (8 * ((3 * q + c) & 3));
      }
      w[2 * q] = pack_bf16x2(v0, v1);
      w[2 * q + 1] = pack_bf16x2(v2, q == 3 ? 1.0f : 0.0f);   // the block's last pad slot carries the constant 1 (see above)
    }
    X2[2 * idx] = make_uint4(w[0], w[1], w[2], w[3]);
    X2[2 * idx + 1] = make_uint4(w[4], w[5], w[6], w[7]);
    if (XB != nullptr) XB[idx] = make_uint4(rb[0], rb[1], rb[2], 0u);
  }
}

// uint8 images: one CTA per image stages the 12 288 bytes in shared memory with coalesced 16-byte loads (the kernel
// above issues twelve 1-byte loads per block: 16 us for 1024 images against ~8 us of HBM time), then every thread builds
// blocks from shared memory.  Same table lookup, same output bits.
__global__ void __launch_bounds__(256) prep_x2_u8_staged_kernel(const uint8_t* __restrict__ x, int batch, uint4* __restrict__ X2,
                                                                uint4* __restrict__ XB) {
  pdl_launch_dependents();
  __shared__ float s_lut[256];
  __shared__ __align__(16) uint8_t s_img[64 * 64 * 3];
  s_lut[threadIdx.x] = g_u8lut[threadIdx.x];
  pdl_wait();
  for (int n = blockIdx.x; n < batch; n += gridDim.x) {
    __syncthreads();   // the previous image's readers are done (and the table is in place)
    const uint4* src = reinterpret_cast<const uint4*>(x + (size_t)n * 12288);
#pragma unroll
    for (int t = 0; t < 3; ++t) reinterpret_cast<uint4*>(s_img)[threadIdx.x + 256 * t] = __ldg(src + threadIdx.x + 256 * t);
    __syncthreads();
    for (int blk = threadIdx.x; blk < 33 * 33; blk += 256) {
      const int j = blk % 33, i = blk / 33;
      uint32_t w[8];
      uint32_t rb[3] = {0u, 0u, 0u};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int Y = 2 * i - 1 + (q >> 1), X = 2 * j - 1 + (q & 1);
        float v0 = 0.f, v1 = 0.f, v2 = 0.f;
        if ((unsigned)Y < 64u && (unsigned)X < 64u) {
          const uint8_t* px = s_img + (Y * 64 + X) * 3;
          v0 = s_lut[px[0]]; v1 = s_lut[px[1]]; v2 = s_lut[px[2]];
#pragma unroll
          for (int c = 0; c < 3; ++c) rb[(3 * q + c) >> 2] |= (uint32_t)px[c] << (8 * ((3 * q + c) & 3));
        }
        w[2 * q] = pack_bf16x2(v0, v1);
        w[2 * q + 1] = pack_bf16x2(v2, q == 3 ? 1.0f : 0.0f);
      }
      const size_t o = ((size_t)n * 1089 + blk) * 2;
      X2[o] = make_uint4(w[0], w[1], w[2], w[3]);
      X2[o + 1] = make_uint4(w[4], w[5], w[6], w[7]);
      if (XB != nullptr) XB[(size_t)n * 1089 + blk] = make_uint4(rb[0], rb[1], rb[2], 0u);
    }
  }
}

// conv5t = Conv2DTranspose(32 -> 3, k4, s2, same) + sigmoid, with one of four epilogues (OUT):
//   RECON      Laplace log-likelihood (utils.py:101-105) + its gradient w.r.t. the logits, written in block form D2 (the
//              operand of conv5t's dgrad and wgrad); optional fp32 reconstruction and bias gradient - the training step
//   LL         Laplace log-likelihood of decoded row n against source image n / kc - the importance-weighted likelihood
//   IMAGE_F32  the sigmoid into the [B,64,64,3] fp32 image - the generation path
//   IMAGE_U8   the same as uint8 min(255, rint(255 x))
//   COMPLETE   the sigmoid, bf16-rounded, into the unobserved pixel slots of the encoder's input blocks X2 in place - the
//              composite of one iteration of image completion (gccvae_convt_complete_bf16)
// Output block (i, j) of an image = sum over the 2x2 taps (a, b) of g4[i - a, j - b, :] . W_ab  (K = 32 per tap, N = 16).
// Tile = 128 CONSECUTIVE blocks f = 33 i + j of one image (9 tiles per image, the last one holds 65).  The operand of
// all four taps is ONE TMA box of the decoder activation g4 [B,32,32,32]: 6 image rows x 33 columns starting at column
// -1 (TMA zero-fills the column and the rows outside the image), i.e. the rows' pixels with pitch 33 and a zero pixel
// between consecutive rows.  In that buffer the tap (a, b) of block f0 + m is row  m + d0 + 34 - 33 a - b  (d0 = f0 mod
// 33): a start-address offset of the A descriptor.  The swizzle XOR is taken from the absolute shared-memory address, so
// a K-major operand may start at ANY row of a swizzled buffer (scripts/microbench/desc_offset.cu,
// profiles/r02_microbench_desc_offset.txt) - 198 box rows per tile instead of the 4 x 121 of one box per tap.
enum ConvtOut { RECON, LL, IMAGE_F32, IMAGE_U8, COMPLETE };

struct alignas(64) CtParams {
  CUtensorMap tmA, tmB;
  const void* x;       // RECON / LL: the image operand (form XM)
  int x_u8;
  const float* bias;   // [3]
  const float* coef;   // RECON: [B] dLoss/dlog_pxz per image (NULL: forward only, D2 is not written)
  float* log_pxz;      // RECON / LL: [rows], pre-set to -12288 ln 2; -|x - xhat|_1 is added
  uint4* D2;           // RECON: [B,33,33,16] bf16
  float* xhat;         // RECON: optional [B,64,64,3] fp32 reconstruction
  float* db;           // RECON: optional [3] += sum of dlogit (bias gradient of conv5t)
  int batch, total_tiles, stages;
  long long* timeline;
  void* out;           // IMAGE_*: [B,64,64,3] fp32 or uint8; COMPLETE: the x2 blocks [B,33,33,16] bf16, rewritten in place
  int kc;              // LL: decoded rows per source image
  const uint8_t* mask; // COMPLETE: [B,33,33], bit dy * 2 + dx of block (i, j) set = pixel (2i-1+dy, 2j-1+dx) observed
};

constexpr int CTR_BOX_ROWS = 6 * 33;          // rows of the A box (64 bytes each)
constexpr int CTR_A_STAGE = 13 * 1024;        // >= CTR_BOX_ROWS * 64, a multiple of the swizzle pattern

__device__ __forceinline__ float ex2_approx(float v) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ float rcp_approx(float v) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

// XM = form of the image operand of RECON / LL: 0 fp32 NHWC, 1 uint8 NHWC, 2 uint8 raw-byte blocks XB [B,33,33,16]
// (prep_x2).  The IMAGE kinds and COMPLETE read no image and are instantiated with XM = 0.
// XM = 2: the 2 KB of raw bytes of a tile's 128 blocks travel with the tile's operand box (one bulk copy into the same
// pipeline stage, same barrier); the stage is free again when the MMAs have read the box AND the four epilogue warps have
// taken their bytes.  A register prefetch one tile ahead (XM = 0 / 1) is too short: a tile's epilogue is ~0.3 us of work,
// an HBM access under load ~1.3 us (scripts/timeline_ctr.py: the epilogue warps sat ~1.1 us per tile on that load).
constexpr int CTR_X_BYTES = 128 * 16;
template <int OUT, int XM>
__global__ void __launch_bounds__(TG_THREADS, 4) convt_kernel(const __grid_constant__ CtParams p) {
  constexpr bool HAS_X = OUT == RECON || OUT == LL;   // reads an image operand
  static_assert(HAS_X || XM == 0, "the IMAGE kinds and COMPLETE are instantiated with XM = 0");
  constexpr bool RAW_X = HAS_X && XM == 2;            // the raw image bytes travel with the pipeline stage
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  constexpr int B_TAP = 1024;
  constexpr int STAGE = CTR_A_STAGE + (RAW_X ? CTR_X_BYTES : 0);   // [A box][raw bytes of the tile's blocks]
  uint8_t* sB = smem;                 // 4 taps x [16 rows x 64 B]
  uint8_t* sA = smem + 4 * B_TAP;
  uint64_t* full = reinterpret_cast<uint64_t*>(sA + p.stages * STAGE);
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;
  uint64_t* tempty = tfull + 2;
  uint64_t* bfull = tempty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);
  float* s_db = reinterpret_cast<float*>(tmem_slot + 4);   // [4]
  float* s_lut = s_db + 4;                                 // [256] uint8 -> float(u) / 255
  // the source image of decoded row n
  auto src_image = [&](int n) {
    if constexpr (OUT == LL) return n / p.kc;
    else return n;
  };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  const int per_cta = (p.total_tiles + (int)gridDim.x - 1) / (int)gridDim.x;
  const int tile_beg = blockIdx.x * per_cta;
  const int tile_end = min(tile_beg + per_cta, p.total_tiles);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmB);
    // empty[s] completes when the MMA commit AND, when RAW_X, the four epilogue warps (which take their raw bytes from
    // the stage) have arrived: the count must be 5 exactly when the epilogue warps arrive on it, else the producer hangs
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], RAW_X ? 5 : 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 4);
    }
    mbar_init(bfull, 1);
    fence_mbar_init();
  }
  if (OUT == RECON && threadIdx.x < 4) s_db[threadIdx.x] = 0.0f;
  if constexpr (HAS_X)
    for (int i = threadIdx.x; i < 256; i += TG_THREADS) s_lut[i] = g_u8lut[i];
  if (RAW_X)   // the last tile of an image brings 65 blocks: the other rows read whatever the stage holds (masked)
    for (int i = threadIdx.x; i < p.stages * (CTR_X_BYTES / 16); i += TG_THREADS)
      reinterpret_cast<uint4*>(sA + (i / (CTR_X_BYTES / 16)) * STAGE + CTR_A_STAGE)[i % (CTR_X_BYTES / 16)] = make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes above, async-proxy (bulk copy) writes later
  if (warp == 2) tmem_alloc(tmem_slot, 64);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (TL_ON(p) && threadIdx.x == 0 && blockIdx.x < 1024) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    p.timeline[40 * 8 + 2 * blockIdx.x] = (long long)gt;
  }
  pdl_wait();

  if (warp == 0) {
    if (elect_one() && tile_beg < tile_end) {
      mbar_expect_tx(bfull, 4 * B_TAP);
      for (int t = 0; t < 4; ++t) tma_load_2d(sB + t * B_TAP, &p.tmB, bfull, t * 32, 0);
      int stage = 0;
      uint32_t ph = 0;
      int n = tile_beg / 9, k = tile_beg - n * 9;
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        const int i_first = (k * 128) / 33;
        const uint32_t xbytes = RAW_X ? (uint32_t)min(128, 33 * 33 - k * 128) * 16u : 0u;
        mbar_wait_relaxed(&empty[stage], ph ^ 1);   // runs stages ahead of its consumers: back off instead of spinning
        TL(tile - tile_beg, 0);
        mbar_expect_tx(&full[stage], CTR_BOX_ROWS * 64 + xbytes);
        tma_load_4d(sA + stage * STAGE, &p.tmA, &full[stage], 0, -1, i_first - 1, n);
        if (RAW_X)
          bulk_load_1d(sA + stage * STAGE + CTR_A_STAGE,
                       reinterpret_cast<const uint4*>(p.x) + ((size_t)src_image(n) * 1089 + (size_t)k * 128), xbytes,
                       &full[stage]);
        TL(tile - tile_beg, 1);
        if (++stage == p.stages) { stage = 0; ph ^= 1; }
        if (++k == 9) { k = 0; ++n; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && tile_beg < tile_end) {
      const uint32_t idesc = instr_desc_bf16(128, 16, 0, 0);
      const uint64_t dproto = smem_desc(0, 16, 8u * 64u, SW_64);
      const uint64_t adesc0 = dproto + (uint64_t)(smem_u32(sA) >> 4), bdesc0 = dproto + (uint64_t)(smem_u32(sB) >> 4);
      int stage = 0;
      uint32_t ph = 0;
      int k = tile_beg % 9;
      mbar_wait(bfull, 0);
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        const int li = tile - tile_beg, as = li & 1;
        const int f0 = k * 128, d0 = f0 - (f0 / 33) * 33;
        mbar_wait(&tempty[as], ((uint32_t)(li >> 1) & 1u) ^ 1u);
        TL(li, 2);
        mbar_wait(&full[stage], ph);
        tc_fence_after();
        TL(li, 3);
        // descriptor units are 16 bytes: one operand row = 4
        const uint64_t a_st = adesc0 + (uint64_t)((uint32_t)stage * (STAGE >> 4) + (uint32_t)(d0 + 34) * 4u);
        const uint32_t tacc = tmem_base + (uint32_t)as * 32u;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const uint32_t row_off = (uint32_t)(33 * (t >> 1) + (t & 1)) * 4u;   // tap (a, b) = (t >> 1, t & 1)
#pragma unroll
          for (int kk = 0; kk < 2; ++kk)
            umma_bf16(tacc, a_st - (uint64_t)row_off + (uint64_t)(2 * kk), bdesc0 + (uint64_t)(t * (B_TAP >> 4) + 2 * kk),
                      idesc, (t > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(&empty[stage]);
        umma_commit(&tfull[as]);
        TL(li, 7);
        if (++stage == p.stages) { stage = 0; ph ^= 1; }
        if (++k == 9) k = 0;
      }
    }
  } else {
    const int q = warp & 3;
    const int m = q * 32 + lane;
    constexpr float LOG2E = 1.4426950408889634f;
    const float nb0 = -LOG2E * __ldg(p.bias), nb1 = -LOG2E * __ldg(p.bias + 1), nb2 = -LOG2E * __ldg(p.bias + 2);
    float d0 = 0.f, d1 = 0.f, d2 = 0.f;
    // XM = 0 / 1: the image pixels of a block are fetched from the NHWC image one tile AHEAD (register double buffer),
    // branch-free - coordinates clamped into the image, out-of-image pixels masked by `ok` below - and keep their RAW
    // form; the uint8 -> float table lookup happens when the values are consumed.
    using XT = typename std::conditional<XM == 0, float, uint8_t>::type;
    XT xn[XM == 2 ? 1 : 12];
    auto fetch_x = [&](int n, int k) {
      if constexpr (HAS_X && XM != 2) {
        const int f = k * 128 + m;
        const XT* xs = reinterpret_cast<const XT*>(p.x);
        const int i = f / 33, j = f - i * 33;
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
          const int Y = min(max(2 * i - 1 + (qq >> 1), 0), 63), X = min(max(2 * j - 1 + (qq & 1), 0), 63);
          const XT* px = xs + (((size_t)src_image(n) * 64 + Y) * 64 + X) * 3;
          xn[3 * qq] = __ldg(px); xn[3 * qq + 1] = __ldg(px + 1); xn[3 * qq + 2] = __ldg(px + 2);
        }
      }
    };
    int n = tile_beg / 9, k = tile_beg - n * 9;
    if (tile_beg < tile_end) fetch_x(n, k);
    float l1 = 0.0f;   // |x - xhat|_1 of this thread's blocks of the current row
    int stage = 0;
    uint32_t ph = 0;
    for (int tile = tile_beg; tile < tile_end; ++tile) {
      const int li = tile - tile_beg, as = li & 1;
      const int f = k * 128 + m, i = f / 33, j = f - i * 33;
      const bool row_ok = f < 33 * 33;
      const int n_cur = n;
      uint32_t mbits = 0xfu;   // COMPLETE: the block's mask byte, loaded here so that its latency hides behind the wait below
      if constexpr (OUT == COMPLETE)
        if (row_ok) mbits = __ldg(p.mask + (size_t)n_cur * 1089 + f);
      // (consumed at the very end of the tile: an L2 access that needs no prefetch)
      const float cb = OUT == RECON && p.coef != nullptr ? __ldg(p.coef + n_cur) : 0.0f;
      float xv[12];
      uint4 xb = make_uint4(0u, 0u, 0u, 0u);
      if constexpr (RAW_X) {
        mbar_wait(&full[stage], ph);     // the MMA thread waits on the same phase; here it makes the bulk copy visible
        xb = lds_u4(smem_u32(sA + stage * STAGE + CTR_A_STAGE) + (uint32_t)m * 16u);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
        if (++stage == p.stages) { stage = 0; ph ^= 1; }
      } else if constexpr (HAS_X) {
#pragma unroll
        for (int k2 = 0; k2 < 12; ++k2) xv[k2] = px_value<XT>(xn[k2], s_lut);
      }
      if (++k == 9) { k = 0; ++n; }
      if (tile + 1 < tile_end) fetch_x(n, k);
      mbar_wait(&tfull[as], (uint32_t)(li >> 1) & 1u);
      tc_fence_after();
      if (threadIdx.x == 64) TL(li, 4);
      uint32_t acc[16];
      tmem_ld16(tmem_base + (uint32_t)as * 32u + ((uint32_t)(q * 32) << 16), acc);
      tmem_ld_wait();
      tc_fence_before();
      if (lane == 0) mbar_arrive(&tempty[as]);
      if (threadIdx.x == 64) TL(li, 5);
      if constexpr (RAW_X) {   // table lookups: their shared-memory latency hides behind the sigmoid chains below
        const uint32_t w[3] = {xb.x, xb.y, xb.z};
#pragma unroll
        for (int k2 = 0; k2 < 12; ++k2) xv[k2] = s_lut[(w[k2 >> 2] >> (8 * (k2 & 3))) & 0xffu];
      }
      // pixel (dy, dx) of block (i, j) lies in the image unless the block touches that border
      const bool oky[2] = {row_ok && i > 0, row_ok && i < 32}, okx[2] = {j > 0, j < 32};
      bool ok[4];
      float okf[4];
#pragma unroll
      for (int qq = 0; qq < 4; ++qq) {
        ok[qq] = oky[qq >> 1] && okx[qq & 1];
        okf[qq] = ok[qq] ? 1.0f : 0.0f;
      }
      // branch-free arithmetic, 12 independent chains: xhat = 1 / (1 + 2^(-(a + b) log2 e)); every row of the tile reads
      // operand rows the box has written (zero-filled outside the image), so rows without work hold finite values
      float xh[12];
#pragma unroll
      for (int k2 = 0; k2 < 12; ++k2) {
        const int qq = k2 / 3, c = k2 % 3;
        const float t = fmaf(__uint_as_float(acc[4 * qq + c]), -LOG2E, c == 0 ? nb0 : (c == 1 ? nb1 : nb2));
        xh[k2] = rcp_approx(1.0f + ex2_approx(t));
      }
      if constexpr (OUT == RECON) {
        float g[12], cq[4];
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) cq[qq] = okf[qq] * cb;
#pragma unroll
        for (int k2 = 0; k2 < 12; ++k2) {
          const int qq = k2 / 3;
          const float e = xv[k2] - xh[k2];
          l1 = fmaf(okf[qq], fabsf(e), l1);
          // dLoss/dlogit = coef * sign(x - xhat) * xhat (1 - xhat):  the sign bit of e flips s, e == 0 gives 0
          const float s = fmaf(-xh[k2], xh[k2], xh[k2]) * cq[qq];
          const float sg = __uint_as_float(__float_as_uint(s) ^ (__float_as_uint(e) & 0x80000000u));
          g[k2] = e != 0.0f ? sg : 0.0f;
        }
        d0 += g[0] + g[3] + g[6] + g[9];
        d1 += g[1] + g[4] + g[7] + g[10];
        d2 += g[2] + g[5] + g[8] + g[11];
        if (p.D2 != nullptr && row_ok) {
          uint4* dst = p.D2 + ((size_t)n_cur * 1089 + f) * 2;
          dst[0] = make_uint4(pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], 0.0f), pack_bf16x2(g[3], g[4]), pack_bf16x2(g[5], 0.0f));
          dst[1] = make_uint4(pack_bf16x2(g[6], g[7]), pack_bf16x2(g[8], 0.0f), pack_bf16x2(g[9], g[10]), pack_bf16x2(g[11], 0.0f));
        }
        if (p.xhat != nullptr) {   // optional fp32 reconstruction (tests / module API), off the training path
#pragma unroll
          for (int qq = 0; qq < 4; ++qq)
            if (ok[qq]) {
              const int Y = 2 * i - 1 + (qq >> 1), X = 2 * j - 1 + (qq & 1);
              float* dstx = p.xhat + (((size_t)n_cur * 64 + Y) * 64 + X) * 3;
              dstx[0] = xh[3 * qq]; dstx[1] = xh[3 * qq + 1]; dstx[2] = xh[3 * qq + 2];
            }
        }
      } else if constexpr (OUT == LL) {
#pragma unroll
        for (int k2 = 0; k2 < 12; ++k2) l1 = fmaf(okf[k2 / 3], fabsf(xv[k2] - xh[k2]), l1);
      } else if constexpr (OUT == COMPLETE) {
        // an unobserved pixel's 8 bytes are rewritten as prep_x2 writes them: its three channels, then the pad lane (0, or
        // the block's constant 1.0 in element 15); observed and out-of-image pixels keep their bytes, and a block without
        // an unobserved pixel is not stored at all
        uint2* dst = static_cast<uint2*>(p.out) + ((size_t)n_cur * 1089 + f) * 4;
#pragma unroll
        for (int qq = 0; qq < 4; ++qq)
          if (ok[qq] && !((mbits >> qq) & 1u))
            dst[qq] = make_uint2(pack_bf16x2(xh[3 * qq], xh[3 * qq + 1]), pack_bf16x2(xh[3 * qq + 2], qq == 3 ? 1.0f : 0.0f));
      } else {
#pragma unroll
        for (int qq = 0; qq < 4; ++qq)
          if (ok[qq]) {
            const int Y = 2 * i - 1 + (qq >> 1), X = 2 * j - 1 + (qq & 1);
            const size_t o = (((size_t)n_cur * 64 + Y) * 64 + X) * 3;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              if constexpr (OUT == IMAGE_U8)
                static_cast<uint8_t*>(p.out)[o + c] = (uint8_t)min(255u, __float2uint_rn(__fmul_rn(255.0f, xh[3 * qq + c])));
              else
                static_cast<float*>(p.out)[o + c] = xh[3 * qq + c];
            }
          }
      }
      // the likelihood sum leaves the registers once per row (and at the end of the CTA's range), not once per tile:
      // five dependent shuffles per tile were 10 % of the kernel's stall samples
      if (HAS_X && (k == 0 || tile + 1 == tile_end)) {
        l1 = warp_sum(l1);
        if (lane == 0 && l1 != 0.0f) atomicAdd(p.log_pxz + n_cur, -l1);
        l1 = 0.0f;
      }
      if (threadIdx.x == 64) TL(li, 6);
    }
    if (OUT == RECON && p.db != nullptr) {
      d0 = warp_sum(d0); d1 = warp_sum(d1); d2 = warp_sum(d2);
      if (lane == 0) { atomicAdd(&s_db[0], d0); atomicAdd(&s_db[1], d1); atomicAdd(&s_db[2], d2); }
    }
    tc_fence_before();
  }
  if (TL_ON(p) && threadIdx.x == 0 && blockIdx.x < 1024) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    p.timeline[40 * 8 + 2 * blockIdx.x + 1] = (long long)gt;
  }
  __syncthreads();
  if (OUT == RECON && p.db != nullptr && threadIdx.x < 3 && s_db[threadIdx.x] != 0.0f) atomicAdd(p.db + threadIdx.x, s_db[threadIdx.x]);
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 64);
  }
}

// ---------------------------------------------------------------------------------------------------
// L -> S convolution of a 3-channel image in x2 block form (conv1 forward, conv5t dgrad) with the im2col tile
// built by four producer warps instead of TMA: TMA moves one box row per ~1.3 cycles whatever its width, so
// four taps of 128 32-byte rows cost as much as 128 KB of traffic, while 128 threads gather the same four
// 32-byte blocks per output pixel with 8 coalesced 16-byte loads and write ONE 128-byte K-major row each
// (SWIZZLE_128B pattern: 16-byte chunk c of row r lands at chunk c ^ (r & 7)).  K = 64 = (a, b, dy, dx, c4).
// Warps 0-3: producers, warp 4: MMA issuer, warps 5-8: epilogue (TMEM lane quadrant = warp % 4).
// ---------------------------------------------------------------------------------------------------
struct alignas(64) C3Params {
  CUtensorMap tmB;          // packed weights [N rows][64] bf16 (pack kind 7), box (64, N)
  const uint4* in2;         // [B,33,33,16] bf16 blocks (2 x uint4 per block)
  void* out;                // [B,32,32,N] bf16
  const void* mask;         // optional [B,32,32,N] bf16: out *= (mask > 0)
  const float* bias;        // optional [N]
  int act, N, batch, total_tiles, stages;
  int out_s2d;              // store the 32x32xN output in s2d block form [B,17,17,4N]
  long long* timeline;      // debug (see TL)
};
constexpr int C3_THREADS = 288;

template <int NCH>   // N / 16
__global__ void __launch_bounds__(C3_THREADS, 2) c3conv_kernel(const __grid_constant__ C3Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  constexpr int A_TILE = 128 * 128;
  uint8_t* sB = smem;                       // N x 128 B (<= 8 KB reserved)
  uint8_t* sA = smem + 8192;
  uint64_t* full = reinterpret_cast<uint64_t*>(sA + p.stages * A_TILE);
  uint64_t* empty = full + p.stages;
  constexpr int ACC = 4;                 // accumulator stages in TMEM
  uint64_t* tfull = empty + p.stages;
  uint64_t* tempty = tfull + ACC;
  uint64_t* bfull = tempty + ACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);
  float* s_bias = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 15) & ~(uintptr_t)15);   // [64]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  const int per_cta = (p.total_tiles + (int)gridDim.x - 1) / (int)gridDim.x;
  const int tile_beg = blockIdx.x * per_cta;
  const int tile_end = min(tile_beg + per_cta, p.total_tiles);
  uint32_t acc_cols = 32;
  while ((int)acc_cols < p.N) acc_cols <<= 1;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 128);   // one asynchronous arrival per producer thread (its cp.async group landed)
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < ACC; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 4);
    }
    mbar_init(bfull, 1);
    fence_mbar_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, acc_cols * ACC);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 128 && tile_beg < tile_end) {   // weights are parameters: not produced by the predecessor
    mbar_expect_tx(bfull, (uint32_t)(p.N * 128));
    tma_load_2d(sB, &p.tmB, bfull, 0, 0);
  }
  pdl_wait();

  if (warp < 4) {
    // ===== producers: thread m builds row m of the im2col tile with 8 cp.async of 16 bytes; completion is
    // tracked by the stage's mbarrier (cp.async.mbarrier.arrive.noinc), so up to `stages` tiles are in flight =====
    const int m = threadIdx.x;
    const int dy = m >> 5, dx = m & 31;
    const uint32_t row_off = (uint32_t)m * 128u, sw = (uint32_t)(m & 7);
    int stage = 0;
    uint32_t ph = 0;
    for (int tile = tile_beg; tile < tile_end; ++tile) {
      const int n = tile >> 3, h0 = (tile & 7) * 4;
      const uint4* src = p.in2 + (((size_t)n * 33 + (h0 + dy)) * 33 + dx) * 2;
      mbar_wait_relaxed(&empty[stage], ph ^ 1);
      if (m == 0) TL(tile - tile_beg, 0);
      const uint32_t dst = smem_u32(sA + stage * A_TILE) + row_off;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const uint4* sp = src + ((t >> 1) * 33 + (t & 1)) * 2;
#pragma unroll
        for (int h = 0; h < 2; ++h)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + ((((uint32_t)(2 * t + h)) ^ sw) << 4)),
                       "l"(sp + h)
                       : "memory");
      }
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&full[stage])) : "memory");
      if (m == 0) TL(tile - tile_beg, 1);
      if (++stage == p.stages) { stage = 0; ph ^= 1; }
    }
  } else if (warp == 4) {
    if (lane == 0 && tile_beg < tile_end) {
      const uint32_t idesc = instr_desc_bf16(128, p.N, 0, 0);
      const uint64_t dproto = smem_desc(0, 16, 1024, SW_128);
      const uint64_t adesc0 = dproto + (uint64_t)(smem_u32(sA) >> 4), bdesc = dproto + (uint64_t)(smem_u32(sB) >> 4);
      int stage = 0;
      uint32_t ph = 0;
      mbar_wait(bfull, 0);
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        const int li = tile - tile_beg, as = li & (ACC - 1);
        mbar_wait(&tempty[as], ((uint32_t)(li / ACC) & 1u) ^ 1u);
        TL(li, 2);
        mbar_wait(&full[stage], ph);
        TL(li, 3);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // cp.async (generic proxy) -> MMA (async proxy)
        tc_fence_after();
        const uint64_t ad = adesc0 + (uint64_t)((uint32_t)stage * (A_TILE >> 4));
        const uint32_t tacc = tmem_base + (uint32_t)as * acc_cols;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) umma_bf16(tacc, ad + 2u * kk, bdesc + 2u * kk, idesc, kk > 0 ? 1u : 0u);
        umma_commit(&empty[stage]);
        umma_commit(&tfull[as]);
        TL(li, 7);
        if (++stage == p.stages) { stage = 0; ph ^= 1; }
      }
    }
  } else {
    // ===== epilogue =====
    const int q = warp & 3;
    const int m = q * 32 + lane;
    const int dy = m >> 5, dx = m & 31;
    // the bias lives in shared memory: a global load per tile would miss L1 (the image stream evicts it) and put an
    // L2 round trip on the epilogue's critical path
    {
      const int et = threadIdx.x - 160;
      if (et < 64) s_bias[et] = (p.bias != nullptr && et < p.N) ? p.bias[et] : 0.0f;
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    const uint32_t s_bias_u32 = smem_u32(s_bias);
    // the ReLU mask does not depend on the accumulator: it is fetched one tile ahead (register double buffer)
    const bool use_mask = p.mask != nullptr;
    uint32_t mnext[NCH][8];
    auto fetch_mask = [&](int tile, uint32_t (&mm)[NCH][8]) {
      const int n = tile >> 3, h0 = (tile & 7) * 4;
      const size_t opix = ((size_t)n * 32 + (h0 + dy)) * 32 + dx;
      const __nv_bfloat16* mk = reinterpret_cast<const __nv_bfloat16*>(p.mask) + opix * p.N;
#pragma unroll
      for (int i = 0; i < NCH; ++i) ld_global_nc_256(mk + i * 16, mm[i]);
    };
    if (use_mask && tile_beg < tile_end) fetch_mask(tile_beg, mnext);
    for (int tile = tile_beg; tile < tile_end; ++tile) {
      const int li = tile - tile_beg, as = li & (ACC - 1);
      const int n = tile >> 3, h0 = (tile & 7) * 4;
      const size_t opix = p.out_s2d ? s2d_slot(n, h0 + dy, dx, 32, 32) : ((size_t)n * 32 + (h0 + dy)) * 32 + dx;
      uint32_t mpre[NCH][8];
      if (use_mask) {
#pragma unroll
        for (int i = 0; i < NCH; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) mpre[i][j] = mnext[i][j];
        if (tile + 1 < tile_end) fetch_mask(tile + 1, mnext);
      }
      mbar_wait(&tfull[as], (uint32_t)(li / ACC) & 1u);
      tc_fence_after();
      if (threadIdx.x == 160) TL(li, 4);
      const uint32_t tacc = tmem_base + (uint32_t)as * acc_cols + ((uint32_t)(q * 32) << 16);
      // all TMEM loads of the tile are issued back to back, ONE wait, and the accumulator stage goes back to the MMA
      // warp before any arithmetic
      uint32_t r[NCH][16];
#pragma unroll
      for (int c = 0; c < NCH; ++c) tmem_ld16(tacc + (uint32_t)(c * 16), r[c]);
      tmem_ld_wait();
      tc_fence_before();
      if (lane == 0) mbar_arrive(&tempty[as]);
      if (threadIdx.x == 160) TL(li, 5);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int c0 = c * 16;
        float v[16];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 t = lds_f4(s_bias_u32 + (uint32_t)(c0 + 4 * i) * 4u);
          v[4 * i] = __uint_as_float(r[c][4 * i]) + t.x;
          v[4 * i + 1] = __uint_as_float(r[c][4 * i + 1]) + t.y;
          v[4 * i + 2] = __uint_as_float(r[c][4 * i + 2]) + t.z;
          v[4 * i + 3] = __uint_as_float(r[c][4 * i + 3]) + t.w;
        }
        if (p.act == GCCVAE_ACT_RELU) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.0f);
        }
        if (use_mask) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t mwi = mpre[c][i];
            const uint32_t lo = mwi & 0xffffu, hi = mwi >> 16;
            if (!(lo != 0 && lo < 0x8000u)) v[2 * i] = 0.0f;
            if (!(hi != 0 && hi < 0x8000u)) v[2 * i + 1] = 0.0f;
          }
        }
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
        st_global_256(reinterpret_cast<__nv_bfloat16*>(p.out) + opix * p.N + c0, w);
      }
      if (threadIdx.x == 160) TL(li, 6);
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, acc_cols * ACC);
  }
}

// debug aid: one 4-D TMA box load, raw shared-memory image copied out (layout / OOB / stride checks)
__global__ void tma_dump_kernel(const __grid_constant__ CUtensorMap tm, int c0, int c1, int c2, int c3, int bytes,
                                uint8_t* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  __shared__ uint64_t bar;
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) smem[i] = 0xEE;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar, (uint32_t)bytes);
    tma_load_4d(smem, &tm, &bar, c0, c1, c2, c3);
  }
  mbar_wait(&bar, 0);
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) out[i] = smem[i];
}

// ---------------------------------------------------------------------------------------------------
// weight packing: fp32 Keras kernel W[kh,kw,CL,CS] -> bf16 GEMM operands
//   ls[cs][ (kh,kw,cl) ]                       (rows padded to a multiple of 16, zero filled)
//   sl[phase][cl][ (th,tw,cs) ], kh = (ph+1)%2 + 2 th  (k4/s2/p1 only)
//   dense S->L:  sl[(kh,kw,cl)][cs] is W itself cast to bf16
// ---------------------------------------------------------------------------------------------------
__global__ void pack_ls_kernel(const float* __restrict__ W, int taps, int CL, int CS, int rows_pad,
                               __nv_bfloat16* __restrict__ out) {
  const int K = taps * CL;
  const long long n = (long long)rows_pad * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int cs = (int)(i / K), k = (int)(i % K);
    out[i] = __float2bfloat16(cs < CS ? W[(size_t)k * CS + cs] : 0.0f);
  }
}
__global__ void pack_sl2_kernel(const float* __restrict__ W, int CL, int CS, int rows_pad,
                                __nv_bfloat16* __restrict__ out) {
  const int K = 4 * CS;
  const long long n = 4LL * rows_pad * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % K);
    const int cl = (int)((i / K) % rows_pad), phase = (int)(i / ((long long)K * rows_pad));
    const int ph = phase >> 1, pw = phase & 1, t = k / CS, cs = k % CS;
    const int kh = ((ph + 1) & 1) + 2 * (t >> 1), kw = ((pw + 1) & 1) + 2 * (t & 1);
    out[i] = __float2bfloat16(cl < CL ? W[((size_t)(kh * 4 + kw) * CL + cl) * CS + cs] : 0.0f);
  }
}
__global__ void cast_bf16_kernel(const float* __restrict__ in, long long n, __nv_bfloat16* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16(in[i]);
}
__global__ void cast_f32_kernel(const __nv_bfloat16* __restrict__ in, long long n, float* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __bfloat162float(in[i]);
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)f;
  });
  return fn;
}

static CUtensorMapSwizzle tma_swizzle_for(int inner_bytes) {
  return inner_bytes >= 128 ? CU_TENSOR_MAP_SWIZZLE_128B
         : inner_bytes >= 64 ? CU_TENSOR_MAP_SWIZZLE_64B
         : inner_bytes >= 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                             : CU_TENSOR_MAP_SWIZZLE_NONE;
}
static int umma_swizzle_for(int inner_bytes) {
  return inner_bytes >= 128 ? SW_128 : inner_bytes >= 64 ? SW_64 : inner_bytes >= 32 ? SW_32 : SW_NONE;
}

// bf16 NHWC tensor [N,H,W,C] -> 4-D map (c,w,h,n); box = (kc, bw, bh, bn) OUTPUT pixels traversed with
// element stride `es` along w and h.
static int encode_act_map(CUtensorMap* m, const void* ptr, int N, int H, int W, int C, int kc, int bw, int bh, int bn,
                          int es) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)");
    return GCCVAE_ECUDA;
  }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)kc, (cuuint32_t)(bw * es), (cuuint32_t)(bh * es), (cuuint32_t)bn};
  cuuint32_t estr[4] = {1, (cuuint32_t)es, (cuuint32_t)es, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, tma_swizzle_for(kc * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(act %dx%dx%dx%d box %d,%d,%d,%d es %d) failed: %d", N, H, W, C, kc, bw * es,
              bh * es, bn, es, (int)r);
    return GCCVAE_ECUDA;
  }
  return GCCVAE_OK;
}

// bf16 row-major matrix [rows, K] -> 2-D map (k, row); box = (kc, nrows)
static int encode_mat_map(CUtensorMap* m, const void* ptr, long long rows, long long K, int kc, int nrows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)");
    return GCCVAE_ECUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)kc, (cuuint32_t)nrows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, tma_swizzle_for(kc * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(mat %lldx%lld box %d,%d) failed: %d", rows, K, kc, nrows, (int)r);
    return GCCVAE_ECUDA;
  }
  return GCCVAE_OK;
}

static int pick_kc(int C) {
  if (C % 64 == 0) return 64;
  if (C == 32) return 32;
  if (C == 16) return 16;
  return 0;
}

// tile box for a plane of H x W output pixels: BW*BH*BN = 128
static int pick_tile(int H, int W, int* bw, int* bh, int* bn) {
  if (W >= 128 || 128 % W != 0) return -1;
  *bw = W;
  int rest = 128 / W;
  if (H >= rest) {
    if (H % rest != 0) return -1;
    *bh = rest;
    *bn = 1;
  } else {
    if (rest % H != 0) return -1;
    *bh = H;
    *bn = rest / H;
  }
  return 0;
}

// CTAs per SM of the weight-gradient kernels and their shared-memory budget per CTA (KB).  They run on a side stream
// UNDER the dgrad chain: what they occupy is not available to the critical path's persistent CTAs.
constexpr int WG_PER_SM = 2, WG_SMEM_KB = 100;

// tensor-core kernels: launched with programmatic dependent launch (their prologues overlap the predecessor's tail)
template <class Params>
static cudaError_t launch_pdl(void (*kernel)(const Params), dim3 grid, int threads, size_t smem, cudaStream_t st,
                              const Params& p) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = dim3(threads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, p);
}

static long long* g_timeline = nullptr;

static int launch_tapgemm(TapGemmParams& p, int groups, int phases, cudaStream_t st, const char* name) {
  p.timeline = g_timeline;
  if (p.rows_valid <= 0) p.rows_valid = 128;
  if (p.a_box_rows <= 0) p.a_box_rows = 128;
  const int a_stride = (p.a_box_rows * p.KC * 2 + 1023) & ~1023,
            b_stride = ((p.halo2 ? 2 : 1) * p.N * p.KC * 2 + 1023) & ~1023;
  // Persistent CTAs, `per_sm` of them per SM (their epilogues and issue threads overlap).  The single MMA-issuing
  // thread pays ~400 cycles per pipeline stage (barrier wait, fences, commit) and ~50 per MMA, so a stage carries
  // `tps` k-blocks (taps x chunks): few, fat stages.  TMEM: two accumulator stages per CTA, 512 columns per SM.
  uint32_t acc_cols = 32;
  while ((int)acc_cols < p.N) acc_cols <<= 1;
  const int k_iters = p.num_taps * p.chunks;
  int per_sm = 2;
  if (per_sm > 512 / (2 * (int)acc_cols)) per_sm = 512 / (2 * (int)acc_cols);
  if (per_sm < 1) per_sm = 1;
  const int budget = 200 * 1024 / per_sm - 4608;
  const int stage_target = 48 * 1024;
  int tps = 1;
  for (int d = 1; d <= k_iters; ++d)
    if (k_iters % d == 0 && d * (a_stride + b_stride) <= stage_target && 2 * d * (a_stride + b_stride) <= budget) tps = d;
  p.tps = tps;
  int stages = budget / (tps * (a_stride + b_stride));
  if (stages > 8) stages = 8;
  if (stages < 2) stages = 2;
  p.stages = stages;
  const size_t smem = (size_t)stages * tps * (a_stride + b_stride) + 1024 + 256 + 2048 + 64;
  static bool attr_set = false;
  if (!attr_set) {
    GCC_CUDA(cudaFuncSetAttribute(tapgemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    attr_set = true;
  }
  GCC_REQUIRE(smem <= 200 * 1024, "%s: %zu bytes of shared memory", name, smem);
  if (p.n_slabs < 1) p.n_slabs = 1;
  if (p.bias_mod < 1 || p.bias == nullptr) p.bias_mod = 1 << 30;
  if (p.bias_n < 1) p.bias_n = p.n_store;
  GCC_REQUIRE(p.bias_mod >= p.n_store || p.bias_mod % p.N == 0, "%s: bias_mod %d incompatible with N slab %d", name,
              p.bias_mod, p.N);
  GCC_REQUIRE(p.bias == nullptr || ((uintptr_t)p.bias % 16) == 0, "%s: bias must be 16-byte aligned", name);
  p.phases = phases;
  p.total_items = groups * p.tiles_w * p.tiles_h * p.n_slabs * phases;
  // never launch more persistent CTAs than are resident at once: a second wave would serialise behind the first.
  // Residency limits: registers (64K per SM), shared memory (227 KB per SM, 1 KB reserved per CTA), TMEM (above).
  static int regs_per_cta = 0;
  if (regs_per_cta == 0) {
    cudaFuncAttributes fa;
    GCC_CUDA(cudaFuncGetAttributes(&fa, tapgemm_kernel));
    const int per_warp = ((fa.numRegs + 7) / 8) * 8 * 32;
    regs_per_cta = per_warp * (TG_THREADS / 32);
  }
  int occ = 65536 / regs_per_cta;
  const int occ_smem = (int)((227 * 1024) / (smem + 1024));
  if (occ > occ_smem) occ = occ_smem;
  if (occ < 1) occ = 1;
  if (per_sm > occ) per_sm = occ;
  if (getenv("GCCVAE_DEBUG_LAUNCH"))
    fprintf(stderr, "%s: N=%d KC=%d k_iters=%d tps=%d stages=%d smem=%zu per_sm=%d (occ %d) items=%d\n", name, p.N, p.KC,
            k_iters, tps, stages, smem, per_sm, occ, p.total_items);
  int ctas = p.total_items < 148 * per_sm ? p.total_items : 148 * per_sm;
  // even out the work: with ceil(total/ctas) items per CTA fewer CTAs may carry the same maximum
  {
    const int per_cta = (p.total_items + ctas - 1) / ctas;
    ctas = (p.total_items + per_cta - 1) / per_cta;
  }
  dim3 grid(ctas, 1, 1);
  GCC_CUDA(launch_pdl(tapgemm_kernel, grid, TG_THREADS, smem, st, p));
  GCC_CHECK_LAUNCH(name);
  return GCCVAE_OK;
}

}  // namespace gccvae

using namespace gccvae;

// S = act(gather(L) W + b) (* mask>0): bf16 NHWC in/out, Wp = pack "ls" layout.
extern "C" int gccvae_ls_bf16(const gccvae_geom* g, const void* L, const void* Wp_ls, const float* bias, int act,
                              const void* mask, void* S, int out_f32, void* stream) {
  GCC_REQUIRE(g && L && Wp_ls && S, "ls_bf16: null pointer");
  const int kc = pick_kc(g->CL);
  GCC_REQUIRE(kc > 0, "ls_bf16: CL=%d unsupported (need 16, 32 or a multiple of 64)", g->CL);
  GCC_REQUIRE(g->CS % 16 == 0 && g->CS <= 256, "ls_bf16: CS=%d must be a multiple of 16, <= 256", g->CS);
  TapGemmParams p;
  memset(&p, 0, sizeof(p));
  const bool dense = (g->HS == 1 && g->WS == 1 && g->pad == 0 && g->stride == 1);
  int rc, n_slab = g->CS;
  if (dense) {
    // [B, KH*KW*CL] x [KH*KW*CL, CS]: one tap, many chunks
    const int Kt = g->KH * g->KW * g->CL;
    if ((rc = encode_act_map(&p.tmA, L, g->batch, 1, 1, Kt, kc, 1, 1, 128, 1))) return rc;
    p.num_taps = 1; p.chunks = Kt / kc; p.a_scale = 1; p.BW = 1; p.BH = 1; p.BN = 128; p.tiles_w = p.tiles_h = 1;
    p.b_tap_stride = 0;
    // few M tiles (conv5: batch/128): tile N in slabs of 64 so that more SMs take part
    const int m_tiles = (g->batch + 127) / 128;
    n_slab = (m_tiles < 74 && g->CS % 64 == 0 && g->CS > 64) ? 64 : g->CS;
    if ((rc = encode_mat_map(&p.tmB, Wp_ls, g->CS, Kt, kc, n_slab))) return rc;
  } else {
    GCC_REQUIRE(g->KH == 4 && g->KW == 4 && g->stride == 2 && g->pad == 1, "ls_bf16: only k4/s2/p1 or dense");
    int bw, bh, bn;
    GCC_REQUIRE(pick_tile(g->HS, g->WS, &bw, &bh, &bn) == 0, "ls_bf16: cannot tile %dx%d", g->HS, g->WS);
    if ((rc = encode_act_map(&p.tmA, L, g->batch, g->HL, g->WL, g->CL, kc, bw, bh, bn, 2))) return rc;
    p.num_taps = 16; p.chunks = g->CL / kc; p.a_scale = 2; p.BW = bw; p.BH = bh; p.BN = bn;
    p.tiles_w = g->WS / bw; p.tiles_h = g->HS / bh;
    for (int t = 0; t < 16; ++t) { p.a_dh[0][t] = (short)(t / 4 - 1); p.a_dw[0][t] = (short)(t % 4 - 1); }
    p.b_tap_stride = g->CL;
    if ((rc = encode_mat_map(&p.tmB, Wp_ls, g->CS, 16LL * g->CL, kc, g->CS))) return rc;
  }
  p.KC = kc; p.swz = umma_swizzle_for(kc * 2);
  p.N = n_slab; p.n_store = g->CS; p.n_slabs = g->CS / n_slab;
  p.out = S; p.mask = mask; p.bias = bias; p.act = act & ~GCCVAE_LAYOUT_FLAGS; p.out_f32 = out_f32;
  p.out_s2d = (act & GCCVAE_OUT_S2D) ? 1 : 0; p.mask_s2d = (act & GCCVAE_MASK_S2D) ? 1 : 0;
  GCC_REQUIRE(!p.out_s2d || (out_f32 == 0 && !dense), "ls_bf16: s2d output needs a bf16 spatial output");
  p.OH = g->HS; p.OW = g->WS; p.OC = g->CS; p.oys = p.oxs = 1;
  p.batch = g->batch;
  const int groups = (g->batch + p.BN - 1) / p.BN;
  return launch_tapgemm(p, groups, 1, (cudaStream_t)stream, "ls_bf16");
}

// L = act(scatter(S) W^T + b) (* mask>0): bf16 NHWC in/out, Wp = pack "sl" layout.
extern "C" int gccvae_sl_bf16(const gccvae_geom* g, const void* S, const void* Wp_sl, const float* bias, int act,
                              const void* mask, void* L, int out_f32, void* stream) {
  GCC_REQUIRE(g && S && Wp_sl && L, "sl_bf16: null pointer");
  const int kc = pick_kc(g->CS);
  GCC_REQUIRE(kc > 0, "sl_bf16: CS=%d unsupported (need 16, 32 or a multiple of 64)", g->CS);
  TapGemmParams p;
  memset(&p, 0, sizeof(p));
  int rc, phases;
  const bool dense = (g->HS == 1 && g->WS == 1 && g->pad == 0 && g->stride == 1);
  if (dense) {
    // [B, CS] x [CS, KH*KW*CL]: N = KH*KW*CL is tiled in slabs of <= 256 over blockIdx.y
    const int Nt = g->KH * g->KW * g->CL;
    const int nslab = Nt <= 256 ? Nt : (Nt % 256 == 0 ? 256 : (Nt % 128 == 0 ? 128 : 0));
    GCC_REQUIRE(nslab > 0 && nslab % 16 == 0, "sl_bf16(dense): N=%d unsupported", Nt);
    phases = 1;
    if ((rc = encode_act_map(&p.tmA, S, g->batch, 1, 1, g->CS, kc, 1, 1, 128, 1))) return rc;
    p.num_taps = 1; p.chunks = g->CS / kc; p.a_scale = 1; p.BW = 1; p.BH = 1; p.BN = 128; p.tiles_w = p.tiles_h = 1;
    if ((rc = encode_mat_map(&p.tmB, Wp_sl, Nt, g->CS, kc, nslab))) return rc;
    p.N = nslab; p.n_store = Nt; p.n_slabs = Nt / nslab;
    p.OH = 1; p.OW = 1; p.OC = Nt; p.oys = p.oxs = 1;
    p.bias_mod = g->CL;
  } else {
    GCC_REQUIRE(g->KH == 4 && g->KW == 4 && g->stride == 2 && g->pad == 1, "sl_bf16: only k4/s2/p1 or dense");
    int bw, bh, bn;
    GCC_REQUIRE(pick_tile(g->HS, g->WS, &bw, &bh, &bn) == 0, "sl_bf16: cannot tile %dx%d", g->HS, g->WS);
    const int rows_pad = (g->CL + 15) / 16 * 16;
    GCC_REQUIRE(rows_pad <= 256, "sl_bf16: CL too large");
    GCC_REQUIRE(g->CL % 16 == 0 || (g->CL == 3 && out_f32 == 2 && mask == nullptr),
                "sl_bf16: CL=%d must be a multiple of 16 (or 3 with the float4 image output)", g->CL);
    phases = 4;
    if ((rc = encode_act_map(&p.tmA, S, g->batch, g->HS, g->WS, g->CS, kc, bw, bh, bn, 1))) return rc;
    p.num_taps = 4; p.chunks = g->CS / kc; p.a_scale = 1; p.BW = bw; p.BH = bh; p.BN = bn;
    p.tiles_w = g->WS / bw; p.tiles_h = g->HS / bh;
    for (int z = 0; z < 4; ++z) {
      const int ph = z >> 1, pw = z & 1;
      for (int t = 0; t < 4; ++t) { p.a_dh[z][t] = (short)(ph - (t >> 1)); p.a_dw[z][t] = (short)(pw - (t & 1)); }
      p.b_row0[z] = z * rows_pad;
      p.oy0[z] = ph; p.ox0[z] = pw;
    }
    p.b_tap_stride = g->CS;
    if ((rc = encode_mat_map(&p.tmB, Wp_sl, 4LL * rows_pad, 4LL * g->CS, kc, rows_pad))) return rc;
    p.N = rows_pad; p.n_store = g->CL;
    p.OH = g->HL; p.OW = g->WL; p.OC = g->CL; p.oys = p.oxs = 2;
  }
  p.KC = kc; p.swz = umma_swizzle_for(kc * 2);
  p.out = L; p.mask = mask; p.bias = bias; p.act = act & ~GCCVAE_LAYOUT_FLAGS; p.out_f32 = out_f32;
  p.mask_s2d = (act & GCCVAE_MASK_S2D) ? 1 : 0;
  GCC_REQUIRE(!(act & GCCVAE_OUT_S2D), "sl_bf16: s2d output is not supported");
  p.batch = g->batch;
  const int groups = (g->batch + p.BN - 1) / p.BN;
  return launch_tapgemm(p, groups, phases, (cudaStream_t)stream, "sl_bf16");
}

extern "C" void gccvae_debug_set_timeline(long long* dev_buf) { g_timeline = dev_buf; }

extern "C" int gccvae_debug_tma4d(const void* src_bf16, int N, int H, int W, int C, int kc, int bw, int bh, int bn, int es,
                                  int c0, int c1, int c2, int c3, void* out, int out_bytes, void* stream) {
  CUtensorMap tm;
  if (int rc = encode_act_map(&tm, src_bf16, N, H, W, C, kc, bw, bh, bn, es)) return rc;
  const int bytes = kc * bw * bh * bn * 2;
  GCC_REQUIRE(out && out_bytes >= bytes && bytes <= 64 * 1024, "debug_tma4d: bad output size (%d needed)", bytes);
  GCC_CUDA(cudaFuncSetAttribute(tma_dump_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
  tma_dump_kernel<<<1, 128, bytes + 1024, (cudaStream_t)stream>>>(tm, c0, c1, c2, c3, bytes, (uint8_t*)out);
  GCC_CHECK_LAUNCH("debug_tma4d");
  return GCCVAE_OK;
}

// dW[kh,kw,cl,cs] (fp32, Keras layout) += wgrad; dW must be zeroed by the caller (accumulating entry).
static int wg_bf16_impl(const gccvae_geom* g, const void* L, const void* S, const gccvae_wg_out* out, int c4_rows,
                        void* stream) {
  GCC_REQUIRE(g && L && S && out && out->n_seg >= 1 && out->n_seg <= 2 && out->seg[0].dst, "wg_bf16: null pointer");
  const int CL = g->CL, CS = g->CS, taps = g->KH * g->KW;
  GCC_REQUIRE(CL == 32 || CL % 64 == 0, "wg_bf16: CL=%d unsupported (32 or a multiple of 64)", CL);
  GCC_REQUIRE(CS % 32 == 0 && CS <= 256, "wg_bf16: CS=%d unsupported (multiple of 32, <= 256)", CS);
  WgParams p;
  memset(&p, 0, sizeof(p));
  p.kcA = CL > 64 ? 64 : CL;
  p.blocks_per_tap = CL / p.kcA;
  p.blocks_per_mtile = 128 / p.kcA;
  p.taps = taps;
  p.c4_rows = c4_rows;
  p.kcB = (CS % 64 == 0) ? 64 : 32;
  p.b_loads = CS / p.kcB;
  p.swzA = umma_swizzle_for(p.kcA * 2);
  p.swzB = umma_swizzle_for(p.kcB * 2);
  int rc, bw, bh, bn, es;
  const bool dense = (g->HS == 1 && g->WS == 1 && g->pad == 0 && g->stride == 1);
  if (dense) {
    bw = 1; bh = 1; bn = 128; es = 1; p.a_scale = 1;
    for (int t = 0; t < taps; ++t) { p.a_dh[t] = (short)(t / g->KW); p.a_dw[t] = (short)(t % g->KW); }
  } else {
    GCC_REQUIRE(g->KH == 4 && g->KW == 4 && g->stride == 2 && g->pad == 1, "wg_bf16: only k4/s2/p1 or 1x1-spatial S");
    GCC_REQUIRE(pick_tile(g->HS, g->WS, &bw, &bh, &bn) == 0, "wg_bf16: cannot tile %dx%d", g->HS, g->WS);
    es = 2; p.a_scale = 2;
    for (int t = 0; t < 16; ++t) { p.a_dh[t] = (short)(t / 4 - 1); p.a_dw[t] = (short)(t % 4 - 1); }
  }
  if ((rc = encode_act_map(&p.tmA, L, g->batch, g->HL, g->WL, CL, p.kcA, bw, bh, bn, es))) return rc;
  if ((rc = encode_act_map(&p.tmB, S, g->batch, g->HS, g->WS, CS, p.kcB, bw, bh, bn, 1))) return rc;
  p.BW = bw; p.BH = bh; p.BN = bn; p.tiles_w = g->WS / bw; p.tiles_h = g->HS / bh;
  p.N = CS; p.out = *out;
  const int groups = (g->batch + bn - 1) / bn;
  p.tiles_total = groups * p.tiles_w * p.tiles_h;
  const int mtiles = (taps * p.blocks_per_tap + p.blocks_per_mtile - 1) / p.blocks_per_mtile;
  int splits = (148 * 2 + mtiles - 1) / mtiles;
  if (splits > p.tiles_total) splits = p.tiles_total;
  if (splits < 1) splits = 1;
  p.tiles_per_cta = (p.tiles_total + splits - 1) / splits;
  splits = (p.tiles_total + p.tiles_per_cta - 1) / p.tiles_per_cta;
  const int stage_bytes = 128 * 128 * 2 + 128 * CS * 2;
  int stages = (188 * 1024) / stage_bytes;
  if (stages > 4) stages = 4;
  if (stages > p.tiles_per_cta) stages = p.tiles_per_cta;
  if (stages < 1) stages = 1;
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + 1024 + 256 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    GCC_CUDA(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    attr_set = true;
  }
  dim3 grid(splits, mtiles, 1);
  p.timeline = g_timeline;
  GCC_CUDA(launch_pdl(wgrad_kernel, grid, TG_THREADS, smem, (cudaStream_t)stream, p));
  GCC_CHECK_LAUNCH("wg_bf16");
  return GCCVAE_OK;
}

extern "C" int gccvae_wg_bf16(const gccvae_geom* g, const void* L, const void* S, float* dW, void* stream) {
  GCC_REQUIRE(g && dW, "wg_bf16: null pointer");
  gccvae_wg_out o;
  memset(&o, 0, sizeof(o));
  o.n_seg = 1; o.m_valid = g->KH * g->KW * g->CL;
  o.seg[0].col0 = 0; o.seg[0].ncols = g->CS; o.seg[0].ld = g->CS; o.seg[0].dst = dW;
  return wg_bf16_impl(g, L, S, &o, 0, stream);
}

// D[M, N] += A^T B for row-major bf16 A [rows, M], B [rows, N] (M multiple of 64, N multiple of 32, <= 256);
// the result is scattered to 1-2 column segments (e.g. the two [256,45] head kernels).
extern "C" int gccvae_gemm_tn_bf16(long long rows, int M, int N, const void* A, const void* B, const gccvae_wg_out* out,
                                   void* stream) {
  GCC_REQUIRE(rows > 0 && rows < (1LL << 31), "gemm_tn: bad row count");
  gccvae_geom g = {(int)rows, 1, 1, M, 1, 1, N, 1, 1, 1, 0};
  return wg_bf16_impl(&g, A, B, out, 0, stream);
}

// out[c] += sum_r in[r,c] for a bf16 [rows, cols] tensor (out fp32, pre-zeroed by the caller)
extern "C" int gccvae_colsum_bf16(const void* in, long long rows, int cols, int n_valid, float* out, void* stream) {
  GCC_REQUIRE(in && out && rows > 0 && cols > 0 && cols % 2 == 0 && cols <= 256 && (256 % (cols / 2)) == 0,
              "colsum_bf16: bad args (cols=%d)", cols);
  if (n_valid <= 0 || n_valid > cols) n_valid = cols;
  // One CTA per 256 rows, not more: these kernels run on a side stream next to the dgrad chain, and spreading a
  // short tensor over more SMs made the whole step slower (1.505 vs 1.480 ms per pair, measured)
  long long ctas = (rows + 255) / 256;
  if (ctas > 148 * 4) ctas = 148 * 4;
  const int rpc = (int)((rows + ctas - 1) / ctas);
  ctas = (rows + rpc - 1) / rpc;
  if (cols % 8 == 0 && 256 % (cols / 8) == 0 && (uintptr_t)in % 16 == 0)
    GCC_CUDA(launch_aux(colsum_bf16_v8_kernel, dim3((int)ctas), dim3(256), 0, (cudaStream_t)stream,
                        (const __nv_bfloat16*)in, rows, cols, rpc, n_valid, out));
  else
    GCC_CUDA(launch_aux(colsum_bf16_kernel, dim3((int)ctas), dim3(256), 0, (cudaStream_t)stream,
                        (const __nv_bfloat16*)in, rows, cols, rpc, n_valid, out));
  GCC_CHECK_LAUNCH("colsum_bf16");
  return GCCVAE_OK;
}

// out[rows, N] = act(A[rows, K] * Wp[N, K]^T + bias) (* mask > 0): dense layers on the tensor cores.
// K multiple of 16/32/64, N multiple of 16; N > 256 is tiled in slabs.  bias[(n % bias_mod)] for n < bias_n.
extern "C" int gccvae_gemm_bf16(long long rows, int K, int N, const void* A, const void* Wp, const float* bias,
                                int bias_n, int bias_mod, int act, const void* mask, void* out, int out_f32,
                                void* stream) {
  GCC_REQUIRE(A && Wp && out && rows > 0 && rows < (1LL << 31), "gemm_bf16: bad args");
  const int kc = (K % 64 == 0) ? 64 : (K % 32 == 0 ? 32 : (K % 16 == 0 ? 16 : 0));
  GCC_REQUIRE(kc > 0, "gemm_bf16: K=%d must be a multiple of 16", K);
  GCC_REQUIRE(N % 16 == 0, "gemm_bf16: N=%d must be a multiple of 16", N);
  int nslab = N;
  const int m_tiles = (int)((rows + 127) / 128);
  if (N > 256 || (m_tiles < 74 && N > 64)) {
    nslab = (N % 64 == 0) ? 64 : ((N % 48 == 0) ? 48 : ((N % 32 == 0) ? 32 : 16));
    if (N > 256 && m_tiles >= 74) nslab = (N % 256 == 0) ? 256 : ((N % 128 == 0) ? 128 : nslab);
  }
  GCC_REQUIRE(N % nslab == 0, "gemm_bf16: cannot tile N=%d", N);
  TapGemmParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = encode_act_map(&p.tmA, A, (int)rows, 1, 1, K, kc, 1, 1, 128, 1))) return rc;
  if ((rc = encode_mat_map(&p.tmB, Wp, N, K, kc, nslab))) return rc;
  p.num_taps = 1; p.chunks = K / kc; p.a_scale = 1; p.BW = 1; p.BH = 1; p.BN = 128; p.tiles_w = p.tiles_h = 1;
  p.KC = kc; p.swz = umma_swizzle_for(kc * 2);
  p.N = nslab; p.n_store = N; p.n_slabs = N / nslab;
  p.out = out; p.mask = mask; p.bias = bias; p.act = act; p.out_f32 = out_f32;
  p.bias_n = bias ? (bias_n > 0 ? bias_n : N) : 0;
  p.bias_mod = bias_mod;
  p.OH = 1; p.OW = 1; p.OC = N; p.oys = p.oxs = 1;
  p.batch = (int)rows;
  return launch_tapgemm(p, m_tiles, 1, (cudaStream_t)stream, "gemm_bf16");
}

static bool halo_supported(const gccvae_geom* g, int* bw_out, int* bh_out) {
  if (!(g->KH == 4 && g->KW == 4 && g->stride == 2 && g->pad == 1)) return false;
  int bw, bh, bn;
  if (pick_tile(g->HS, g->WS, &bw, &bh, &bn) != 0) return false;
  const int rows_pad = (g->CL + 15) / 16 * 16;
  if (!(bn == 1 && bw == g->WS && (g->CS == 32 || g->CS == 64) && rows_pad <= 64)) return false;
  if (bw_out) { *bw_out = bw; *bh_out = bh; }
  return true;
}
extern "C" int gccvae_sl_halo_supported(const gccvae_geom* g) { return g && halo_supported(g, nullptr, nullptr) ? 1 : 0; }

// S -> L through the halo kernel (weights packed "sl9", gccvae_pack_jobs_bf16 kind 6).
extern "C" int gccvae_sl_halo_bf16(const gccvae_geom* g, const void* S, const void* Wp_sl9, const float* bias, int act,
                                   const void* mask, void* L, int out_f32, void* stream) {
  GCC_REQUIRE(g && S && Wp_sl9 && L, "sl_halo: null pointer");
  int bw = 0, bh = 0, rc;
  GCC_REQUIRE(halo_supported(g, &bw, &bh), "sl_halo: geometry not supported (use gccvae_sl_bf16)");
  const int rows_pad = (g->CL + 15) / 16 * 16;
  GCC_REQUIRE(g->CL % 16 == 0 || (g->CL == 3 && out_f32 == 2 && mask == nullptr),
              "sl_halo: CL=%d must be a multiple of 16 (or 3 with the float4 image output)", g->CL);
  SlHaloParams hp;
  memset(&hp, 0, sizeof(hp));
  EncodeTiledFn enc = get_encode();
  GCC_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled unavailable");
  {
    cuuint64_t dims[4] = {(cuuint64_t)g->CS, (cuuint64_t)g->WS, (cuuint64_t)g->HS, (cuuint64_t)g->batch};
    cuuint64_t strides[3] = {(cuuint64_t)g->CS * 2, (cuuint64_t)g->WS * g->CS * 2, (cuuint64_t)g->HS * g->WS * g->CS * 2};
    cuuint32_t box[4] = {(cuuint32_t)g->CS, (cuuint32_t)bw, (cuuint32_t)(bh + 2), 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&hp.tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(S), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, tma_swizzle_for(g->CS * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    GCC_REQUIRE(r == CUDA_SUCCESS, "sl_halo: cuTensorMapEncodeTiled failed: %d", (int)r);
  }
  if ((rc = encode_mat_map(&hp.tmB, Wp_sl9, 9LL * 4 * rows_pad, g->CS, g->CS, 4 * rows_pad))) return rc;
  hp.C = g->CS; hp.BW = bw; hp.BH = bh; hp.tiles_h = g->HS / bh;
  hp.N = rows_pad; hp.n_store = g->CL; hp.swz = umma_swizzle_for(g->CS * 2);
  hp.out = L; hp.mask = mask; hp.bias = bias; hp.bias_n = bias ? g->CL : 0; hp.act = act & ~GCCVAE_LAYOUT_FLAGS;
  hp.out_f32 = out_f32; hp.mask_s2d = (act & GCCVAE_MASK_S2D) ? 1 : 0;
  GCC_REQUIRE(!(act & GCCVAE_OUT_S2D), "sl_halo: s2d output is not supported");
  hp.OH = g->HL; hp.OW = g->WL; hp.OC = g->CL; hp.batch = g->batch;
  hp.total_tiles = g->batch * hp.tiles_h;
  hp.timeline = g_timeline;
  const int rowb = g->CS * 2, a_stage = 3 * (bh + 2) * bw * rowb, b_bytes = (9 * 4 * rows_pad * rowb + 1023) & ~1023;
  int stages = (196 * 1024 - b_bytes - 5120) / a_stage;
  if (stages > 5) stages = 5;
  GCC_REQUIRE(stages >= 2, "sl_halo: shared memory");
  hp.stages = stages;
  const size_t smem = (size_t)b_bytes + (size_t)stages * a_stage + 1024 + 3072;
  static bool attr_set = false;
  if (!attr_set) {
    GCC_CUDA(cudaFuncSetAttribute(sl_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    attr_set = true;
  }
  const int ctas = hp.total_tiles < 148 ? hp.total_tiles : 148;
  GCC_CUDA(launch_pdl(sl_halo_kernel, dim3(ctas, 1, 1), HALO_THREADS, smem, (cudaStream_t)stream, hp));
  GCC_CHECK_LAUNCH("sl_halo_bf16");
  return GCCVAE_OK;
}


// ---- x2 (space-to-depth) end layers ----------------------------------------------------------------------
// x [B,64,64,3] (fp32 in [0,1], or uint8 0..255 which is divided by 255 on the fly) -> X2 [B,33,33,16] bf16 and, for
// uint8 images, optionally XB [B,33,33,16] uint8: the raw bytes of every block (gccvae_convt_recon_bf16 with x_u8 = 2)
extern "C" int gccvae_prep_x2_bf16(const void* x, int x_u8, int batch, void* X2, void* XB, void* stream) {
  GCC_REQUIRE(x && X2 && batch > 0, "prep_x2: bad args");
  GCC_REQUIRE(XB == nullptr || x_u8, "prep_x2: the raw-byte blocks exist for uint8 images only");
  GCC_REQUIRE(((uintptr_t)X2 % 16) == 0 && ((uintptr_t)XB % 16) == 0, "prep_x2: outputs must be 16-byte aligned");
  const long long total = (long long)batch * 33 * 33;
  long long ctas = (total + 255) / 256;
  if (ctas > 148 * 16) ctas = 148 * 16;
  if (int rc2 = ensure_u8lut()) return rc2;
  if (x_u8 && (uintptr_t)x % 16 == 0)
    GCC_CUDA(launch_aux(prep_x2_u8_staged_kernel, dim3(batch < 148 * 8 ? batch : 148 * 8), dim3(256), 0, (cudaStream_t)stream,
                        (const uint8_t*)x, batch, (uint4*)X2, (uint4*)XB));
  else if (x_u8)
    GCC_CUDA(launch_aux(prep_x2_kernel<uint8_t>, dim3((int)ctas), dim3(256), 0, (cudaStream_t)stream, (const uint8_t*)x,
                        total, (uint4*)X2, (uint4*)XB));
  else
    GCC_CUDA(launch_aux(prep_x2_kernel<float>, dim3((int)ctas), dim3(256), 0, (cudaStream_t)stream, (const float*)x, total,
                        (uint4*)X2, (uint4*)nullptr));
  GCC_CHECK_LAUNCH("prep_x2");
  return GCCVAE_OK;
}

// out[n, y, x, :] = act( sum_{a,b in {0,1}} in2[n, y+a, x+b, :] . Wp[:, (a,b), :] + bias ) (* mask > 0)
// in2 = [B, HB, WB, CB] bf16 blocks, out = [B, HB-1, WB-1, CS] bf16 NHWC, Wp = [CS][4][CB] bf16 (pack kind 7).
extern "C" int gccvae_tap4_ls_bf16(int batch, int HB, int WB, int CB, const void* in2, const void* Wp, int CS,
                                   const float* bias, int act, const void* mask, void* out, void* stream) {
  GCC_REQUIRE(in2 && Wp && out && batch > 0, "tap4_ls: null pointer");
  const int kc = CB >= 64 ? 64 : CB;
  GCC_REQUIRE((kc == 16 || kc == 32 || kc == 64) && CB % kc == 0, "tap4_ls: CB=%d unsupported", CB);
  GCC_REQUIRE(CS % 16 == 0 && CS <= 256, "tap4_ls: CS=%d must be a multiple of 16, <= 256", CS);
  const int HS = HB - 1, WS = WB - 1;
  int bw, bh, bn, rc;
  GCC_REQUIRE(pick_tile(HS, WS, &bw, &bh, &bn) == 0, "tap4_ls: cannot tile %dx%d", HS, WS);
  TapGemmParams p;
  memset(&p, 0, sizeof(p));
  // halo2 form (GCCVAE_TAP_HALO): full-width tiles of one image, 128-byte operand rows, the row shift a multiple of the
  // 1 KB swizzle atom, the box of (bh + 1) x bw rows within TMA's limits
  const bool halo2 = (act & GCCVAE_TAP_HALO) && bn == 1 && bw == WS && kc == 64 && (bw * kc * 2) % 1024 == 0 &&
                     (size_t)(bh + 1) * bw * kc * 2 <= 24 * 1024 && CS * kc * 2 % 1024 == 0;
  if ((rc = encode_act_map(&p.tmA, in2, batch, HB, WB, CB, kc, bw, halo2 ? bh + 1 : bh, bn, 1))) return rc;
  if ((rc = encode_mat_map(&p.tmB, Wp, CS, 4LL * CB, kc, CS))) return rc;
  p.chunks = CB / kc; p.a_scale = 1; p.BW = bw; p.BH = bh; p.BN = bn;
  p.tiles_w = WS / bw; p.tiles_h = HS / bh;
  if (halo2) {
    p.halo2 = 1; p.num_taps = 2; p.a_box_rows = (bh + 1) * bw;
    for (int t = 0; t < 2; ++t) { p.a_dh[0][t] = 0; p.a_dw[0][t] = (short)t; }
  } else {
    p.num_taps = 4;
    for (int t = 0; t < 4; ++t) { p.a_dh[0][t] = (short)(t >> 1); p.a_dw[0][t] = (short)(t & 1); }
  }
  p.b_tap_stride = CB;
  p.KC = kc; p.swz = umma_swizzle_for(kc * 2);
  p.N = CS; p.n_store = CS; p.n_slabs = 1;
  p.out = out; p.mask = mask; p.bias = bias; p.act = act & ~GCCVAE_LAYOUT_FLAGS; p.out_f32 = 0;
  p.out_s2d = (act & GCCVAE_OUT_S2D) ? 1 : 0; p.mask_s2d = (act & GCCVAE_MASK_S2D) ? 1 : 0;
  p.OH = HS; p.OW = WS; p.OC = CS; p.oys = p.oxs = 1;
  p.batch = batch;
  const int groups = (batch + bn - 1) / bn;
  return launch_tapgemm(p, groups, 1, (cudaStream_t)stream, "tap4_ls");
}

// dW[(kh,kw,c<3), cs] (fp32, Keras layout) += sum_pix gather4(in2)[pix, (a,b,dy,dx,c4)] * S[pix, cs]
// in2 = [B,33,33,16] bf16 x2 blocks of a 3-channel 64x64 tensor, S = [B,32,32,CS] bf16.
// db (optional, blocks written by gccvae_prep_x2_bf16 only - element 15 of every block is 1.0): db[cs] += sum_pix S[pix, cs].
extern "C" int gccvae_tap4_wg_bf16(int batch, const void* in2, const void* S, int CS, float* dW, float* db, void* stream) {
  GCC_REQUIRE(in2 && S && dW && batch > 0, "tap4_wg: null pointer");
  GCC_REQUIRE(CS % 32 == 0 && CS <= 256, "tap4_wg: CS=%d unsupported (multiple of 32, <= 256)", CS);
  WgParams p;
  memset(&p, 0, sizeof(p));
  // A tile built by the (otherwise idle) epilogue warps: one 128-byte row per pixel, SWIZZLE_128B, which is an
  // MN-major operand with M = 64 (a,b,dy,dx,c4); the instruction's rows 64..127 come from the unused second slab
  // Only ONE 16 KB slab per stage is built and reserved: the second slab the M = 128 instruction reads (LBO = 16 KB
  // further on: the stage's B tile and the next stage, or the slack behind the last stage) feeds accumulator rows
  // 64..127, which nobody reads.  24 KB stages instead of 40: four pipeline stages in the same 100 KB per CTA - the
  // kernel is bound by the round trip of a stage (profiles/r02_timeline_wgrad.txt), so depth is what it needs.
  p.in2 = (const uint4*)in2;
  p.kcA = 64; p.blocks_per_tap = 1; p.blocks_per_mtile = 1; p.taps = 1; p.c4_rows = 2;
  p.kcB = (CS % 64 == 0) ? 64 : 32;
  p.b_loads = CS / p.kcB;
  p.swzA = umma_swizzle_for(p.kcA * 2);
  p.swzB = umma_swizzle_for(p.kcB * 2);
  int rc, bw, bh, bn;
  GCC_REQUIRE(pick_tile(32, 32, &bw, &bh, &bn) == 0, "tap4_wg: tile");
  p.a_scale = 1;
  for (int t = 0; t < 4; ++t) { p.a_dh[t] = (short)(t >> 1); p.a_dw[t] = (short)(t & 1); }
  if ((rc = encode_act_map(&p.tmA, in2, batch, 33, 33, 16, 16, bw, bh, bn, 1))) return rc;   // prefetched, never loaded
  if ((rc = encode_act_map(&p.tmB, S, batch, 32, 32, CS, p.kcB, bw, bh, bn, 1))) return rc;
  p.BW = bw; p.BH = bh; p.BN = bn; p.tiles_w = 32 / bw; p.tiles_h = 32 / bh;
  p.N = CS;
  p.out.n_seg = 1; p.out.m_valid = 64;
  p.out.seg[0].col0 = 0; p.out.seg[0].ncols = CS; p.out.seg[0].ld = CS; p.out.seg[0].dst = dW;
  p.ones_db = db;
  const int groups = (batch + bn - 1) / bn;
  p.tiles_total = groups * p.tiles_w * p.tiles_h;
  int splits = 148 * WG_PER_SM;
  if (splits > p.tiles_total) splits = p.tiles_total;
  p.tiles_per_cta = (p.tiles_total + splits - 1) / splits;
  splits = (p.tiles_total + p.tiles_per_cta - 1) / p.tiles_per_cta;
  const int stage_bytes = 128 * 128 * p.blocks_per_mtile + 128 * CS * 2;
  int stages = (WG_SMEM_KB * 1024) / stage_bytes;   // two CTAs per SM
  if (stages > 8) stages = 8;
  if (stages > p.tiles_per_cta) stages = p.tiles_per_cta;
  if (stages < 1) stages = 1;
  p.stages = stages;
  size_t smem = (size_t)stages * stage_bytes + 1024 + 256 + 1024;
  // the unread second slab of the LAST stage's A tile must still lie inside the allocation (layout: [A stages][B stages])
  if (smem < (size_t)(stages + 1) * 16384 + 1024) smem = (size_t)(stages + 1) * 16384 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    GCC_CUDA(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    attr_set = true;
  }
  p.timeline = g_timeline;
  GCC_CUDA(launch_pdl(wgrad_kernel, dim3(splits, 1, 1), TG_THREADS, smem, (cudaStream_t)stream, p));
  GCC_CHECK_LAUNCH("tap4_wg");
  return GCCVAE_OK;
}

extern "C" int gccvae_fill_f32(float* p, long long n, float v, void* stream) {
  GCC_REQUIRE(p && n > 0 && n < (1LL << 31), "fill_f32: bad args");
  fill_kernel<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p, (int)n, v);
  GCC_CHECK_LAUNCH("fill_f32");
  return GCCVAE_OK;
}

// Launch shape of every conv5t kind: more resident CTAs = more tiles in flight (the per-tile chain TMA -> MMA -> epilogue
// is latency-bound).  Limits: registers x 192 threads, 64 TMEM columns and the shared memory of convt_smem per CTA.
// 4 CTAs per SM beat 2 and 3 in the training step (profiles/r01d_ab_log.txt).
constexpr int CT_PER_SM = 4, CT_STAGES = 3;
constexpr int convt_smem(bool raw_x) { return 4096 + CT_STAGES * (CTR_A_STAGE + (raw_x ? CTR_X_BYTES : 0)) + 1024 + 2048; }
static_assert(CT_PER_SM * (convt_smem(true) + 1024) <= 227 * 1024, "conv5t: CT_PER_SM CTAs do not fit in shared memory");

// The common launch of conv5t over `rows` decoded rows of g4 [rows,32,32,32] bf16 (Wp8 = pack kind 8): the tensor maps,
// the launch shape, and the (out, x_form) instantiation; the caller fills the rest of p.
static int launch_convt(int out, int rows, const void* g4, const void* Wp8, CtParams& p, int x_form, cudaStream_t st) {
  static const char* const name[5] = {"convt_recon", "convt_ll", "convt_image", "convt_image", "convt_complete"};
  EncodeTiledFn enc = get_encode();
  GCC_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled unavailable");
  {
    cuuint64_t dims[4] = {32, 32, 32, (cuuint64_t)rows};
    cuuint64_t strides[3] = {64, 32 * 64, 32 * 32 * 64};
    cuuint32_t box[4] = {32, 33, 6, 1};   // 6 image rows x (zero column + 32 pixels): CTR_BOX_ROWS rows of 64 bytes
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&p.tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(g4), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    GCC_REQUIRE(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed: %d", name[out], (int)r);
  }
  int rc;
  if ((rc = encode_mat_map(&p.tmB, Wp8, 16, 128, 32, 16))) return rc;
  if ((out == RECON || out == LL) && (rc = ensure_u8lut())) return rc;
  p.total_tiles = rows * 9;
  p.stages = CT_STAGES;
  const size_t smem = convt_smem((out == RECON || out == LL) && x_form == 2);
  using Kernel = void (*)(const CtParams);
  static const Kernel kernels[5][3] = {{convt_kernel<RECON, 0>, convt_kernel<RECON, 1>, convt_kernel<RECON, 2>},
                                       {convt_kernel<LL, 0>, convt_kernel<LL, 1>, convt_kernel<LL, 2>},
                                       {convt_kernel<IMAGE_F32, 0>, nullptr, nullptr},
                                       {convt_kernel<IMAGE_U8, 0>, nullptr, nullptr},
                                       {convt_kernel<COMPLETE, 0>, nullptr, nullptr}};
  static bool attr_set[5][3] = {};
  const Kernel kernel = kernels[out][x_form];
  if (!attr_set[out][x_form]) {
    GCC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[out][x_form] = true;
  }
  int ctas = p.total_tiles < 148 * CT_PER_SM ? p.total_tiles : 148 * CT_PER_SM;
  {
    const int per_cta = (p.total_tiles + ctas - 1) / ctas;
    ctas = (p.total_tiles + per_cta - 1) / per_cta;
  }
  GCC_CUDA(launch_pdl(kernel, dim3(ctas, 1, 1), TG_THREADS, smem, st, p));
  GCC_CHECK_LAUNCH(name[out]);
  return GCCVAE_OK;
}

// Fused conv5t forward (Conv2DTranspose 32 -> 3, k4, s2, same) + sigmoid + Laplace log-likelihood + dLoss/dlogit.
//   g4 [B,32,32,32] bf16, Wp8 = pack kind 8 ([16][4][32] bf16), bias [3], x [B,64,64,3] fp32 or uint8.
//   log_pxz[b] = -|x - xhat|_1 - 12288 ln 2.  coef != NULL: D2 [B,33,33,16] bf16 = coef[b] sign(x - xhat) xhat (1 - xhat)
//   in x2 block form and db[3] += its sums.  xhat (optional): the reconstruction, fp32 [B,64,64,3].
extern "C" int gccvae_convt_recon_bf16(int batch, const void* g4, const void* Wp8, const float* bias, const void* x,
                                       int x_u8, const float* coef, float* log_pxz, void* D2, float* xhat, float* db,
                                       int log_pxz_ready, void* stream) {
  GCC_REQUIRE(g4 && Wp8 && bias && x && log_pxz && batch > 0, "convt_recon: null pointer");
  GCC_REQUIRE((coef == nullptr) == (D2 == nullptr), "convt_recon: coef and D2 go together");
  GCC_REQUIRE(x_u8 >= 0 && x_u8 <= 2 && (x_u8 != 2 || (uintptr_t)x % 16 == 0), "convt_recon: x_u8 = %d (0 fp32 image, 1 uint8 image, 2 raw-byte blocks, 16-byte aligned)", x_u8);
  cudaStream_t st = (cudaStream_t)stream;
  CtParams p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.x_u8 = x_u8; p.bias = bias; p.coef = coef; p.log_pxz = log_pxz; p.D2 = (uint4*)D2; p.xhat = xhat; p.db = db;
  p.batch = batch;
  p.timeline = g_timeline;
  if (!log_pxz_ready) {   // otherwise the caller pre-set log_pxz[b] = -12288 ln 2 (gccvae_fill_f32) off the critical path
    fill_kernel<<<(batch + 255) / 256, 256, 0, st>>>(log_pxz, batch, (float)(-12288.0 * 0.6931471805599453));
    GCC_CHECK_LAUNCH("recon_fill");
  }
  return launch_convt(RECON, batch, g4, Wp8, p, x_u8, st);
}

// conv5t forward + sigmoid into the image (generation path): g4 [B,32,32,32] bf16, Wp8 = pack kind 8, bias [3],
// out [B,64,64,3] fp32 (out_u8 = 0) or uint8 min(255, rint(255 xhat)) (out_u8 = 1).
extern "C" int gccvae_convt_image_bf16(int batch, const void* g4, const void* Wp8, const float* bias, void* out,
                                       int out_u8, void* stream) {
  GCC_REQUIRE(g4 && Wp8 && bias && out, "convt_image: null pointer");
  GCC_REQUIRE(batch > 0 && batch <= (1 << 26), "convt_image: bad batch %d", batch);
  GCC_REQUIRE(out_u8 == 0 || out_u8 == 1, "convt_image: out_u8 = %d (0 fp32, 1 uint8)", out_u8);
  GCC_REQUIRE((uintptr_t)out % 16 == 0 && (uintptr_t)g4 % 16 == 0, "convt_image: out and g4 must be 16-byte aligned");
  CtParams p;
  memset(&p, 0, sizeof(p));
  p.bias = bias; p.out = out; p.batch = batch;
  return launch_convt(out_u8 ? IMAGE_U8 : IMAGE_F32, batch, g4, Wp8, p, 0, (cudaStream_t)stream);
}

// conv5t forward + sigmoid written into the unobserved pixels of the x2 blocks X2 [B,33,33,16] bf16, in place (one
// iteration of image completion): mask_blocks [B,33,33] uint8, bit dy * 2 + dx set = pixel (2i-1+dy, 2j-1+dx) observed.
extern "C" int gccvae_convt_complete_bf16(int batch, const void* g4, const void* Wp8, const float* bias,
                                          const void* mask_blocks, void* X2, void* stream) {
  GCC_REQUIRE(g4 && Wp8 && bias && mask_blocks && X2, "convt_complete: null pointer");
  GCC_REQUIRE(batch > 0 && batch <= (1 << 26), "convt_complete: bad batch %d", batch);
  GCC_REQUIRE((uintptr_t)X2 % 16 == 0 && (uintptr_t)g4 % 16 == 0, "convt_complete: X2 and g4 must be 16-byte aligned");
  CtParams p;
  memset(&p, 0, sizeof(p));
  p.bias = bias; p.out = X2; p.mask = (const uint8_t*)mask_blocks; p.batch = batch;
  return launch_convt(COMPLETE, batch, g4, Wp8, p, 0, (cudaStream_t)stream);
}

// conv5t forward + sigmoid + Laplace log-likelihood of `rows` decoded rows, row r against source image r / kc
// (importance-weighted likelihood): log_pxz[r] (pre-set to -12288 ln 2) += -|x - xhat|_1.
extern "C" int gccvae_convt_ll_bf16(int rows, int kc, const void* g4, const void* Wp8, const float* bias, const void* x,
                                    int x_u8, float* log_pxz, void* stream) {
  GCC_REQUIRE(g4 && Wp8 && bias && x && log_pxz, "convt_ll: null pointer");
  GCC_REQUIRE(rows > 0 && rows <= (1 << 26) && kc >= 1 && rows % kc == 0, "convt_ll: bad rows %d / kc %d", rows, kc);
  GCC_REQUIRE(x_u8 >= 0 && x_u8 <= 2 && (x_u8 != 2 || (uintptr_t)x % 16 == 0),
              "convt_ll: x_u8 = %d (0 fp32 image, 1 uint8 image, 2 raw-byte blocks, 16-byte aligned)", x_u8);
  GCC_REQUIRE((uintptr_t)g4 % 16 == 0, "convt_ll: g4 must be 16-byte aligned");
  CtParams p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.x_u8 = x_u8; p.bias = bias; p.log_pxz = log_pxz; p.batch = rows; p.kc = kc;
  return launch_convt(LL, rows, g4, Wp8, p, x_u8, (cudaStream_t)stream);
}


// conv1 forward / conv5t dgrad from x2 blocks with thread-built im2col tiles (see c3conv_kernel):
// out[B,32,32,CS] = act(conv_k4s2p1(image of in2) + bias) (* mask > 0), Wp = pack kind 7 ([CS][64] bf16), CS in {32, 64}.
extern "C" int gccvae_c3conv_bf16(int batch, const void* in2, const void* Wp, int CS, const float* bias, int act,
                                  const void* mask, void* out, void* stream) {
  GCC_REQUIRE(in2 && Wp && out && batch > 0, "c3conv: null pointer");
  GCC_REQUIRE(CS == 32 || CS == 64, "c3conv: CS=%d unsupported (32 or 64)", CS);
  GCC_REQUIRE(bias == nullptr || ((uintptr_t)bias % 16) == 0, "c3conv: bias must be 16-byte aligned");
  C3Params p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = encode_mat_map(&p.tmB, Wp, CS, 64, 64, CS))) return rc;
  p.in2 = (const uint4*)in2; p.out = out; p.mask = mask; p.bias = bias; p.act = act & ~GCCVAE_LAYOUT_FLAGS; p.N = CS;
  p.batch = batch; p.out_s2d = (act & GCCVAE_OUT_S2D) ? 1 : 0;
  GCC_REQUIRE(!(act & GCCVAE_MASK_S2D), "c3conv: s2d mask is not supported");
  p.total_tiles = batch * 8;
  p.timeline = g_timeline;
  // __launch_bounds__(288, 2): no register spills in the epilogue.  TMEM: 2 CTAs x 4 accumulator stages x <= 64 columns
  constexpr int per_sm = 2;
  int stages = (200 * 1024 / per_sm - 8192 - 3072) / (128 * 128);
  if (stages > 6) stages = 6;
  GCC_REQUIRE(stages >= 2, "c3conv: shared memory");
  p.stages = stages;
  const size_t smem = 8192 + (size_t)stages * 128 * 128 + 1024 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    GCC_CUDA(cudaFuncSetAttribute(c3conv_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    GCC_CUDA(cudaFuncSetAttribute(c3conv_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    attr_set = true;
  }
  int ctas = p.total_tiles < 148 * per_sm ? p.total_tiles : 148 * per_sm;
  {
    const int per_cta = (p.total_tiles + ctas - 1) / ctas;
    ctas = (p.total_tiles + per_cta - 1) / per_cta;
  }
  if (CS == 32) GCC_CUDA(launch_pdl(c3conv_kernel<2>, dim3(ctas, 1, 1), C3_THREADS, smem, (cudaStream_t)stream, p));
  else GCC_CUDA(launch_pdl(c3conv_kernel<4>, dim3(ctas, 1, 1), C3_THREADS, smem, (cudaStream_t)stream, p));
  GCC_CHECK_LAUNCH("c3conv");
  return GCCVAE_OK;
}


// dW[kh,kw,cl,cs] (fp32, Keras layout) += gather(L)^T S for a k4/s2/p1 layer whose L operand is stored in s2d block
// form in2 = [B, HL/2+1, WL/2+1, 4 CL] bf16; S = [B, HS, WS, CS] bf16 NHWC (HS = HL/2).  CL in {32, 64}.
extern "C" int gccvae_wg_s2d_bf16(int batch, int HS, int WS, int CL, const void* in2, const void* S, int CS, float* dW,
                                  void* stream) {
  GCC_REQUIRE(in2 && S && dW && batch > 0, "wg_s2d: null pointer");
  GCC_REQUIRE(CL == 16 || CL == 32 || CL == 64, "wg_s2d: CL=%d unsupported", CL);
  GCC_REQUIRE(CS % 32 == 0 && CS <= 256, "wg_s2d: CS=%d unsupported (multiple of 32, <= 256)", CS);
  WgParams p;
  memset(&p, 0, sizeof(p));
  const int CB = 4 * CL;
  p.kcA = 64; p.blocks_per_tap = CB / 64; p.blocks_per_mtile = 2; p.taps = 4; p.c4_rows = 3; p.s2d_cl = CL;
  p.kcB = (CS % 64 == 0) ? 64 : 32;
  p.b_loads = CS / p.kcB;
  p.swzA = umma_swizzle_for(p.kcA * 2);
  p.swzB = umma_swizzle_for(p.kcB * 2);
  int rc, bw, bh, bn;
  GCC_REQUIRE(pick_tile(HS, WS, &bw, &bh, &bn) == 0, "wg_s2d: cannot tile %dx%d", HS, WS);
  p.a_scale = 1;
  for (int t = 0; t < 4; ++t) { p.a_dh[t] = (short)(t >> 1); p.a_dw[t] = (short)(t & 1); }
  if ((rc = encode_act_map(&p.tmA, in2, batch, HS + 1, WS + 1, CB, p.kcA, bw, bh, bn, 1))) return rc;
  if ((rc = encode_act_map(&p.tmB, S, batch, HS, WS, CS, p.kcB, bw, bh, bn, 1))) return rc;
  p.BW = bw; p.BH = bh; p.BN = bn; p.tiles_w = WS / bw; p.tiles_h = HS / bh;
  p.N = CS;
  p.out.n_seg = 1; p.out.m_valid = 16 * CL;
  p.out.seg[0].col0 = 0; p.out.seg[0].ncols = CS; p.out.seg[0].ld = CS; p.out.seg[0].dst = dW;
  const int groups = (batch + bn - 1) / bn;
  p.tiles_total = groups * p.tiles_w * p.tiles_h;
  const int mtiles = (16 * CL) / 128;
  int splits = (148 * WG_PER_SM + mtiles - 1) / mtiles;
  if (splits > p.tiles_total) splits = p.tiles_total;
  if (splits < 1) splits = 1;
  p.tiles_per_cta = (p.tiles_total + splits - 1) / splits;
  splits = (p.tiles_total + p.tiles_per_cta - 1) / p.tiles_per_cta;
  const int stage_bytes = 128 * 128 * 2 + 128 * CS * 2;
  int stages = (WG_SMEM_KB * 1024) / stage_bytes;   // two CTAs per SM
  if (stages > 4) stages = 4;
  if (stages > p.tiles_per_cta) stages = p.tiles_per_cta;
  if (stages < 1) stages = 1;
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + 1024 + 256 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    GCC_CUDA(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    attr_set = true;
  }
  p.timeline = g_timeline;
  GCC_CUDA(launch_pdl(wgrad_kernel, dim3(splits, mtiles, 1), TG_THREADS, smem, (cudaStream_t)stream, p));
  GCC_CHECK_LAUNCH("wg_s2d");
  return GCCVAE_OK;
}

extern "C" size_t gccvae_packed_weight_elems(const gccvae_geom* g, int which) {
  if (!g) return 0;
  const int taps = g->KH * g->KW;
  if (which == 2) return (size_t)9 * 4 * ((g->CL + 15) / 16 * 16) * g->CS;                 // sl9 (halo kernel)
  if (which == 0) return (size_t)((g->CS + 15) / 16 * 16) * taps * g->CL;                 // ls
  if (g->HS == 1 && g->WS == 1) return (size_t)taps * g->CL * g->CS;                        // sl dense
  return (size_t)4 * ((g->CL + 15) / 16 * 16) * 4 * g->CS;                                  // sl phases
}

extern "C" int gccvae_pack_weights_bf16(const gccvae_geom* g, const float* W, void* Wp_ls, void* Wp_sl, void* stream) {
  GCC_REQUIRE(g && W, "pack_weights: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int taps = g->KH * g->KW;
  if (Wp_ls) {
    const int rows_pad = (g->CS + 15) / 16 * 16;
    const long long n = (long long)rows_pad * taps * g->CL;
    pack_ls_kernel<<<(int)((n + 255) / 256 > 1184 ? 1184 : (n + 255) / 256), 256, 0, st>>>(W, taps, g->CL, g->CS,
                                                                                         rows_pad, (__nv_bfloat16*)Wp_ls);
    GCC_CHECK_LAUNCH("pack_ls");
  }
  if (Wp_sl) {
    if (g->HS == 1 && g->WS == 1) {
      const long long n = (long long)taps * g->CL * g->CS;
      cast_bf16_kernel<<<(int)((n + 255) / 256 > 1184 ? 1184 : (n + 255) / 256), 256, 0, st>>>(W, n,
                                                                                             (__nv_bfloat16*)Wp_sl);
      GCC_CHECK_LAUNCH("pack_sl_dense");
    } else {
      GCC_REQUIRE(g->KH == 4 && g->KW == 4 && g->stride == 2 && g->pad == 1, "pack_weights: sl needs k4/s2/p1");
      const int rows_pad = (g->CL + 15) / 16 * 16;
      const long long n = 4LL * rows_pad * 4 * g->CS;
      pack_sl2_kernel<<<(int)((n + 255) / 256 > 1184 ? 1184 : (n + 255) / 256), 256, 0, st>>>(W, g->CL, g->CS, rows_pad,
                                                                                            (__nv_bfloat16*)Wp_sl);
      GCC_CHECK_LAUNCH("pack_sl2");
    }
  }
  return GCCVAE_OK;
}

extern "C" int gccvae_pack_jobs_bf16(const gccvae_pack_job* jobs, int n_jobs, void* stream) {
  GCC_REQUIRE(jobs && n_jobs > 0 && n_jobs <= 48, "pack_jobs: 1..48 jobs");
  PackJobs pj;
  memset(&pj, 0, sizeof(pj));
  for (int i = 0; i < n_jobs; ++i) {
    GCC_REQUIRE(jobs[i].W && jobs[i].out && jobs[i].kind >= 0 && jobs[i].kind <= 9, "pack_jobs: bad job %d", i);
    pj.j[i] = jobs[i];
  }
  GCC_CUDA(launch_aux(pack_jobs_kernel, dim3(64, n_jobs, 1), dim3(256), 0, (cudaStream_t)stream, pj));
  GCC_CHECK_LAUNCH("pack_jobs");
  return GCCVAE_OK;
}

extern "C" int gccvae_cast_f32_to_bf16(const float* in, long long n, void* out, void* stream) {
  GCC_REQUIRE(in && out && n > 0, "cast: bad args");
  cast_bf16_kernel<<<(int)((n + 255) / 256 > 2368 ? 2368 : (n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      in, n, (__nv_bfloat16*)out);
  GCC_CHECK_LAUNCH("cast_bf16");
  return GCCVAE_OK;
}
extern "C" int gccvae_cast_bf16_to_f32(const void* in, long long n, float* out, void* stream) {
  GCC_REQUIRE(in && out && n > 0, "cast: bad args");
  cast_f32_kernel<<<(int)((n + 255) / 256 > 2368 ? 2368 : (n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)in, n, out);
  GCC_CHECK_LAUNCH("cast_f32");
  return GCCVAE_OK;
}
