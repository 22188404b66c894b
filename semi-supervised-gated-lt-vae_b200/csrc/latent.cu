// Fused latent kernels of the Gated-CCVAE ELBO step (forward + backward) and the per-step gate.
//
// Reference math (all fp32): gated_ccvae.py:62-64,90-93,102-111 (samplers), :167-182 (K-sample
// log q(y|x)), :187-218 / :237-268,280-287 (latent part of unsup/sup loss); networks.py:17-18,
// 33-34 (posterior heads' activations), :72-74,83-86 (gated classifier), :104-106,118-127 (gated
// conditional prior); utils.py:108-119 (Normal KL); TFP Bernoulli.log_prob / .sample.
//
// Mapping: one warp per image (warps stride over the batch).  The 45 latent dims, the 18 labels
// and the 18 classify dims are spread over lanes; the K importance samples are spread over lanes
// too (lane l owns k = l, l+32, ...), with an online log-sum-exp joined by shuffles.  The gated
// 18x18 products shared by the whole batch live in shared memory (written once per step by
// gate_fwd into `gate_ws`).  HBM traffic per image: 2x[45] heads + (fixed-noise mode only)
// eps[45] + eps_k[K,18]; outputs 3x[45] + 6 scalars + [18] logits.
#include <cuda_bf16.h>

#include "common.cuh"
#include "latent_math.cuh"
#include "tc_common.cuh"

namespace gccvae {

// ---------------------------------------------------------------------------------------------
// gate forward: c = relaxed-Bernoulli(mu, T) and everything derived from it.  One CTA.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(352) gate_fwd_kernel(const float* __restrict__ mu, const float* __restrict__ c_in,
                                                       const float* __restrict__ U1,
                                                       const float* __restrict__ U2, uint64_t seed, uint64_t offset,
                                                       const int* __restrict__ step_dev, float T,
                                                       const float* __restrict__ T_dev,
                                                       const float* __restrict__ Wcls,
                                                       const float* __restrict__ bcls, const float* __restrict__ Wlt,
                                                       const float* __restrict__ Wlf, const float* __restrict__ Wst,
                                                       const float* __restrict__ Wsf, float* __restrict__ ws,
                                                       float* __restrict__ c_out) {
  pdl_prologue();
  const int p = threadIdx.x;
  if (T_dev != nullptr) T = *T_dev;   // a captured step follows the host's per-epoch decay (gated_ccvae.py:404-406)
  if (p < 32) ws[GW_B + p] = (p < Y) ? bcls[p] : 0.0f;
  if (p >= NP) return;
  const int i = p / Y, j = p % Y;
  if (c_in != nullptr) {  // caller-provided gate (classifier_loss(x, y, c)): no sampling, no route to mu
    const float c = c_in[p];
    const int q = j * ZC + i;
    ws[GW_C + p] = c;
    ws[GW_M + p] = c * Wcls[p];
    ws[GW_PLT + q] = c * Wlt[q];
    ws[GW_PLF + q] = c * Wlf[q];
    ws[GW_PST + q] = c * Wst[q];
    ws[GW_PSF + q] = c * Wsf[q];
    ws[GW_DCDM + p] = 0.0f;
    if (c_out != nullptr) c_out[p] = c;
    return;
  }
  float u1, u2;
  if (U1 != nullptr) {
    u1 = U1[p];
    u2 = U2[p];
  } else {
    uint32_t r[4];
    if (step_dev) offset += (uint64_t)(*step_dev);
    philox4x32(seed, offset, PH_GATE, (uint64_t)p, r);
    u1 = u32_to_unit(r[0]);
    u2 = u32_to_unit(r[1]);
  }
  const float EPS = 1e-20f;
  const float muv = mu[p];
  const float m = clip_f(muv, 0.0f, 1.0f);
  const float g1 = -logf(-logf(u1 + EPS) + EPS);
  const float g2 = -logf(-logf(u2 + EPS) + EPS);
  const float a = 1.0f / T;
  const float num = expf((g2 - g1) / T);
  const float omm = 1.0f - m;
  const float t1 = powf(m, a);
  const float t2 = powf(omm, a) * num;
  const float den = t1 + t2 + EPS;
  const float c = t1 / den;
  // d c / d mu   (autograd of the expression above; clip passes gradient on the closed interval)
  const float t1p = a * powf(m, a - 1.0f);
  const float t2p = -a * powf(omm, a - 1.0f) * num;
  float dcdm = (t1p * (t2 + EPS) - t1 * t2p) / (den * den);
  if (!(muv >= 0.0f && muv <= 1.0f)) dcdm = 0.0f;
  ws[GW_C + p] = c;
  ws[GW_M + p] = c * Wcls[p];
  const int q = j * ZC + i;  // prior kernels are [j, i]
  ws[GW_PLT + q] = c * Wlt[q];
  ws[GW_PLF + q] = c * Wlf[q];
  ws[GW_PST + q] = c * Wst[q];
  ws[GW_PSF + q] = c * Wsf[q];
  ws[GW_DCDM + p] = dcdm;
  if (c_out != nullptr) c_out[p] = c;
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
template <bool SUP>
__global__ void __launch_bounds__(WARPS * 32) latent_fwd_kernel(gccvae_latent_fwd_args a) {
  pdl_prologue();
  __shared__ __align__(16) GateSmem g;
  __shared__ float s_locc[WARPS][ZC], s_scc[WARPS][ZC], s_zc[WARPS][ZC];
  load_gate_smem(g, a.gate_ws);
  __syncthreads();
  if (a.step_dev) a.offset += (uint64_t)(*a.step_dev);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int B = a.batch;
  const int ldp = a.ld_pre > 0 ? a.ld_pre : Z;
  const float invBg = 1.0f / (float)a.batch_global;
  float* locc = s_locc[wid];
  float* scc = s_scc[wid];
  float* zcs = s_zc[wid];

  for (int b = blockIdx.x * WARPS + wid; b < B; b += gridDim.x * WARPS) {
    // --- posterior, z, style KL -------------------------------------------------------------
    float kl_part = 0.0f;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int d = lane + 32 * h;
      if (d < Z) {
        float loc, sc;
        head_act(a.loc_pre[(size_t)b * ldp + d], a.scale_pre[(size_t)b * ldp + d], loc, sc);
        const float e = draw_eps(a.eps, a.seed, a.offset, b, d);
        const float z = fmaf(sc, e, loc);
        if (a.z16 != nullptr) reinterpret_cast<__nv_bfloat16*>(a.z16)[(size_t)b * 64 + d] = __float2bfloat16(z);
        a.loc[(size_t)b * Z + d] = loc;
        a.scale[(size_t)b * Z + d] = sc;
        a.z[(size_t)b * Z + d] = z;
        if (d < ZS) {
          kl_part += kl_dim(loc, sc, 0.0f, 1.0f);
        } else {
          locc[d - ZS] = loc;
          scc[d - ZS] = sc;
          zcs[d - ZS] = z;
        }
      } else if (d < 64 && a.z16 != nullptr) {
        reinterpret_cast<__nv_bfloat16*>(a.z16)[(size_t)b * 64 + d] = __float2bfloat16(0.0f);
      }
    }
    __syncwarp();
    // --- classifier at z, labels ---------------------------------------------------------------
    float logit = 0.0f;
    bool y1 = false;
    if (lane < Y) {
      float acc = g.b[lane];
#pragma unroll
      for (int i = 0; i < ZC; ++i) acc = fmaf(zcs[i], g.M[i * Y + lane], acc);
      logit = acc;
      if (SUP) {
        y1 = a.y[(size_t)b * Y + lane] != 0;
      } else {
        float u;
        if (a.U_y != nullptr) {
          u = a.U_y[(size_t)b * Y + lane];
        } else {
          uint32_t r[4];
          philox4x32(a.seed, a.offset, PH_UY, (uint64_t)b * 5 + (lane >> 2), r);
          u = u32_to_unit(r[lane & 3]);
        }
        y1 = u < sigmoid_f(logit);
      }
      a.logits[(size_t)b * Y + lane] = logit;
      if (a.y_out != nullptr) a.y_out[(size_t)b * Y + lane] = y1 ? 1 : 0;
    }
    const uint32_t ymask = __ballot_sync(0xffffffffu, y1);
    const float lq = warp_sum(lane < Y ? bern_lp(logit, y1) : 0.0f);
    // --- conditional prior + classify-dim KL -----------------------------------------------------
    if (lane < ZC) {
      float mp, spr;
      prior_i(g, ymask, lane, mp, spr);
      const float sp = clip_f(softplus_f(spr), 1e-3f, 1e3f);
      kl_part += kl_dim(locc[lane], scc[lane], mp, sp);
    }
    const float kl = warp_sum(kl_part);
    // --- K-sample log q(y|x) -----------------------------------------------------------------------
    float lqx = 0.0f, w = 1.0f;
    if (SUP) {
      float lc[ZC], sc[ZC];
#pragma unroll
      for (int i = 0; i < ZC; ++i) {
        lc[i] = locc[i];
        sc[i] = scc[i];
      }
      float m_run = -INFINITY, s_run = 0.0f;
      for (int k = lane; k < a.K; k += 32) {
        float e[ZC], zk[ZC], l[Y];
        draw_eps_k(a.eps_k, a.seed, a.offset, b, k, B, a.K, e);
#pragma unroll
        for (int i = 0; i < ZC; ++i) zk[i] = fmaf(sc[i], e[i], lc[i]);
        sample_logits(g, zk, l);
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < Y; ++j) acc += bern_lp(l[j], (ymask >> j) & 1u);
        const float m_new = fmaxf(m_run, acc);
        s_run = s_run * expf(m_run - m_new) + expf(acc - m_new);
        m_run = m_new;
      }
      const float mx = warp_max(m_run);
      const float part = (m_run == -INFINITY) ? 0.0f : s_run * expf(m_run - mx);
      const float tot = warp_sum(part);
      lqx = mx + logf(tot) - logf((float)a.K);
      w = expf(lq - lqx);
    }
    if (lane == 0) {
      a.terms[0 * (size_t)B + b] = kl;
      a.terms[1 * (size_t)B + b] = lq;
      a.terms[2 * (size_t)B + b] = lqx;
      a.terms[3 * (size_t)B + b] = w;
      a.terms[4 * (size_t)B + b] = (float)Y * logf(0.5f);
      a.terms[5 * (size_t)B + b] = -w * invBg;
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
struct BwdWarpSmem {
  float locc[ZC], scc[ZC], zc[ZC];
  float ev[48];
  float G[Y + 2], Gz[Y + 2], D[Y + 2];
  float dmp[ZC], dspr[ZC], dlockl[ZC], dsckl[ZC];
  float dzc[ZC], dlx[ZC], dsx[ZC];
  float E[NP];
  float stE[32][ZC + 1], stD[32][Y + 1];  // staging of one 32-sample chunk for the outer products
  float acc[5][NP];                       // dM | dPlt | dPlf | dPst | dPsf   ([i][j] pair order)
  float db[Y + 2];
};

template <bool SUP>
__global__ void __launch_bounds__(WARPS * 32) latent_bwd_kernel(gccvae_latent_bwd_args a) {
  pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GateSmem& g = *reinterpret_cast<GateSmem*>(smem_raw);
  BwdWarpSmem* wsm_all = reinterpret_cast<BwdWarpSmem*>(smem_raw + ((sizeof(GateSmem) + 15) / 16) * 16);
  __shared__ float s_loss[WARPS];
  load_gate_smem(g, a.gate_ws);
  if (a.step_dev) a.offset += (uint64_t)(*a.step_dev);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  BwdWarpSmem& s = wsm_all[wid];
  for (int t = lane; t < 5 * NP; t += 32) (&s.acc[0][0])[t] = 0.0f;
  if (lane < Y + 2) s.db[lane] = 0.0f;
  __syncthreads();
  const int B = a.batch;
  const int ldp = a.ld_pre > 0 ? a.ld_pre : Z, lddz = a.ld_dz > 0 ? a.ld_dz : Z;
  const float invBg = 1.0f / (float)a.batch_global;
  const float logK = SUP ? logf((float)a.K) : 0.0f;
  float loss_acc = 0.0f;
  float dbl[2] = {0.0f, 0.0f}, dbs[2] = {0.0f, 0.0f};  // bias-gradient partial sums of the two heads

  for (int b = blockIdx.x * WARPS + wid; b < B; b += gridDim.x * WARPS) {
    // --- recompute the forward quantities ---------------------------------------------------------
    float locv[2], scv[2], lpre[2], spre[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int d = lane + 32 * h;
      locv[h] = scv[h] = lpre[h] = spre[h] = 0.0f;
      if (d < Z) {
        lpre[h] = a.loc_pre[(size_t)b * ldp + d];
        spre[h] = a.scale_pre[(size_t)b * ldp + d];
        head_act(lpre[h], spre[h], locv[h], scv[h]);
        const float e = draw_eps(a.eps, a.seed, a.offset, b, d);
        s.ev[d] = e;
        if (d >= ZS) {
          s.locc[d - ZS] = locv[h];
          s.scc[d - ZS] = scv[h];
          s.zc[d - ZS] = fmaf(scv[h], e, locv[h]);
        }
      }
    }
    const bool y1 = (lane < Y) ? (a.y[(size_t)b * Y + lane] != 0) : false;
    const uint32_t ymask = __ballot_sync(0xffffffffu, y1);
    const float kl = a.terms[1 * 0 + b];
    const float lq = a.terms[1 * (size_t)B + b];
    const float lqx = a.terms[2 * (size_t)B + b];
    const float w = a.terms[3 * (size_t)B + b];
    const float lpy = a.terms[4 * (size_t)B + b];
    const float lpx = a.log_pxz[b];
    const float A = lpx - kl - lq;
    const float cA = w * invBg;                              // dL/dkl = dL/dlq = -dL/dlog_pxz
    const float g_lqp = SUP ? -A * w * invBg : 0.0f;         // dL/d log_qy_zc_ (detached-z copy)
    const float g_lqx = SUP ? (A * w - 1.0f) * invBg : 0.0f; // dL/d log_qy_x
    if (lane == 0) loss_acc += SUP ? -(w * A + lpy + lqx) * invBg : -(lpx + lpy - kl - lq) * invBg;
    __syncwarp();
    // --- classifier at z ------------------------------------------------------------------------------
    if (lane < Y) {
      float acc = g.b[lane];
#pragma unroll
      for (int i = 0; i < ZC; ++i) acc = fmaf(s.zc[i], g.M[i * Y + lane], acc);
      const float r = (y1 ? 1.0f : 0.0f) - sigmoid_f(acc);
      s.G[lane] = (cA + g_lqp) * r;
      s.Gz[lane] = cA * r;
    }
    // --- prior / KL on classify dims --------------------------------------------------------------------
    if (lane < ZC) {
      float mp, spr;
      prior_i(g, ymask, lane, mp, spr);
      const float spv = softplus_f(spr);
      const float sp = clip_f(spv, 1e-3f, 1e3f);
      const float inv = 1.0f / sp;
      const float lqv = s.locc[lane], sq = s.scc[lane];
      const float dq = lqv - mp;
      const float dl = cA * dq * inv * inv;
      s.dlockl[lane] = dl;
      s.dsckl[lane] = cA * (sq * inv * inv - 1.0f / sq);
      s.dmp[lane] = -dl;
      const float dsp = cA * (-(dq * dq) * inv * inv * inv - sq * sq * inv * inv * inv + inv);
      s.dspr[lane] = (spv >= 1e-3f && spv <= 1e3f) ? dsp * sigmoid_f(spr) : 0.0f;
    }
    // --- K-sample responsibilities, D_j = sum_k dl^k_j, E[i][j] = sum_k eps^k_i dl^k_j ------------------------
    float Eacc[PAIR_SLOTS];
#pragma unroll
    for (int r = 0; r < PAIR_SLOTS; ++r) Eacc[r] = 0.0f;
    float Dl[Y];
#pragma unroll
    for (int j = 0; j < Y; ++j) Dl[j] = 0.0f;
    if (SUP) {
      const float lse = lqx + logK;
      for (int k0 = 0; k0 < a.K; k0 += 32) {
        const int k = k0 + lane;
        float e[ZC], l[Y];
        if (k < a.K) {
          float zk[ZC];
          draw_eps_k(a.eps_k, a.seed, a.offset, b, k, B, a.K, e);
#pragma unroll
          for (int i = 0; i < ZC; ++i) zk[i] = fmaf(s.scc[i], e[i], s.locc[i]);
          sample_logits(g, zk, l);
          float acc = 0.0f;
#pragma unroll
          for (int j = 0; j < Y; ++j) acc += bern_lp(l[j], (ymask >> j) & 1u);
          const float rho = expf(acc - lse) * g_lqx;
#pragma unroll
          for (int j = 0; j < Y; ++j) {
            const float dlj = rho * ((((ymask >> j) & 1u) ? 1.0f : 0.0f) - sigmoid_f(l[j]));
            Dl[j] += dlj;
            s.stD[lane][j] = dlj;
          }
#pragma unroll
          for (int i = 0; i < ZC; ++i) s.stE[lane][i] = e[i];
        } else {
#pragma unroll
          for (int j = 0; j < Y; ++j) s.stD[lane][j] = 0.0f;
#pragma unroll
          for (int i = 0; i < ZC; ++i) s.stE[lane][i] = 0.0f;
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < PAIR_SLOTS; ++r) {
          const int p = lane + 32 * r;
          if (p < NP) {
            const int i = p / Y, j = p % Y;
            float accE = Eacc[r];
#pragma unroll 8
            for (int t = 0; t < 32; ++t) accE = fmaf(s.stE[t][i], s.stD[t][j], accE);
            Eacc[r] = accE;
          }
        }
        __syncwarp();
      }
#pragma unroll
      for (int j = 0; j < Y; ++j) Dl[j] = warp_sum(Dl[j]);
    }
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < Y; ++j) s.D[j] = Dl[j];
    }
#pragma unroll
    for (int r = 0; r < PAIR_SLOTS; ++r) {
      const int p = lane + 32 * r;
      if (p < NP) s.E[p] = Eacc[r];
    }
    __syncwarp();
    // --- per-pair accumulation into the batch sums (each pair is owned by exactly one lane) -----------------
#pragma unroll
    for (int r = 0; r < PAIR_SLOTS; ++r) {
      const int p = lane + 32 * r;
      if (p < NP) {
        const int i = p / Y, j = p % Y;
        const float yj = ((ymask >> j) & 1u) ? 1.0f : 0.0f;
        s.acc[0][p] += s.zc[i] * s.G[j] + s.locc[i] * s.D[j] + s.scc[i] * Eacc[r];
        s.acc[1][p] += yj * s.dmp[i];
        s.acc[2][p] += (1.0f - yj) * s.dmp[i];
        s.acc[3][p] += yj * s.dspr[i];
        s.acc[4][p] += (1.0f - yj) * s.dspr[i];
      }
    }
    if (lane < Y) s.db[lane] += s.G[lane] + s.D[lane];
    // --- back through the gated classifier matrix to z_c / loc_c / scale_c --------------------------------------
    if (lane < ZC) {
      float dz = 0.0f, dlx = 0.0f, dsx = 0.0f;
#pragma unroll
      for (int j = 0; j < Y; ++j) {
        const float m = g.M[lane * Y + j];
        dz = fmaf(m, s.Gz[j], dz);
        dlx = fmaf(m, s.D[j], dlx);
        dsx = fmaf(m, s.E[lane * Y + j], dsx);
      }
      s.dzc[lane] = dz;
      s.dlx[lane] = dlx;
      s.dsx[lane] = dsx;
    }
    __syncwarp();
    // --- assemble d loc / d scale and go through the head activations -------------------------------------------
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int d = lane + 32 * h;
      if (d < Z) {
        float dzt = a.dz[(size_t)b * lddz + d];
        float dloc, dsc;
        if (d < ZS) {
          dloc = dzt + cA * locv[h];
          dsc = dzt * s.ev[d] + cA * (scv[h] - 1.0f / scv[h]);
        } else {
          const int i = d - ZS;
          dzt += s.dzc[i];
          dloc = dzt + s.dlockl[i] + s.dlx[i];
          dsc = dzt * s.ev[d] + s.dsckl[i] + s.dsx[i];
        }
        const float spv = softplus_f(spre[h]);
        const float gl = (lpre[h] > 0.0f) ? dloc : 0.0f;
        const float gs = (spv >= 1e-3f && spv <= 1e3f) ? dsc * sigmoid_f(spre[h]) : 0.0f;
        if (a.dloc_pre != nullptr) {
          a.dloc_pre[(size_t)b * Z + d] = gl;
          a.dscale_pre[(size_t)b * Z + d] = gs;
        }
        if (a.dpre16 != nullptr) {
          __nv_bfloat16* row = reinterpret_cast<__nv_bfloat16*>(a.dpre16) + (size_t)b * 96;
          row[d] = __float2bfloat16(gl);
          row[48 + d] = __float2bfloat16(gs);
        }
        dbl[h] += gl;
        dbs[h] += gs;
      } else if (d < 48 && a.dpre16 != nullptr) {
        __nv_bfloat16* row = reinterpret_cast<__nv_bfloat16*>(a.dpre16) + (size_t)b * 96;
        row[d] = __float2bfloat16(0.0f);
        row[48 + d] = __float2bfloat16(0.0f);
      }
    }
    __syncwarp();
  }
  if (a.db_loc != nullptr) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int d = lane + 32 * h;
      if (d < Z) {
        atomicAdd(a.db_loc + d, dbl[h]);
        atomicAdd(a.db_scale + d, dbs[h]);
      }
    }
  }
  // --- CTA reduction of the per-warp batch sums -> one partial row per CTA ---------------------------------------
  if (lane == 0) s_loss[wid] = loss_acc;
  __syncthreads();
  float* out = a.partials + (size_t)blockIdx.x * PT_TOTAL;
  for (int t = threadIdx.x; t < 5 * NP; t += blockDim.x) {
    const int mtx = t / NP, p = t % NP;
    float v = 0.0f;
#pragma unroll
    for (int wq = 0; wq < WARPS; ++wq) v += wsm_all[wq].acc[mtx][p];
    // prior matrices are stored [j][i] like the reference kernels
    const int dst = (mtx == 0) ? p : (p % Y) * ZC + (p / Y);
    out[mtx * NP + dst] = v;
  }
  if (threadIdx.x < 32) {
    float v = 0.0f;
    if (threadIdx.x < Y) {
#pragma unroll
      for (int wq = 0; wq < WARPS; ++wq) v += wsm_all[wq].db[threadIdx.x];
    } else if (threadIdx.x == Y) {
#pragma unroll
      for (int wq = 0; wq < WARPS; ++wq) v += s_loss[wq];
    }
    if (PT_DB + threadIdx.x < PT_TOTAL) out[PT_DB + threadIdx.x] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// gate backward: reduce partials, un-gate, chain to mu, add L1.  One CTA.
// ---------------------------------------------------------------------------------------------
// (partial rows are read with ld.global.cg: in the merged kernel below they were written by OTHER blocks of the same
// grid, which a non-coherent / L1-cached load is not guaranteed to see)
__device__ __forceinline__ void gate_bwd_body(const float* partials, int n_partials,
                                              const float* __restrict__ mu, const float* __restrict__ Wcls,
                                              const float* __restrict__ Wlt, const float* __restrict__ Wlf,
                                              const float* __restrict__ Wst, const float* __restrict__ Wsf,
                                              const float* __restrict__ ws, float gating_reg, float l1_scale,
                                              float* __restrict__ dWcls, float* __restrict__ dbcls,
                                              float* __restrict__ dWlt, float* __restrict__ dWlf,
                                              float* __restrict__ dWst, float* __restrict__ dWsf,
                                              float* __restrict__ dmu, float* __restrict__ loss_inout) {
  __shared__ float s_dc[NP];
  __shared__ float s_red[352 / 32];
  const int p = threadIdx.x;
  float absmu = 0.0f;
  float sum[5] = {0, 0, 0, 0, 0};
  // thread p handles element p of each matrix IN THAT MATRIX'S OWN layout:
  // dM is [i][j] (p = i*18+j); the four prior sums are [j][i] (p = j2*18+i2).
  const int i2 = p % ZC, j2 = p / ZC;
  if (p < NP) {
    for (int n = 0; n < n_partials; ++n) {
      const float* row = partials + (size_t)n * PT_TOTAL;
#pragma unroll
      for (int m = 0; m < 5; ++m) sum[m] += __ldcg(row + m * NP + p);
    }
    const float c_ij = ws[GW_C + p];
    const float c_prior = ws[GW_C + i2 * Y + j2];
    if (dWcls) dWcls[p] = sum[0] * c_ij;
    if (dWlt) dWlt[p] = sum[1] * c_prior;
    if (dWlf) dWlf[p] = sum[2] * c_prior;
    if (dWst) dWst[p] = sum[3] * c_prior;
    if (dWsf) dWsf[p] = sum[4] * c_prior;
    s_dc[p] = sum[0] * Wcls[p];
  } else if (p - NP < Y && dbcls) {
    const int j = p - NP;
    float v = 0.0f;
    for (int n = 0; n < n_partials; ++n) v += __ldcg(partials + (size_t)n * PT_TOTAL + PT_DB + j);
    dbcls[j] = v;
  }
  __syncthreads();
  // second phase touches each s_dc element exactly once (p -> (i2,j2) is a permutation)
  if (p < NP) s_dc[i2 * Y + j2] += sum[1] * Wlt[p] + sum[2] * Wlf[p] + sum[3] * Wst[p] + sum[4] * Wsf[p];
  __syncthreads();
  if (p < NP && dmu) {
    const float muv = mu[p];
    const float sgn = (muv > 0.0f) ? 1.0f : ((muv < 0.0f) ? -1.0f : 0.0f);
    dmu[p] = s_dc[p] * ws[GW_DCDM + p] + l1_scale * gating_reg * sgn / (float)NP;
    absmu = fabsf(muv);
  }
  // loss: sum of partial losses + L1
  float lossv = 0.0f;
  if (p == NP + Y) {
    for (int n = 0; n < n_partials; ++n) lossv += __ldcg(partials + (size_t)n * PT_TOTAL + PT_LOSS);
  }
  float tot = warp_sum(absmu);
  if ((p & 31) == 0) s_red[p >> 5] = tot;
  __syncthreads();
  if (p == NP + Y) {
    float l1 = 0.0f;
    for (int q = 0; q < 352 / 32; ++q) l1 += s_red[q];
    if (dmu == nullptr) l1 = 0.0f;
    if (loss_inout) loss_inout[0] = lossv + l1_scale * gating_reg * l1 / (float)NP;
  }
}

// Both steps in ONE launch (one dependent launch less on the step's critical path): every block reduces 352 columns
// of the partial rows into `reduced` (4 independent accumulators per thread, fixed order: deterministic), takes a ticket, and the
// block that draws the last ticket - all columns are then visible - runs the gate backward on the reduced row.
// The ticket is slot GW_B + 31 of the gate workspace: gate_fwd zeroes it every step, the last block re-zeroes it.
__global__ void __launch_bounds__(352) reduce_gate_bwd_kernel(const float* __restrict__ partials, int n_partials,
                                                              float* reduced, unsigned int* ticket,
                                                              const float* __restrict__ mu, const float* __restrict__ Wcls,
                                                              const float* __restrict__ Wlt, const float* __restrict__ Wlf,
                                                              const float* __restrict__ Wst, const float* __restrict__ Wsf,
                                                              const float* __restrict__ ws, float gating_reg,
                                                              float l1_scale, float* __restrict__ dWcls,
                                                              float* __restrict__ dbcls, float* __restrict__ dWlt,
                                                              float* __restrict__ dWlf, float* __restrict__ dWst,
                                                              float* __restrict__ dWsf, float* __restrict__ dmu,
                                                              float* __restrict__ loss_inout) {
  pdl_prologue();
  __shared__ int s_last;
  const int c = blockIdx.x * 352 + threadIdx.x;
  if (c < PT_TOTAL) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int n = 0;
    for (; n + 4 <= n_partials; n += 4) {
      a0 += partials[(size_t)(n + 0) * PT_TOTAL + c];
      a1 += partials[(size_t)(n + 1) * PT_TOTAL + c];
      a2 += partials[(size_t)(n + 2) * PT_TOTAL + c];
      a3 += partials[(size_t)(n + 3) * PT_TOTAL + c];
    }
    for (; n < n_partials; ++n) a0 += partials[(size_t)n * PT_TOTAL + c];
    reduced[c] = (a0 + a1) + (a2 + a3);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (threadIdx.x == 0) *ticket = 0u;
  gate_bwd_body(reduced, 1, mu, Wcls, Wlt, Wlf, Wst, Wsf, ws, gating_reg, l1_scale, dWcls, dbcls, dWlt, dWlf, dWst, dWsf,
                dmu, loss_inout);
}

// ---------------------------------------------------------------------------------------------
// tiled module API + standalone KL (API sugar; the fused kernels above are the hot path)
// ---------------------------------------------------------------------------------------------
__global__ void classifier_tiled_kernel(const float* __restrict__ zt, long long sb, long long si, long long sj,
                                        int batch, const float* __restrict__ gates, const float* __restrict__ W,
                                        const float* __restrict__ bias, float* __restrict__ logits) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= batch * Y) return;
  const int b = t / Y, j = t % Y;
  float acc = 0.0f;
  for (int i = 0; i < ZC; ++i) acc += (zt[b * sb + i * si + j * sj] * gates[i * Y + j]) * W[i * Y + j];
  logits[t] = acc + bias[j];
}

__global__ void cond_prior_tiled_kernel(const float* __restrict__ yt, long long sb, long long sj, long long si,
                                        int batch, const float* __restrict__ c, const float* __restrict__ Wlt,
                                        const float* __restrict__ Wlf, const float* __restrict__ Wst,
                                        const float* __restrict__ Wsf, float* __restrict__ loc,
                                        float* __restrict__ scale) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= batch * ZC) return;
  const int b = t / ZC, i = t % ZC;
  float l = 0.0f, l2 = 0.0f, s = 0.0f, s2 = 0.0f;
  for (int j = 0; j < Y; ++j) {
    const float yv = yt[b * sb + j * sj + i * si];
    const float ct = c[i * Y + j];
    l += (yv * ct) * Wlt[j * ZC + i];
    l2 += ((1.0f - yv) * ct) * Wlf[j * ZC + i];
    s += (yv * ct) * Wst[j * ZC + i];
    s2 += ((1.0f - yv) * ct) * Wsf[j * ZC + i];
  }
  loc[t] = l + l2;
  scale[t] = clip_f(softplus_f(s + s2), 1e-3f, 1e3f);
}

__global__ void gaussian_kl_kernel(const float* __restrict__ lq, const float* __restrict__ sq,
                                   const float* __restrict__ lp, const float* __restrict__ sp, int batch, int dims,
                                   float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= batch) return;
  float acc = 0.0f;
  for (int d = lane; d < dims; d += 32) {
    const size_t o = (size_t)b * dims + d;
    acc += kl_dim(lq[o], sq[o], lp ? lp[o] : 0.0f, sp ? sp[o] : 1.0f);
  }
  acc = warp_sum(acc);
  if (lane == 0) out[b] = acc;
}

__global__ void draw_noise_kernel(int kind, uint64_t seed, uint64_t offset, int B, int K, float* __restrict__ out) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (kind == 0) {
    if (t < (long long)B * Z) out[t] = draw_eps(nullptr, seed, offset, (int)(t / Z), (int)(t % Z));
  } else if (kind == 1) {
    if (t < (long long)B * K) {
      const int b = (int)(t / K), k = (int)(t % K);
      float e[ZC];
      draw_eps_k(nullptr, seed, offset, b, k, B, K, e);
      for (int i = 0; i < ZC; ++i) out[((size_t)k * B + b) * ZC + i] = e[i];
    }
  } else if (kind == 2) {
    if (t < (long long)B * Y) {
      const int b = (int)(t / Y), j = (int)(t % Y);
      uint32_t r[4];
      philox4x32(seed, offset, PH_UY, (uint64_t)b * 5 + (j >> 2), r);
      out[t] = u32_to_unit(r[j & 3]);
    }
  } else {
    if (t < NP) {
      uint32_t r[4];
      philox4x32(seed, offset, PH_GATE, (uint64_t)t, r);
      out[t] = u32_to_unit(r[0]);
      out[NP + t] = u32_to_unit(r[1]);
    }
  }
}

__global__ void head_act_kernel(const float* __restrict__ lp, const float* __restrict__ sp, long long n,
                                float* __restrict__ loc, float* __restrict__ scale) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float l, s;
  head_act(lp[i], sp[i], l, s);
  loc[i] = l;
  scale[i] = s;
}

// mean(round(sigmoid(logit)) == y); round-half-even of exactly 0.5 is 0, so y_hat = sigmoid > 0.5
__global__ void __launch_bounds__(256) accuracy_kernel(const float* __restrict__ logits,
                                                       const long long* __restrict__ y, int n,
                                                       float* __restrict__ out) {
  __shared__ int red[8];
  int hit = 0;
  for (int i = threadIdx.x; i < n; i += 256) {
    const int yh = sigmoid_f(logits[i]) > 0.5f ? 1 : 0;
    hit += (yh == (int)y[i]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) hit += __shfl_xor_sync(0xffffffffu, hit, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = hit;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int q = 0; q < 8; ++q) t += red[q];
    out[0] = (float)t / (float)n;
  }
}

// ---------------------------------------------------------------------------------------------
// latent code of the forward-only image calls (gccvae_gen_latent, include/gccvae.h): one warp per frame
// ---------------------------------------------------------------------------------------------
// prior_i with label l at the real value alpha: at alpha = 0 / 1 the term of l is the prior's own select (so the result is
// prior_i's bit for bit), otherwise alpha P_true + (1 - alpha) P_false as one fmaf; the sum keeps prior_i's order.
// l = Y, alpha = 0 walks no label: ymask has no bit Y, so every term is prior_i's select
__device__ __forceinline__ void prior_walk_i(const GateSmem& g, uint32_t ymask, int l, float alpha, int i, float& mp,
                                             float& spr) {
  const bool between = !(alpha == 0.0f || alpha == 1.0f);
  const uint32_t m = alpha == 1.0f ? (ymask | (1u << l)) : (ymask & ~(1u << l));
  float a = 0.0f, s = 0.0f;
#pragma unroll
  for (int j = 0; j < Y; ++j) {
    const int q = j * ZC + i;
    const bool y1 = (m >> j) & 1u;
    float ta = y1 ? g.Plt[q] : g.Plf[q], ts = y1 ? g.Pst[q] : g.Psf[q];
    if (between && j == l) {
      ta = fmaf(alpha, g.Plt[q] - g.Plf[q], g.Plf[q]);
      ts = fmaf(alpha, g.Pst[q] - g.Psf[q], g.Psf[q]);
    }
    a += ta;
    s += ts;
  }
  mp = a;
  spr = s;
}

__global__ void __launch_bounds__(WARPS * 32) gen_latent_kernel(gccvae_gen_latent_args a) {
  pdl_prologue();
  __shared__ __align__(16) GateSmem g;
  __shared__ float s_zc[WARPS][ZC];
  load_gate_smem(g, a.gate_ws);
  __syncthreads();
  // a local, not a.offset +=: a written parameter struct of this size loses its pointers' global address space
  const uint64_t offset = a.offset + (a.step_dev ? (uint64_t)(*a.step_dev) : 0ull);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int ldp = a.ld_pre > 0 ? a.ld_pre : Z;
  const bool from_image = a.mode != GCCVAE_GEN_GENERATE;
  const int n_sel = a.n_labels > 0 ? a.n_labels : a.n_dims;    // walked labels or traversed dims (at most one is > 0)
  const int per_image = n_sel > 0 ? n_sel * a.n_alpha : (a.pair ? a.n_alpha : 1);
  float* zcs = s_zc[wid];

  for (int r = blockIdx.x * WARPS + wid; r < a.rows; r += gridDim.x * WARPS) {
    const int gr = a.row0 + r, b = gr / per_image, f = gr - b * per_image;
    int l = Y;          // walked label; Y: none, and then prior_walk_i ignores alpha
    int dt = Z;         // traversed dim; Z: none
    float alpha = 0.0f; // the frame's value: of label l, of dim dt, or the pair's t
    if (n_sel > 0) {
      const int si = f / a.n_alpha;
      alpha = a.alphas[f - si * a.n_alpha];
      // constant-bank reads: a dynamic index would copy the params to the stack
      if (a.n_labels > 0) {
#pragma unroll
        for (int k = 0; k < Y; ++k) l = k == si ? a.labels[k] : l;
      } else {
#pragma unroll
        for (int k = 0; k < Z; ++k) dt = k == si ? a.dims[k] : dt;
      }
    } else if (a.pair) {
      alpha = a.alphas[f];
    }
    // --- posterior (Reconstruct / Intervene) or N(0,1) style dims (Generate) ------------------------------------
    float zv[2] = {0.0f, 0.0f};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int d = lane + 32 * h;
      if (d >= Z) continue;
      float z = 0.0f;
      if (from_image) {
        float loc, sc;
        head_act(a.loc_pre[(size_t)b * ldp + d], a.scale_pre[(size_t)b * ldp + d], loc, sc);
        z = a.sample ? fmaf(sc, draw_eps(a.eps, a.seed, offset, b, d), loc) : loc;
        if (a.pair && d >= a.mix_lo && d < a.mix_hi) {   // z_a -> z_b, both ends exact (as prior_walk_i)
          float loc_b, sc_b;
          head_act(a.loc_pre[(size_t)(a.batch + b) * ldp + d], a.scale_pre[(size_t)(a.batch + b) * ldp + d], loc_b, sc_b);
          z = alpha == 0.0f ? z : (alpha == 1.0f ? loc_b : fmaf(alpha, loc_b - z, z));
        }
      } else if (d < ZS && a.sample) {
        z = draw_eps(a.eps, a.seed, offset, b, d);
      }
      zv[h] = z;
      if (d >= ZS) zcs[d - ZS] = z;
    }
    __syncwarp();
    // --- labels: (Intervene) source = given or the classifier's decision on z_c; target = given or the source --------
    bool yt = false, ys = false;
    if (lane < Y) {
      if (a.mode == GCCVAE_GEN_INTERVENE) {
        if (a.y_src != nullptr) {
          ys = a.y_src[(size_t)b * Y + lane] != 0;
        } else {
          float acc = g.b[lane];
#pragma unroll
          for (int i = 0; i < ZC; ++i) acc = fmaf(zcs[i], g.M[i * Y + lane], acc);
          ys = sigmoid_f(acc) > 0.5f;
        }
        if (a.y_src_out != nullptr && f == 0) a.y_src_out[(size_t)b * Y + lane] = ys ? 1 : 0;
      }
      if (a.mode != GCCVAE_GEN_RECONSTRUCT) yt = a.y_tgt != nullptr ? a.y_tgt[(size_t)b * Y + lane] != 0 : ys;
    }
    const uint32_t tmask = __ballot_sync(0xffffffffu, yt), smask = __ballot_sync(0xffffffffu, ys);
    // --- classify dims through the conditional prior at the target, label l at alpha (lane i < ZC: classify dim i) -----
    if (lane < ZC && a.mode != GCCVAE_GEN_RECONSTRUCT) {
      float mt, st;
      prior_walk_i(g, tmask, l, alpha, lane, mt, st);
      const float spt = clip_f(softplus_f(st), 1e-3f, 1e3f);
      float zc;
      if (a.mode == GCCVAE_GEN_GENERATE) {
        zc = a.sample ? fmaf(spt, draw_eps(a.eps, a.seed, offset, b, ZS + lane), mt) : mt;
      } else {
        float ms, ss;
        prior_i(g, smask, lane, ms, ss);
        const float sps = clip_f(softplus_f(ss), 1e-3f, 1e3f);
        const float z0 = zcs[lane];
        const float e = (z0 - ms) / sps;
        zc = fmaf(spt - sps, e, z0 + (mt - ms));   // incremental form: an unchanged prior leaves z_c bit-identical
      }
      zcs[lane] = zc;
    }
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int d = lane + 32 * h;
      if (d < Z) {
        const float z = d == dt ? alpha : (d >= ZS ? zcs[d - ZS] : zv[h]);
        if (a.z != nullptr) a.z[(size_t)r * Z + d] = z;
        if (a.z16 != nullptr) reinterpret_cast<__nv_bfloat16*>(a.z16)[(size_t)r * 64 + d] = __float2bfloat16(z);
      } else if (d < 64 && a.z16 != nullptr) {
        reinterpret_cast<__nv_bfloat16*>(a.z16)[(size_t)r * 64 + d] = __float2bfloat16(0.0f);
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// importance-weighted log-likelihood (gccvae_iw_latent / gccvae_iw_accumulate, include/gccvae.h)
// ---------------------------------------------------------------------------------------------
// Philox index of (image b, sample k): independent of B and of the chunking
__device__ __forceinline__ uint64_t iw_index(int b, int k) { return ((uint64_t)b << 32) | (uint32_t)k; }

__device__ __forceinline__ float draw_iw_eps(const float* __restrict__ eps, uint64_t seed, uint64_t offset, int B, int b,
                                             int k, int d) {
  if (eps != nullptr) return eps[((size_t)k * B + b) * Z + d];
  float n[4];
  philox_normal4(seed, offset, PH_IW_EPS, iw_index(b, k) * 12 + (d >> 2), n);
  return n[d & 3];
}

__device__ __forceinline__ float draw_iw_uy(const float* __restrict__ U_y, uint64_t seed, uint64_t offset, int B, int b,
                                            int k, int j) {
  if (U_y != nullptr) return U_y[((size_t)k * B + b) * Y + j];
  uint32_t r[4];
  philox4x32(seed, offset, PH_IW_UY, iw_index(b, k) * 5 + (j >> 2), r);
  return u32_to_unit(r[j & 3]);
}

// One warp per row.  The Normal normalisers cancel: log p(z_s) + log p(z_c|y) - log q(z|x) carries
// (-27 - 18 + 45) * ln(2 pi) / 2 = 0, so none of the three terms adds it.
__global__ void __launch_bounds__(WARPS * 32) iw_latent_kernel(gccvae_iw_latent_args a) {
  pdl_prologue();
  __shared__ __align__(16) GateSmem g;
  __shared__ float s_zc[WARPS][ZC];
  load_gate_smem(g, a.gate_ws);
  __syncthreads();
  if (a.step_dev) a.offset += (uint64_t)(*a.step_dev);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int ldp = a.ld_pre > 0 ? a.ld_pre : Z;
  const int rows = a.batch * a.kc;
  float* zcs = s_zc[wid];

  for (int r = blockIdx.x * WARPS + wid; r < rows; r += gridDim.x * WARPS) {
    const int b = r / a.kc, k = a.k0 + (r - b * a.kc);
    // --- z_k = loc + scale eps_k; -log q(z_k|x) and log p(z_s) ----------------------------------------------
    float part = 0.0f;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int d = lane + 32 * h;
      if (d < Z) {
        float loc, sc;
        head_act(a.loc_pre[(size_t)b * ldp + d], a.scale_pre[(size_t)b * ldp + d], loc, sc);
        const float e = draw_iw_eps(a.eps, a.seed, a.offset, a.batch, b, k, d);
        const float z = fmaf(sc, e, loc);
        part += fmaf(0.5f * e, e, logf(sc));            // -log q(z_k|x), dimension d
        if (d < ZS) part -= 0.5f * z * z;                 // log p(z_s)
        else zcs[d - ZS] = z;
        if (a.z != nullptr) a.z[(size_t)r * Z + d] = z;
        if (a.z16 != nullptr) reinterpret_cast<__nv_bfloat16*>(a.z16)[(size_t)r * 64 + d] = __float2bfloat16(z);
      } else if (d < 64 && a.z16 != nullptr) {
        reinterpret_cast<__nv_bfloat16*>(a.z16)[(size_t)r * 64 + d] = __float2bfloat16(0.0f);
      }
    }
    __syncwarp();
    // --- labels y_k: given, or drawn from the gated classifier (then -log q(y_k|z_c,k)) ----------------------------
    bool y1 = false;
    float lqy = 0.0f;
    if (lane < Y) {
      if (a.labelled) {
        y1 = a.y[(size_t)b * Y + lane] != 0;
      } else {
        float acc = g.b[lane];
#pragma unroll
        for (int i = 0; i < ZC; ++i) acc = fmaf(zcs[i], g.M[i * Y + lane], acc);
        y1 = draw_iw_uy(a.U_y, a.seed, a.offset, a.batch, b, k, lane) < sigmoid_f(acc);
        lqy = bern_lp(acc, y1);
      }
    }
    part -= lqy;
    const uint32_t ymask = __ballot_sync(0xffffffffu, y1);
    // --- log p(z_c,k|y_k) under the conditional prior ---------------------------------------------------------------
    if (lane < ZC) {
      float mp, spr;
      prior_i(g, ymask, lane, mp, spr);
      const float sp = clip_f(softplus_f(spr), 1e-3f, 1e3f);
      const float t = (zcs[lane] - mp) / sp;
      part -= fmaf(0.5f * t, t, logf(sp));
    }
    const float lw = warp_sum(part);
    if (lane == 0) a.lw_part[r] = lw + (float)Y * logf(0.5f);   // + log p(y_k)
    __syncwarp();
  }
}

// one warp per image: the lanes stride over the chunk's kc rows with their own running (max, sums), joined by shuffles
__global__ void __launch_bounds__(256) iw_accumulate_kernel(int B, int kc, int k0, int K,
                                                            const float* __restrict__ lw_part,
                                                            const float* __restrict__ log_pxz, float* __restrict__ state,
                                                            float* __restrict__ log_w, int first, int finalize,
                                                            float* __restrict__ est, float* __restrict__ ess) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= B) return;
  float m = -INFINITY, s1 = 0.0f, s2 = 0.0f;
  for (int j = lane; j < kc; j += 32) {
    const size_t r = (size_t)b * kc + j;
    const float lw = lw_part[r] + log_pxz[r];
    if (log_w != nullptr) log_w[(size_t)(k0 + j) * B + b] = lw;
    const float m_new = fmaxf(m, lw);
    const float f = m == -INFINITY ? 0.0f : expf(m - m_new), e = expf(lw - m_new);
    s1 = fmaf(s1, f, e);
    s2 = fmaf(s2, f * f, e * e);
    m = m_new;
  }
  // the warp's chunk result, then the state of the earlier chunks (lane 0)
  const float mx = warp_max(m);
  const float f = m == -INFINITY ? 0.0f : expf(m - mx);
  s1 = warp_sum(s1 * f);
  s2 = warp_sum(s2 * f * f);
  if (lane != 0) return;
  m = mx;
  if (!first) {
    const float mo = state[3 * (size_t)b], so1 = state[3 * (size_t)b + 1], so2 = state[3 * (size_t)b + 2];
    const float m_new = fmaxf(mo, m);
    const float fo = mo == -INFINITY ? 0.0f : expf(mo - m_new), fc = m == -INFINITY ? 0.0f : expf(m - m_new);
    s1 = so1 * fo + s1 * fc;
    s2 = so2 * fo * fo + s2 * fc * fc;
    m = m_new;
  }
  state[3 * (size_t)b] = m;
  state[3 * (size_t)b + 1] = s1;
  state[3 * (size_t)b + 2] = s2;
  if (finalize) {
    est[b] = m + logf(s1) - logf((float)K);
    ess[b] = s1 * s1 / s2;
  }
}

// kinds 4 / 5 of gccvae_draw_noise_f32: eps [K,B,45] and U_y [K,B,18] of iw_latent_kernel
__global__ void draw_iw_noise_kernel(int kind, uint64_t seed, uint64_t offset, int B, int K, float* __restrict__ out) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int w = kind == 4 ? Z : Y;
  if (t >= (long long)K * B * w) return;
  const int d = (int)(t % w);
  const long long kb = t / w;
  const int b = (int)(kb % B), k = (int)(kb / B);
  out[t] = kind == 4 ? draw_iw_eps(nullptr, seed, offset, B, b, k, d) : draw_iw_uy(nullptr, seed, offset, B, b, k, d);
}

}  // namespace gccvae

using namespace gccvae;

extern "C" int gccvae_draw_noise_f32(int kind, uint64_t seed, uint64_t offset, int batch, int K, float* out,
                                     void* stream) {
  GCC_REQUIRE(out && kind >= 0 && kind <= 5 && batch > 0, "draw_noise: bad args");
  if (kind >= 4) {
    GCC_REQUIRE(K >= 1, "draw_noise: kinds 4 / 5 need K >= 1");
    const long long n4 = (long long)K * batch * (kind == 4 ? Z : Y);
    draw_iw_noise_kernel<<<(int)((n4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(kind, seed, offset, batch, K, out);
    GCC_CHECK_LAUNCH("draw_noise");
    return GCCVAE_OK;
  }
  long long n = kind == 0 ? (long long)batch * Z : kind == 1 ? (long long)batch * K : kind == 2 ? (long long)batch * Y : NP;
  GCC_REQUIRE(n > 0, "draw_noise: empty");
  draw_noise_kernel<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(kind, seed, offset, batch, K, out);
  GCC_CHECK_LAUNCH("draw_noise");
  return GCCVAE_OK;
}

extern "C" int gccvae_head_act_f32(const float* loc_pre, const float* scale_pre, long long n, float* loc, float* scale,
                                   void* stream) {
  GCC_REQUIRE(loc_pre && scale_pre && loc && scale && n > 0, "head_act: bad args");
  head_act_kernel<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(loc_pre, scale_pre, n, loc, scale);
  GCC_CHECK_LAUNCH("head_act");
  return GCCVAE_OK;
}

extern "C" int gccvae_accuracy_f32(const float* logits, const long long* y, int n, float* out, void* stream) {
  GCC_REQUIRE(logits && y && out && n > 0, "accuracy: bad args");
  accuracy_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(logits, y, n, out);
  GCC_CHECK_LAUNCH("accuracy");
  return GCCVAE_OK;
}

extern "C" int gccvae_gate_fwd(const float* mu, const float* c_in, const float* U1, const float* U2, uint64_t seed,
                               uint64_t offset, const int* step_dev, float temperature, const float* temperature_dev, const float* Wcls, const float* bcls, const float* Wlt,
                               const float* Wlf, const float* Wst, const float* Wsf, float* gate_ws, float* c_out,
                               void* stream) {
  GCC_REQUIRE((mu || c_in) && Wcls && bcls && Wlt && Wlf && Wst && Wsf && gate_ws, "gate_fwd: null pointer");
  GCC_REQUIRE((U1 == nullptr) == (U2 == nullptr), "gate_fwd: U1 and U2 must both be given or both be NULL");
  GCC_REQUIRE(temperature > 0.0f || temperature_dev, "gate_fwd: temperature must be > 0");
  GCC_CUDA(launch_aux(gate_fwd_kernel, dim3(1), dim3(352), 0, (cudaStream_t)stream, mu, c_in, U1, U2, seed, offset,
                      step_dev, temperature, temperature_dev, Wcls, bcls, Wlt, Wlf, Wst, Wsf, gate_ws, c_out));
  GCC_CHECK_LAUNCH("gate_fwd");
  return GCCVAE_OK;
}

static int latent_grid(int batch) {
  int ctas = (batch + WARPS - 1) / WARPS;
  const int cap = 148 * 2;
  return ctas < 1 ? 1 : (ctas > cap ? cap : ctas);
}

extern "C" int gccvae_latent_fwd(const gccvae_latent_fwd_args* a, void* stream) {
  GCC_REQUIRE(a, "latent_fwd: null args");
  GCC_REQUIRE(a->batch > 0 && a->batch_global >= a->batch, "latent_fwd: bad batch %d/%d", a->batch, a->batch_global);
  GCC_REQUIRE(a->loc_pre && a->scale_pre && a->gate_ws && a->loc && a->scale && a->z && a->terms && a->logits,
              "latent_fwd: null pointer");
  if (a->supervised) {
    GCC_REQUIRE(a->y, "latent_fwd: supervised needs y");
    GCC_REQUIRE(a->K >= 1, "latent_fwd: K must be >= 1");
  }
  GCC_REQUIRE((uintptr_t)a->eps_k % 8 == 0, "latent_fwd: eps_k must be 8-byte aligned");
  const int grid = latent_grid(a->batch);
  if (a->supervised)
    GCC_CUDA(launch_aux(latent_fwd_kernel<true>, dim3(grid), dim3(WARPS * 32), 0, (cudaStream_t)stream, *a));
  else
    GCC_CUDA(launch_aux(latent_fwd_kernel<false>, dim3(grid), dim3(WARPS * 32), 0, (cudaStream_t)stream, *a));
  GCC_CHECK_LAUNCH("latent_fwd");
  return GCCVAE_OK;
}

extern "C" int gccvae_gen_latent(const gccvae_gen_latent_args* a, void* stream) {
  GCC_REQUIRE(a, "gen_latent: null args");
  GCC_REQUIRE(a->mode >= GCCVAE_GEN_GENERATE && a->mode <= GCCVAE_GEN_INTERVENE,
              "gen_latent: mode %d (1 generate, 2 reconstruct, 3 intervene)", a->mode);
  const int kinds = (a->n_labels != 0) + (a->n_dims != 0) + (a->pair != 0);
  GCC_REQUIRE(kinds <= 1, "gen_latent: a row is at most one of a label walk, a traversal and a pair");
  GCC_REQUIRE(a->batch > 0 && a->n_labels >= 0 && a->n_labels <= Y && a->n_dims >= 0 && a->n_dims <= Z &&
                  (a->pair == 0 || a->pair == 1) && (kinds == 0 || a->n_alpha >= 1),
              "gen_latent: bad sizes B=%d labels=%d dims=%d pair=%d alphas=%d", a->batch, a->n_labels, a->n_dims, a->pair,
              a->n_alpha);
  GCC_REQUIRE(a->n_labels == 0 || a->mode != GCCVAE_GEN_RECONSTRUCT, "gen_latent: reconstruct walks no label");
  GCC_REQUIRE(!a->pair || (a->mode == GCCVAE_GEN_RECONSTRUCT && a->sample == 0 && a->mix_lo >= 0 &&
                           a->mix_lo < a->mix_hi && a->mix_hi <= Z),
              "gen_latent: a pair needs reconstruct without sampling and 0 <= mix_lo < mix_hi <= 45 (got mode %d, "
              "sample %d, [%d, %d))", a->mode, a->sample, a->mix_lo, a->mix_hi);
  const long long per_image = a->n_labels > 0 ? (long long)a->n_labels * a->n_alpha
                              : a->n_dims > 0 ? (long long)a->n_dims * a->n_alpha
                              : a->pair       ? (long long)a->n_alpha
                                              : 1LL;
  const long long total = (long long)a->batch * per_image;
  GCC_REQUIRE(total < (1LL << 31), "gen_latent: too many rows");
  GCC_REQUIRE(a->row0 >= 0 && a->rows >= 1 && (long long)a->row0 + a->rows <= total,
              "gen_latent: chunk %d + %d outside the %lld rows", a->row0, a->rows, total);
  unsigned seen = 0;
  for (int i = 0; i < a->n_labels; ++i) {
    GCC_REQUIRE(a->labels[i] >= 0 && a->labels[i] < Y && !((seen >> a->labels[i]) & 1u),
                "gen_latent: labels must be distinct indices in [0, 18)");
    seen |= 1u << a->labels[i];
  }
  unsigned long long seen_d = 0;
  for (int i = 0; i < a->n_dims; ++i) {
    GCC_REQUIRE(a->dims[i] >= 0 && a->dims[i] < Z && !((seen_d >> a->dims[i]) & 1ull),
                "gen_latent: dims must be distinct indices in [0, 45)");
    seen_d |= 1ull << a->dims[i];
  }
  GCC_REQUIRE(a->gate_ws && (a->z || a->z16) && (kinds == 0 || a->alphas), "gen_latent: null pointer");
  GCC_REQUIRE(a->mode == GCCVAE_GEN_GENERATE || (a->loc_pre && a->scale_pre && a->ld_pre >= 0),
              "gen_latent: reconstruct / intervene need loc_pre and scale_pre");
  GCC_REQUIRE(a->mode != GCCVAE_GEN_GENERATE || a->y_tgt, "gen_latent: generate needs y_tgt");
  GCC_REQUIRE(a->mode != GCCVAE_GEN_INTERVENE || a->y_tgt || a->n_labels > 0,
              "gen_latent: intervene needs y_tgt unless it walks labels");
  GCC_REQUIRE((uintptr_t)a->z % 4 == 0 && (uintptr_t)a->eps % 4 == 0 && (uintptr_t)a->alphas % 4 == 0 &&
                  (uintptr_t)a->loc_pre % 4 == 0 && (uintptr_t)a->scale_pre % 4 == 0 && (uintptr_t)a->y_tgt % 8 == 0 &&
                  (uintptr_t)a->y_src % 8 == 0 && (uintptr_t)a->y_src_out % 4 == 0 && (uintptr_t)a->z16 % 16 == 0,
              "gen_latent: misaligned pointer (fp32 / int32: 4 bytes, int64: 8, z16: 16)");
  GCC_CUDA(launch_aux(gen_latent_kernel, dim3(latent_grid(a->rows)), dim3(WARPS * 32), 0, (cudaStream_t)stream, *a));
  GCC_CHECK_LAUNCH("gen_latent");
  return GCCVAE_OK;
}

extern "C" int gccvae_iw_latent(const gccvae_iw_latent_args* a, void* stream) {
  GCC_REQUIRE(a, "iw_latent: null args");
  GCC_REQUIRE(a->batch > 0 && a->K >= 1 && a->kc >= 1 && a->k0 >= 0 && a->k0 + a->kc <= a->K,
              "iw_latent: bad sizes B=%d K=%d k0=%d kc=%d", a->batch, a->K, a->k0, a->kc);
  GCC_REQUIRE((long long)a->batch * a->kc < (1LL << 31), "iw_latent: too many rows");
  GCC_REQUIRE(a->loc_pre && a->scale_pre && a->ld_pre >= 0 && a->gate_ws && a->lw_part, "iw_latent: null pointer");
  GCC_REQUIRE(!a->labelled || a->y, "iw_latent: labelled needs y");
  GCC_REQUIRE((uintptr_t)a->z % 4 == 0 && (uintptr_t)a->eps % 4 == 0 && (uintptr_t)a->U_y % 4 == 0 &&
                  (uintptr_t)a->loc_pre % 4 == 0 && (uintptr_t)a->scale_pre % 4 == 0 && (uintptr_t)a->y % 8 == 0 &&
                  (uintptr_t)a->lw_part % 4 == 0 && (uintptr_t)a->z16 % 16 == 0,
              "iw_latent: misaligned pointer (fp32: 4 bytes, int64: 8, z16: 16)");
  const int rows = a->batch * a->kc;
  GCC_CUDA(launch_aux(iw_latent_kernel, dim3(latent_grid(rows)), dim3(WARPS * 32), 0, (cudaStream_t)stream, *a));
  GCC_CHECK_LAUNCH("iw_latent");
  return GCCVAE_OK;
}

extern "C" int gccvae_iw_accumulate(int batch, int kc, int k0, int K, const float* lw_part, const float* log_pxz,
                                    float* state, float* log_w, int first, int finalize, float* est, float* ess,
                                    void* stream) {
  GCC_REQUIRE(batch > 0 && kc >= 1 && k0 >= 0 && k0 + kc <= K, "iw_accumulate: bad sizes B=%d K=%d k0=%d kc=%d", batch,
              K, k0, kc);
  GCC_REQUIRE(lw_part && log_pxz && state && (!finalize || (est && ess)), "iw_accumulate: null pointer");
  GCC_CUDA(launch_aux(iw_accumulate_kernel, dim3((batch + 7) / 8), dim3(256), 0, (cudaStream_t)stream, batch, kc, k0,
                      K, lw_part, log_pxz, state, log_w, first, finalize, est, ess));
  GCC_CHECK_LAUNCH("iw_accumulate");
  return GCCVAE_OK;
}

extern "C" int gccvae_latent_bwd_partials(int batch) { return latent_grid(batch); }

extern "C" int gccvae_latent_bwd(const gccvae_latent_bwd_args* a, void* stream) {
  GCC_REQUIRE(a, "latent_bwd: null args");
  GCC_REQUIRE(a->batch > 0 && a->batch_global >= a->batch, "latent_bwd: bad batch");
  GCC_REQUIRE(a->loc_pre && a->scale_pre && a->y && a->gate_ws && a->terms && a->log_pxz && a->dz && a->partials,
              "latent_bwd: null pointer");
  GCC_REQUIRE((a->dloc_pre && a->dscale_pre) || a->dpre16, "latent_bwd: no destination for the head gradients");
  GCC_REQUIRE((a->db_loc == nullptr) == (a->db_scale == nullptr), "latent_bwd: db_loc and db_scale go together");
  GCC_REQUIRE((uintptr_t)a->eps_k % 8 == 0, "latent_bwd: eps_k must be 8-byte aligned");
  const int grid = latent_grid(a->batch);
  GCC_REQUIRE(a->n_partials == grid, "latent_bwd: n_partials must be %d", grid);
  const size_t smem = ((sizeof(GateSmem) + 15) / 16) * 16 + sizeof(BwdWarpSmem) * WARPS;
  static bool attr_done[2] = {false, false};
  if (a->supervised) {
    if (!attr_done[1]) {
      GCC_CUDA(cudaFuncSetAttribute(latent_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_done[1] = true;
    }
    GCC_CUDA(launch_aux(latent_bwd_kernel<true>, dim3(grid), dim3(WARPS * 32), smem, (cudaStream_t)stream, *a));
  } else {
    if (!attr_done[0]) {
      GCC_CUDA(cudaFuncSetAttribute(latent_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_done[0] = true;
    }
    GCC_CUDA(launch_aux(latent_bwd_kernel<false>, dim3(grid), dim3(WARPS * 32), smem, (cudaStream_t)stream, *a));
  }
  GCC_CHECK_LAUNCH("latent_bwd");
  return GCCVAE_OK;
}

extern "C" int gccvae_gate_bwd(float* partials, int n_partials, const float* mu, const float* Wcls,
                               const float* Wlt, const float* Wlf, const float* Wst, const float* Wsf,
                               const float* gate_ws, float gating_reg, float l1_scale, float* dWcls, float* dbcls,
                               float* dWlt, float* dWlf, float* dWst, float* dWsf, float* dmu, float* loss_inout,
                               void* stream) {
  GCC_REQUIRE(partials && n_partials > 0 && mu && Wcls && Wlt && Wlf && Wst && Wsf && gate_ws,
              "gate_bwd: null pointer");
  // row n_partials of the buffer receives the column sums (the caller allocates n_partials + 1 rows)
  float* reduced = partials + (size_t)n_partials * PT_TOTAL;
  // block ticket of the merged kernel: a spare slot of the gate workspace (zeroed by every gate_fwd launch and by the
  // kernel itself) - the workspace is caller-owned device memory, const only from the caller's point of view
  unsigned int* ticket = reinterpret_cast<unsigned int*>(const_cast<float*>(gate_ws)) + GW_B + 31;
  GCC_CUDA(launch_aux(reduce_gate_bwd_kernel, dim3((PT_TOTAL + 351) / 352), dim3(352), 0, (cudaStream_t)stream,
                      (const float*)partials, n_partials, reduced, ticket, mu, Wcls, Wlt, Wlf, Wst, Wsf, gate_ws,
                      gating_reg, l1_scale, dWcls, dbcls, dWlt, dWlf, dWst, dWsf, dmu, loss_inout));
  GCC_CHECK_LAUNCH("gate_bwd");
  return GCCVAE_OK;
}

extern "C" int gccvae_classifier_tiled_f32(const float* zt, long long sb, long long si, long long sj, int batch,
                                           const float* gates, const float* W, const float* bias, float* logits,
                                           void* stream) {
  GCC_REQUIRE(zt && gates && W && bias && logits && batch > 0, "classifier_tiled: bad args");
  const int n = batch * Y;
  classifier_tiled_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(zt, sb, si, sj, batch, gates, W, bias,
                                                                             logits);
  GCC_CHECK_LAUNCH("classifier_tiled");
  return GCCVAE_OK;
}

extern "C" int gccvae_cond_prior_tiled_f32(const float* yt, long long sb, long long sj, long long si, int batch,
                                           const float* c, const float* Wlt, const float* Wlf, const float* Wst,
                                           const float* Wsf, float* loc, float* scale, void* stream) {
  GCC_REQUIRE(yt && c && Wlt && Wlf && Wst && Wsf && loc && scale && batch > 0, "cond_prior_tiled: bad args");
  const int n = batch * ZC;
  cond_prior_tiled_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(yt, sb, sj, si, batch, c, Wlt, Wlf, Wst,
                                                                             Wsf, loc, scale);
  GCC_CHECK_LAUNCH("cond_prior_tiled");
  return GCCVAE_OK;
}

extern "C" int gccvae_gaussian_kl_f32(const float* lq, const float* sq, const float* lp, const float* sp, int batch,
                                      int dims, float* out, void* stream) {
  GCC_REQUIRE(lq && sq && out && batch > 0 && dims > 0, "gaussian_kl: bad args");
  gaussian_kl_kernel<<<(batch + 3) / 4, 128, 0, (cudaStream_t)stream>>>(lq, sq, lp, sp, batch, dims, out);
  GCC_CHECK_LAUNCH("gaussian_kl");
  return GCCVAE_OK;
}
