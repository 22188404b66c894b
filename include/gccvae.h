/* gccvae.h — C ABI of the B200-native Gated-CCVAE ELBO-step kernels (libgccvae.so).
 *
 * The reference (jabhinav/Semi-Supervised-Gated-LT-VAE) is a pure TensorFlow-2/Keras script with
 * NO plugin / FFI layer (SURVEY.md §8b): its boundary is the Python class API of gated_ccvae.py
 * and networks.py.  This header is the boundary a maintainer would bind underneath that API
 * (ctypes stub in INTEGRATION.md).  Every entry point cites the reference lines it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is DEVICE memory owned by the caller unless a
 *    parameter is documented as host memory; nothing is allocated inside the library;
 *  - all launches are asynchronous on `stream` (a cudaStream_t passed as void*);
 *  - return value: 0 on success, negative gccvae_status otherwise; gccvae_last_error() returns
 *    a thread-local message for the last failure on the calling thread;
 *  - activations are NHWC, fp32 ("f32" entry points) or bf16 ("bf16" entry points);
 *  - conv kernels are the Keras layouts: Conv2D [kh,kw,Cin,Cout], Conv2DTranspose
 *    [kh,kw,Cout,Cin], Dense [in,out].  Both conv layouts are [kh,kw,C_L,C_S] where L is the
 *    tensor with the LARGER spatial extent and S the smaller one, so one "relation" geometry
 *    describes a layer and three kernels (L->S, S->L, weight-gradient) cover forward, dgrad and
 *    wgrad of Conv2D, Conv2DTranspose and Dense alike.
 */
#ifndef GCCVAE_H
#define GCCVAE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCCVAE_ABI_VERSION 1

typedef enum {
  GCCVAE_OK = 0,
  GCCVAE_EINVAL = -1, /* bad shape / alignment / null pointer */
  GCCVAE_EARCH = -2,  /* device is not sm_100 */
  GCCVAE_ECUDA = -3,  /* CUDA runtime / driver error, see gccvae_last_error() */
  GCCVAE_ENOMEM = -4  /* caller-provided workspace too small */
} gccvae_status;

typedef enum { GCCVAE_ACT_NONE = 0, GCCVAE_ACT_RELU = 1, GCCVAE_ACT_SIGMOID = 2 } gccvae_act;
/* OR-ed into `act`: add the previous contents of the output (out = act(acc + bias + out)) */
#define GCCVAE_ACT_ACCUMULATE 0x100

/* dimensions fixed by the reference model (gated_ccvae.py:481,517-518; configs.py:10) */
#define GCCVAE_Z 45
#define GCCVAE_ZS 27
#define GCCVAE_ZC 18
#define GCCVAE_Y 18

int gccvae_abi_version(void);
const char* gccvae_last_error(void);
/* 0 if `device` is compute capability 10.x, GCCVAE_EARCH otherwise. */
int gccvae_arch_check(int device);
/* number of kernels launched by this library on the calling thread since the last reset */
long long gccvae_launch_count(void);
void gccvae_reset_launch_count(void);
/* a replayed CUDA graph launches the kernels that were counted while it was captured */
void gccvae_add_launch_count(long long n);

/* ---- layer relation ------------------------------------------------------------------------
 * S[n,oh,ow,cs] <-> L[n, stride*oh - pad + kh, stride*ow - pad + kw, cl] through W[kh,kw,cl,cs].
 *   Conv2D   (networks.py:11-15,21-29): L = input, S = output.
 *   Conv2DTranspose (networks.py:45-49,55-58): S = input, L = output.
 *   Dense    (networks.py:17-18,43): KH=KW=HL=WL=HS=WS=1.                                     */
typedef struct {
  int batch;
  int HL, WL, CL; /* large-spatial side */
  int HS, WS, CS; /* small-spatial side */
  int KH, KW, stride, pad;
} gccvae_geom;

/* S = act( gather(L) * W + bias ) [optionally * (mask > 0)]
 * = Conv2D / Dense forward, Conv2DTranspose dgrad.  bias, mask may be NULL. */
int gccvae_ls_f32(const gccvae_geom* g, const float* L, const float* W, const float* bias, int act,
                  const float* mask, float* S, void* stream);
/* L = act( scatter(S) * W^T + bias ) [optionally * (mask > 0)]
 * = Conv2DTranspose forward, Conv2D / Dense dgrad.  Supported: (KH=KW=4,stride 2,pad 1),
 * and any geometry with HS=WS=1, pad=0, stride=1 (Dense, conv5, conv1t). */
int gccvae_sl_f32(const gccvae_geom* g, const float* S, const float* W, const float* bias, int act,
                  const float* mask, float* L, void* stream);
/* dW[kh,kw,cl,cs] = sum_{n,oh,ow} gather(L) * S  = wgrad of all three layer kinds.
 * Deterministic split-K: workspace >= gccvae_wg_f32_workspace_bytes(g). */
size_t gccvae_wg_f32_workspace_bytes(const gccvae_geom* g);
int gccvae_wg_f32(const gccvae_geom* g, const float* L, const float* S, float* dW, void* workspace,
                  size_t workspace_bytes, void* stream);
/* out[c] = sum_r in[r*cols + c]   (bias gradients) */
size_t gccvae_colsum_f32_workspace_bytes(long long rows, int cols);
int gccvae_colsum_f32(const float* in, long long rows, int cols, float* out, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ---- bf16 tensor-core path (tcgen05 + TMEM + TMA), NHWC bf16 activations ------------------------------
 * Same relation as the f32 entry points; weights are pre-packed bf16 GEMM operands:
 *   which=0 "ls": [CS (padded to 16)][(kh,kw,cl)]      used by gccvae_ls_bf16
 *   which=1 "sl": k4/s2/p1: [4 phases][CL (padded to 16)][(th,tw,cs)]; 1x1-spatial S: W itself as bf16.
 * out_f32 != 0 stores the result as fp32 instead of bf16.                                           */
size_t gccvae_packed_weight_elems(const gccvae_geom* g, int which);
/* batched form of the packing entry points below: ONE launch for all layers of a step.
 * kind 0: "ls"; 1: "sl" phases (k4/s2/p1); 2: plain bf16 cast of taps*CL*CS values; 3: "c4" (see below);
 * 4/5: strided copy into a zero-padded bf16 / fp32 operand (the 45-wide dense layers padded to 64 / 96);
 * 6: "sl9" packing of the halo kernel; 7/8: x2 (space-to-depth) packing of a 3-channel k4/s2/p1 kernel,
 * 7 = [CS][(a,b)][(dy,dx,c4)] (gccvae_tap4_ls_bf16), 8 = [(dy,dx,c4)][(a,b)][CS] (gccvae_convt_recon_bf16);
 * 9: s2d packing [CS][(a,b)][(dy,dx,CL)] of a k4/s2/p1 kernel with CL input channels */
typedef struct {
  int kind, taps, CL, CS;
  const float* W;
  void* out;
  /* kinds 4 (bf16 out) / 5 (fp32 out): out[(row_off+r)*ld_out + col_off + k] = W[r*sr + k*sk], r < taps, k < CL */
  int sr, sk, ld_out, row_off, col_off, pad_;
} gccvae_pack_job;
int gccvae_pack_jobs_bf16(const gccvae_pack_job* jobs, int n_jobs, void* stream);
int gccvae_pack_weights_bf16(const gccvae_geom* g, const float* W, void* Wp_ls, void* Wp_sl, void* stream);
int gccvae_ls_bf16(const gccvae_geom* g, const void* L, const void* Wp_ls, const float* bias, int act,
                   const void* mask, void* S, int out_f32, void* stream);
int gccvae_sl_bf16(const gccvae_geom* g, const void* S, const void* Wp_sl, const float* bias, int act,
                   const void* mask, void* L, int out_f32, void* stream);
/* dW (fp32, Keras [kh,kw,cl,cs]) += gather(L)^T S; out[c] += column sums.  Accumulating: zero first. */
int gccvae_wg_bf16(const gccvae_geom* g, const void* L, const void* S, float* dW, void* stream);
/* out[c] += column sums of a bf16 [rows, cols] tensor for c < n_valid (0 = all) */
int gccvae_colsum_bf16(const void* in, long long rows, int cols, int n_valid, float* out, void* stream);
/* dense layers (networks.py:17-18 heads, :43 fc1, :45 conv1t as [B,45]x[45,2048]) with operands zero-padded
 * to tensor-core friendly widths:
 *   gemm:    out[rows,N] = act(A[rows,K] Wp[N,K]^T + bias[n % bias_mod], n < bias_n) (* mask > 0)
 *   gemm_tn: D[M,N] += A[rows,M]^T B[rows,N], scattered to 1-2 column segments of fp32 tensors */
typedef struct {
  int n_seg, m_valid;
  struct { int col0, ncols, ld, pad_; float* dst; } seg[2];
} gccvae_wg_out;
int gccvae_gemm_bf16(long long rows, int K, int N, const void* A, const void* Wp, const float* bias, int bias_n,
                     int bias_mod, int act, const void* mask, void* out, int out_f32, void* stream);
int gccvae_gemm_tn_bf16(long long rows, int M, int N, const void* A, const void* B, const gccvae_wg_out* out,
                        void* stream);
/* s2d storage of the stride-2 layers' L tensors (an H x W x C plane as (H/2+1) x (W/2+1) blocks of 2x2 pixels, block
 * (i,j) = pixels (2i-1+dy, 2j-1+dx) in slot dy*2+dx, zero outside): Conv2D(k4,s2,p1) forward, Conv2DTranspose dgrad and
 * their weight gradients gather 2x2 blocks of 4C channels (gccvae_tap4_ls_bf16 / gccvae_wg_s2d_bf16, weights packed
 * with kind 9) instead of 16 strided taps of C channels.  These flags are OR-ed into the `act` argument of
 * gccvae_ls_bf16 / gccvae_sl_bf16 / gccvae_sl_halo_bf16 / gccvae_tap4_ls_bf16 / gccvae_c3conv_bf16:            */
#define GCCVAE_OUT_S2D 0x10      /* store the (bf16, spatial) output in s2d block form                          */
#define GCCVAE_MASK_S2D 0x20     /* the mask tensor is stored in s2d block form                                 */
#define GCCVAE_TAP_HALO 0x40     /* gccvae_tap4_ls_bf16: two column-shifted boxes with a halo row instead of four boxes */
#define GCCVAE_LAYOUT_FLAGS 0x70
int gccvae_wg_s2d_bf16(int batch, int HS, int WS, int CL, const void* in2, const void* S, int CS, float* dW,
                       void* stream);
/* Space-to-depth ("x2") form of the 3-channel end layers (conv1 = networks.py:11,22; conv5t = :49,58; likelihood =
 * utils.py:101-105).  X2[n,i,j,(dy,dx,c4)] = x[n,2i-1+dy,2j-1+dx,c] (bf16 [B,33,33,16], zero outside the image
 * and in the pad channels - except element 15 of every block, which gccvae_prep_x2_bf16 sets to 1.0, see gccvae_tap4_wg_bf16):
 * Conv2D(k4,s2,p1) over the image is a 2x2-tap stride-1 GEMM over the blocks and Conv2DTranspose(k4,s2,same)
 * produces its output directly in block form.  x may be uint8 (0..255): it is divided by 255 on the device
 * exactly as utils_data.py:57-59 does on the host. */
/* XB (optional, uint8 images only): [B,33,33,16] uint8, the RAW bytes of every block (4 pixels x 3 channels + 4 zero
 * bytes, zero outside the image): the image operand of gccvae_convt_recon_bf16 with x_u8 = 2. */
int gccvae_prep_x2_bf16(const void* x, int x_u8, int batch, void* X2, void* XB, void* stream);
int gccvae_tap4_ls_bf16(int batch, int HB, int WB, int CB, const void* in2, const void* Wp, int CS, const float* bias,
                        int act, const void* mask, void* out, void* stream);
/* same contraction as gccvae_tap4_ls_bf16 for the 33x33x16 blocks of a 64x64x3 image, with the im2col tile built
 * by producer warps (TMA is row-rate bound on 32-byte rows): conv1 forward and conv5t dgrad.  CS in {32, 64}. */
int gccvae_c3conv_bf16(int batch, const void* in2, const void* Wp, int CS, const float* bias, int act, const void* mask,
                       void* out, void* stream);
/* db (optional; in2 must be blocks written by gccvae_prep_x2_bf16, whose element 15 is the constant 1): the bias gradient
 * db[cs] += sum over pixels of S - the ones row of the operand turns it into one more row of the same MMAs. */
int gccvae_tap4_wg_bf16(int batch, const void* in2, const void* S, int CS, float* dW, float* db, void* stream);
/* x_u8: 0 = x is the fp32 image [B,64,64,3], 1 = the uint8 image, 2 = the raw-byte blocks XB of gccvae_prep_x2_bf16 (one
 * 16-byte load per block instead of twelve 1-byte loads).
 * log_pxz_ready != 0: the caller has already set log_pxz[b] = -12288 ln 2 (gccvae_fill_f32), e.g. on a side stream */
int gccvae_convt_recon_bf16(int batch, const void* g4, const void* Wp8, const float* bias, const void* x, int x_u8,
                            const float* coef, float* log_pxz, void* D2, float* xhat, float* db, int log_pxz_ready,
                            void* stream);
int gccvae_fill_f32(float* p, long long n, float v, void* stream);
/* Image of the decoder (no counterpart in the reference: the generation path of gated_ccvae.py's Learner.generate /
 * reconstruct / intervene): conv5t forward (Conv2DTranspose 32 -> 3, k4, s2, same, networks.py:49,58) + sigmoid, with
 * nothing else - no likelihood, no gradient.
 *   g4: [B,32,32,32] bf16, the decoder's conv4t output (after ReLU); Wp8: pack kind 8 ([16][4][32] bf16); bias: [3].
 *   out: [B,64,64,3] NHWC, contiguous, 16-byte aligned;
 *        out_u8 = 0: fp32 sigmoid values xhat;
 *        out_u8 = 1: uint8 u = min(255, rint(255.0f * xhat)) (fp32 product, round half to even).
 *   The uint8 output is the fp32 output of the same call converted by that rule, bit for bit. */
int gccvae_convt_image_bf16(int batch, const void* g4, const void* Wp8, const float* bias, void* out, int out_u8,
                            void* stream);
/* One iteration of image completion (no counterpart in the reference: gated_ccvae.py's Learner.complete): conv5t forward
 * + sigmoid as gccvae_convt_image_bf16 computes it, written straight into the encoder's input blocks for the next
 * iteration instead of into an image.
 *   g4, Wp8, bias: as gccvae_convt_image_bf16.
 *   mask_blocks: [B,33,33] uint8, the pixel mask in x2 block form: bit dy * 2 + dx of block (i, j) is set when pixel
 *     (2i-1+dy, 2j-1+dx) is observed.  Bits of pixels outside the image are ignored.
 *   X2: [B,33,33,16] bf16 x2 blocks as gccvae_prep_x2_bf16 writes them (16-byte aligned), updated IN PLACE: every
 *     unobserved pixel gets bf16(xhat) in its three channel lanes (the bits gccvae_prep_x2_bf16 makes of the fp32 image
 *     that gccvae_convt_image_bf16 writes), and its pad lane is written with the value it already holds (0, or 1.0 in
 *     element 15).  Observed pixels are not written, and a block with no unobserved pixel is not stored at all, so
 *     nothing beyond the B x 1089 blocks - such as the raw-byte blocks XB that may follow them - is touched. */
int gccvae_convt_complete_bf16(int batch, const void* g4, const void* Wp8, const float* bias, const void* mask_blocks,
                               void* X2, void* stream);
/* Likelihood of K decoded rows per source image (no counterpart in the reference: the importance-weighted estimate of
 * gated_ccvae.py's Learner.log_likelihood): conv5t forward + sigmoid + the Laplace log-likelihood of utils.py:101-105,
 * with no gradient, no reconstruction and no bias gradient.
 *   g4: [rows,32,32,32] bf16, the decoder's conv4t output of `rows` decoded rows; Wp8, bias: as gccvae_convt_recon_bf16.
 *   Decoded row r is scored against source image r / kc (rows = B * kc, image-major).  x / x_u8 as for
 *   gccvae_convt_recon_bf16, over the B source images: 0 = fp32 [B,64,64,3], 1 = uint8 [B,64,64,3], 2 = the raw-byte
 *   blocks XB [B,33,33,16] of gccvae_prep_x2_bf16 (16-byte aligned).
 *   log_pxz [rows]: must hold -12288 ln 2 on entry (gccvae_fill_f32); -|x - xhat|_1 is added. */
int gccvae_convt_ll_bf16(int rows, int kc, const void* g4, const void* Wp8, const float* bias, const void* x, int x_u8,
                         float* log_pxz, void* stream);
/* S -> L "halo" kernel for 16x16 / 32x32 S planes with 32 or 64 channels and C_L <= 64: all four output-parity
 * phases per CTA from three column-shifted halo boxes (3.6x less L2 traffic than gccvae_sl_bf16), one MMA per
 * shifted view with N = 4*C_L.  Weights packed "sl9" = [9 views][4 phases][C_L padded to 16][C_S]
 * (gccvae_pack_jobs_bf16 kind 6; gccvae_packed_weight_elems(g, 2) elements). */
int gccvae_sl_halo_supported(const gccvae_geom* g);
int gccvae_sl_halo_bf16(const gccvae_geom* g, const void* S, const void* Wp_sl9, const float* bias, int act,
                        const void* mask, void* L, int out_f32, void* stream);
int gccvae_cast_f32_to_bf16(const float* in, long long n, void* out, void* stream);
int gccvae_cast_bf16_to_f32(const void* in, long long n, float* out, void* stream);

/* ---- gate (gated_ccvae.py:62-64,102-111; networks.py:72-74,83-86,104-106,118-127) ------------
 * One relaxed-Bernoulli sample c[18,18] per step from mu, shared by the batch and by all K
 * importance samples, plus the gated parameter products the latent kernels consume.
 * U1,U2: explicit uniforms [18,18], or NULL to draw them from Philox4x32-10(seed, offset [+ *step_dev]).
 * c_in (optional): use this c instead of sampling (classifier_loss(x,y,c), gated_ccvae.py:167); then
 * mu/U1/U2 are ignored and dc/dmu is zero.
 * temperature_dev (optional): device float that overrides `temperature` - the value is then read when the kernel runs,
 * so a captured CUDA graph of the step follows the per-epoch decay of gated_ccvae.py:404-406 without re-capture.
 * gate_ws: >= GCCVAE_GATE_WS_FLOATS floats: c | M=c*Wcls | bcls | P_lt | P_lf | P_st | P_sf | dc/dmu
 * (P_x[j,i] = c[i,j]*W_x[j,i]; dc/dmu is kept for gccvae_gate_bwd).  `c_out` (may be NULL) receives a copy of c. */
#define GCCVAE_GATE_WS_FLOATS (7 * 324 + 32)
int gccvae_gate_fwd(const float* mu, const float* c_in, const float* U1, const float* U2, uint64_t seed,
                    uint64_t offset, const int* step_dev, float temperature, const float* temperature_dev, const float* Wcls, const float* bcls, const float* Wlt,
                    const float* Wlf, const float* Wst, const float* Wsf, float* gate_ws, float* c_out,
                    void* stream);

/* ---- fused latent kernel (SURVEY.md A3,A6-A10,A12,A13) ------------------------------------------
 * forward: reparameterised z, gated classifier q(y|z_c,c), (sup) K-sample log q(y|x),
 * (unsup) label sampling, conditional prior p(z_c|y,c), KL, importance weight w.
 *   gated_ccvae.py:237-268,280-287 (sup), :187-218 (unsup), :167-182 (K loop);
 *   networks.py:17-18,33-34 (relu / clipped softplus of the posterior heads).              */
typedef struct {
  int batch;         /* images on this rank */
  int batch_global;  /* divisor of the mean (data parallel: sum of all ranks' batches) */
  int supervised;    /* 1: sup_loss, 0: unsup_loss */
  int K;             /* importance samples (gated_ccvae.py:167, k=100); ignored when unsup */
  /* inputs */
  const float* loc_pre;    /* [B,45] encoder locs head BEFORE relu */
  const float* scale_pre;  /* [B,45] encoder std head BEFORE softplus/clip */
  const long long* y;      /* [B,18] int64 labels (sup) */
  const float* eps;        /* [B,45] N(0,1) or NULL -> Philox */
  const float* eps_k;      /* [K,B,18] N(0,1) for the classify dims (cols 27: of the reference's
                              [K,B,45] draw) or NULL -> Philox */
  const float* U_y;        /* [B,18] uniforms (unsup) or NULL -> Philox */
  uint64_t seed, offset;   /* Philox key / per-step counter base */
  const int* step_dev;     /* optional device int added to `offset` (CUDA-graph replay) */
  const float* gate_ws;    /* from gccvae_gate_fwd */
  int ld_pre;              /* row stride (floats) of loc_pre / scale_pre; 0 = 45 */
  /* outputs */
  float* loc;    /* [B,45] */
  float* scale;  /* [B,45] */
  float* z;      /* [B,45] */
  float* terms;  /* [6,B]: kl | log_qy_zc | log_qy_x | w | log_py | coef_pxz (= -w/batch_global) */
  float* logits; /* [B,18] */
  int* y_out;    /* [B,18] int32 sampled labels (unsup) or copy of y (sup); may be NULL */
  void* z16;     /* optional bf16 [B,64] copy of z, columns 45..63 zero (operand of the tensor-core fc1) */
} gccvae_latent_fwd_args;
int gccvae_latent_fwd(const gccvae_latent_fwd_args* a, void* stream);

/* backward of the same: consumes dz (from the decoder) and log_pxz, produces the gradients of
 * the two encoder heads' pre-activations and per-CTA partial sums of the small parameters,
 * which gccvae_gate_bwd reduces.  (gradient routes: SURVEY.md §8a "Gradient routes") */
#define GCCVAE_LATENT_PARTIAL_FLOATS (5 * 324 + 32)
typedef struct {
  int batch, batch_global, supervised, K;
  const float* loc_pre;
  const float* scale_pre;
  const int* y;          /* [B,18] int32 labels as written to y_out by the forward */
  const float* eps;
  const float* eps_k;
  uint64_t seed, offset;
  const int* step_dev;
  const float* gate_ws;
  const float* terms;    /* [6,B] from the forward */
  const float* log_pxz;  /* [B] */
  const float* dz;       /* [B,45] dLoss/dz from the decoder */
  float* dloc_pre;       /* [B,45] (may be NULL when dpre16 is given) */
  float* dscale_pre;     /* [B,45] */
  int ld_pre, ld_dz;     /* row strides (floats) of loc_pre/scale_pre and of dz; 0 = 45 */
  void* dpre16;          /* optional bf16 [B,96]: dloc_pre at cols 0..44, dscale_pre at 48..92, rest zero */
  float* db_loc;         /* optional [45] += column sums of dloc_pre (bias gradient of the locs head) */
  float* db_scale;       /* optional [45] += column sums of dscale_pre */
  float* partials;       /* [n_partials + 1, GCCVAE_LATENT_PARTIAL_FLOATS] (last row: scratch of gate_bwd) */
  int n_partials;        /* = gccvae_latent_bwd_partials(batch) */
  float* loss_out;       /* [1]: sum_b -(elbo_b)/batch_global for this rank (no L1 term) */
} gccvae_latent_bwd_args;
int gccvae_latent_bwd_partials(int batch);
int gccvae_latent_bwd(const gccvae_latent_bwd_args* a, void* stream);

/* ---- latent code of the forward-only image calls (no counterpart in the reference) -----------------------------
 * One warp per frame writes the z the decoder turns into an image.  Every image has F frames, of at most one kind:
 *   one frame (n_labels = n_dims = pair = 0): F = 1;
 *   label walk: F = n_labels * n_alpha, frame (l, t) of image b being row r = (b * n_labels + l) * n_alpha + t, which
 *     walks label labels[l] to the real value alphas[t] in the target prior and keeps the other 17 labels;
 *   latent traversal: F = n_dims * n_alpha, frame (d, t) of image b being row r = (b * n_dims + d) * n_alpha + t: the
 *     mode's z with z_{dims[d]} set to alphas[t] (an absolute value); every other dim keeps the one-frame call's bits;
 *   pair interpolation (RECONSTRUCT, sample = 0 only): B pairs, F = n_alpha, frame t of pair b being row r = b * n_alpha
 *     + t: with z_a, z_b the posterior means of rows b and B + b of loc_pre, z = z_a outside [mix_lo, mix_hi) and inside
 *     it z_a at t = 0, z_b at t = 1, fmaf(t, z_b - z_a, z_a) otherwise (t = alphas[t], any finite value).  Notation: c is
 * the gate sample of gate_ws (gccvae_gate_fwd); loc_p(y,c), scale_p(y,c) are the conditional prior of
 * networks.py:118-127 (scale after softplus and the [1e-3, 1e3] clip); eps [B,45] is N(0,1) with the layout of
 * gccvae_latent_fwd (columns 0..26 style dims, 27..44 classify dims).  Labels are nonzero -> 1.
 *   GCCVAE_GEN_GENERATE:     z_s = eps_s, z_c = loc_p(y_tgt,c) + scale_p(y_tgt,c) eps_c;
 *                            sample = 0: z_s = 0, z_c = loc_p(y_tgt,c).
 *   GCCVAE_GEN_RECONSTRUCT:  z = loc (posterior mean: relu / clipped softplus of the heads, networks.py:17-18,33-34);
 *                            sample = 1: z = loc + scale eps.  No prior step; a walk is rejected.
 *   GCCVAE_GEN_INTERVENE:    z as for RECONSTRUCT, then the classify dims move from y_src to y_tgt by the Gaussian
 *                            counterfactual  e = (z_c - loc_p(y_src,c)) / scale_p(y_src,c),
 *                            z_c' = z_c + (loc_p(y_tgt,c) - loc_p(y_src,c)) + (scale_p(y_tgt,c) - scale_p(y_src,c)) e
 *                            (y_src == y_tgt leaves z_c bit-identical); z_s is never touched.  y_src = NULL: the
 *                            classifier's decision on z_c, sigmoid(logit) > 0.5 (as gccvae_accuracy_f32 decides).
 *                            y_tgt = NULL: y_tgt = y_src, valid only in a walk.
 * In a walk the target prior is the prior at y_tgt with y_tgt,l replaced by alpha.  Its term of label l is exactly the
 * boolean term at alpha = 0 and alpha = 1 and fmaf(alpha, P_true - P_false, P_false) otherwise, summed in the order of
 * the prior (j = 0..17).  So a frame at alpha in {0, 1} is bit for bit the one-frame call of the same mode whose y_tgt
 * has y_tgt,l = alpha, and (INTERVENE, y_tgt = NULL) the frame at alpha = y_src,l is RECONSTRUCT's z.
 * Any finite alpha is valid (beyond [0, 1] the prior extrapolates).
 * Only RECONSTRUCT and INTERVENE read loc_pre / scale_pre; only GENERATE and INTERVENE read y_tgt; eps is read only when
 * sampling (eps = NULL: the Philox stream of gccvae_latent_fwd, which gccvae_draw_noise_f32 kind 0 reproduces).  Noise
 * is drawn once per image (image b, dim d) and shared by all its frames.  The rows row0 .. row0 + rows - 1 are written
 * at z / z16 rows 0 .. rows - 1 (one chunk of the decoder; one-frame calls pass row0 = 0, rows = B); y_src_out rows are
 * written by the chunk that holds the image's first frame. */
#define GCCVAE_GEN_GENERATE 1
#define GCCVAE_GEN_RECONSTRUCT 2
#define GCCVAE_GEN_INTERVENE 3
typedef struct {
  int batch;               /* B images */
  int mode;                /* GCCVAE_GEN_* */
  int sample;              /* 0: means, 1: draw with eps (see above) */
  int ld_pre;              /* row stride (floats) of loc_pre / scale_pre; 0 = 45 */
  int n_labels;            /* labels walked, 0..18 (0: one frame per image) */
  int labels[18];          /* labels[0 .. n_labels-1]: distinct label indices in [0, 18), in row order */
  int n_alpha;             /* values per walked label / traversed dim / pair, >= 1 (walk, traversal, pair) */
  const float* alphas;     /* [n_alpha] device fp32, finite (walk, traversal, pair) */
  int row0, rows;          /* this chunk: rows row0 .. row0 + rows - 1 of the B * F */
  const float* loc_pre;    /* [B,45] encoder locs head BEFORE relu (RECONSTRUCT, INTERVENE) */
  const float* scale_pre;  /* [B,45] encoder std head BEFORE softplus/clip */
  const long long* y_tgt;  /* [B,18] int64 target labels (GENERATE; INTERVENE, or NULL in a walk) */
  const long long* y_src;  /* [B,18] int64 source labels (INTERVENE) or NULL */
  const float* eps;        /* [B,45] N(0,1) or NULL -> Philox */
  uint64_t seed, offset;   /* Philox key / counter base */
  const int* step_dev;     /* optional device int added to `offset` */
  const float* gate_ws;    /* from gccvae_gate_fwd */
  /* outputs (at least one of z, z16) */
  float* z;                /* optional [rows,45] fp32 (operand of the fp32 decoder) */
  void* z16;               /* optional bf16 [rows,64] copy of z, columns 45..63 zero (operand of the tensor-core fc1) */
  int* y_src_out;          /* optional [B,18] int32: the y_src used (INTERVENE) */
  /* latent traversal (any mode) */
  int n_dims;              /* latent dims traversed, 0..45 (0: no traversal) */
  int dims[45];            /* dims[0 .. n_dims-1]: distinct indices in [0, 45), in row order */
  /* pair interpolation (RECONSTRUCT, sample = 0) */
  int pair;                /* 1: loc_pre / scale_pre hold 2B rows, image b's partner at row B + b */
  int mix_lo, mix_hi;      /* the dims [mix_lo, mix_hi) that move; 0 <= mix_lo < mix_hi <= 45 */
} gccvae_gen_latent_args;
int gccvae_gen_latent(const gccvae_gen_latent_args* a, void* stream);

/* ---- importance-weighted log-likelihood (no counterpart in the reference) -------------------------------------
 * log p(x [, y]) >= log p_hat = logsumexp_k log w_k - ln K over K samples per image, with proposal q(z|x) (labelled) or
 * q(z|x) q(y|z_c) (unlabelled) and the gate sample c of gate_ws:
 *   z_k = loc + scale eps_k (eps_k [45]: columns 0..26 style dims, 27..44 classify dims, as gccvae_latent_fwd);
 *   y_k = y (labelled) or [U_k < sigmoid(logit(z_c,k))] (unlabelled, U_k [18] uniform: the rule of gated_ccvae.py:206);
 *   log w_k = log p(x|z_k) + log p(z_s) + log p(z_c,k|y_k) + log p(y_k) - log q(z_k|x) [- log q(y_k|z_c,k) unlabelled]
 * with N(0,1) style prior, the conditional prior of networks.py:118-127, log p(y) = 18 ln 0.5, log q(z|x) computed from
 * eps_k itself (not from (z - loc) / scale) and log p(x|z) = the Laplace likelihood of utils.py:101-105.
 *
 * The K samples are processed in chunks of kc samples per image; rows of a chunk are image-major, r = b * kc + j for
 * sample k0 + j of image b.  The Philox draws of (image b, sample k) depend on (seed, offset, b, k) only - never on the
 * chunking or on B - and gccvae_draw_noise_f32 kinds 4 / 5 reproduce them.
 *
 * gccvae_iw_latent: one warp per row; writes the decoder operand of every row of the chunk and lw_part[row] = every
 * term of log w_k except log p(x|z_k). */
typedef struct {
  int batch;               /* B source images */
  int K;                   /* samples per image of the whole estimate (the explicit noise is [K,B,...]) */
  int k0, kc;              /* this chunk: samples k0 .. k0 + kc - 1 of every image, rows = B * kc */
  int labelled;            /* 1: y given; 0: y_k drawn from the classifier */
  int ld_pre;              /* row stride (floats) of loc_pre / scale_pre; 0 = 45 */
  const float* loc_pre;    /* [B,45] encoder locs head BEFORE relu */
  const float* scale_pre;  /* [B,45] encoder std head BEFORE softplus/clip */
  const long long* y;      /* [B,18] int64 labels, nonzero = 1 (labelled) */
  const float* eps;        /* [K,B,45] N(0,1) or NULL -> Philox */
  const float* U_y;        /* [K,B,18] uniforms (unlabelled) or NULL -> Philox */
  uint64_t seed, offset;   /* Philox key / counter base */
  const int* step_dev;     /* optional device int added to `offset` */
  const float* gate_ws;    /* from gccvae_gate_fwd */
  /* outputs */
  float* lw_part;          /* [rows] */
  float* z;                /* optional [rows,45] fp32 (operand of the fp32 decoder) */
  void* z16;               /* optional bf16 [rows,64], columns 45..63 zero (operand of the tensor-core fc1) */
} gccvae_iw_latent_args;
int gccvae_iw_latent(const gccvae_iw_latent_args* a, void* stream);
/* Online log-sum-exp over the chunks: for every image b the chunk's log w = lw_part[r] + log_pxz[r] of its kc rows
 * r = b * kc + j is folded into state[b] = {max m, sum e^(lw - m), sum e^(2 (lw - m))} (first != 0: the state is
 * started, not read).  log_w (optional): [K,B], log_w[k0 + j][b] = log w.  finalize != 0 (the last chunk):
 * est[b] = m + ln(sum e^(lw - m)) - ln K and ess[b] = (sum w)^2 / sum w^2. */
int gccvae_iw_accumulate(int batch, int kc, int k0, int K, const float* lw_part, const float* log_pxz, float* state,
                         float* log_w, int first, int finalize, float* est, float* ess, void* stream);

/* reduce the partials; chain through c to mu (clip / pow / ratio of gated_ccvae.py:103-109) and
 * add the L1 term gating_reg*mean|mu| (gated_ccvae.py:229-230,297-298) scaled by l1_scale
 * (1/world in data parallel).  d* may be NULL when the tensor is frozen.
 * One launch: every block reduces a slice of the partial rows, the block that draws the last ticket forms the
 * gradients.  The ticket is float slot 2*324 + 31 of gate_ws (a spare slot of the bias row): gccvae_gate_fwd zeroes it
 * on every launch and this kernel leaves it at zero, so gate_ws must come from gccvae_gate_fwd (or be zero-filled). */
int gccvae_gate_bwd(float* partials /* [n_partials + 1 rows]: the last row is scratch */, int n_partials, const float* mu, const float* Wcls,
                    const float* Wlt, const float* Wlf, const float* Wst, const float* Wsf,
                    const float* gate_ws, float gating_reg, float l1_scale, float* dWcls, float* dbcls,
                    float* dWlt, float* dWlf, float* dWst, float* dWsf, float* dmu, float* loss_inout,
                    void* stream);

/* ---- fused dense chain (bf16 engine): everything between the encoder's last convolution and the decoder's first
 * transposed convolution is row-local, so ONE launch each way carries groups of gccvae_chain_rows(batch) images
 * through it (csrc/chain.cu):
 *   forward:  h5 -> heads (networks.py:17-18,31-34) -> the whole of gccvae_latent_fwd -> fc1 + ReLU (networks.py:43,52)
 *             -> conv1t + ReLU (networks.py:45,54);
 *   backward: conv1t dgrad -> ReLU mask -> fc1 dgrad -> the whole of gccvae_latent_bwd -> heads dgrad -> ReLU mask,
 *             plus the bias gradients of conv1t / fc1 / the heads / conv5 (accumulated with atomics: the buffers must
 *             be zero or hold partial sums) and the per-CTA partial rows gccvae_gate_bwd reduces.
 * Weight operands are the packed bf16 matrices of gccvae_pack_jobs_bf16 ([out feature][k], k contiguous, zero padded);
 * activations between the layers are bf16 as on the tensor-core path, everything else fp32.  Noise, seeds, `terms`,
 * `partials` as for the latent kernels; n_partials must equal gccvae_chain_partials(batch). */
typedef struct {
  int batch, batch_global, supervised, K;
  int rows_per_cta;          /* set by the library */
  int pad_;
  const void* h5;            /* bf16 [B,256] conv5 output (after ReLU) */
  const void* w_heads;       /* bf16 [96][256]: rows 0..44 locs, 48..92 std */
  const float* b_heads;      /* [96] (same row layout, pads zero) */
  const void* w_fc1;         /* bf16 [64][64]  [out][in] */
  const float* b_fc1;        /* [45] */
  const void* w_conv1t;      /* bf16 [2048][64] [(kh,kw,co)][ci] */
  const float* b_conv1t;     /* [128] */
  const long long* y;        /* [B,18] int64 labels (sup) */
  const float* eps;          /* [B,45] or NULL -> Philox */
  const float* eps_k;        /* [K,B,18] or NULL -> Philox */
  const float* U_y;          /* [B,18] or NULL -> Philox */
  uint64_t seed, offset;
  const int* step_dev;
  const float* gate_ws;
  float* pre;                /* [B,96] heads' pre-activations: locs at 0..44, std at 48..92 */
  float* loc;                /* [B,45] */
  float* scale;              /* [B,45] */
  float* z;                  /* [B,45] */
  float* terms;              /* [6,B] */
  float* logits;             /* [B,18] */
  int* y_out;                /* [B,18] or NULL */
  void* z16;                 /* bf16 [B,64] */
  void* g0;                  /* bf16 [B,64]  fc1 output (45 real columns) */
  void* g1;                  /* bf16 [B,2048] conv1t output = [B,4,4,128] */
} gccvae_chain_fwd_args;
int gccvae_chain_rows(int batch);
int gccvae_chain_partials(int batch);
int gccvae_chain_fwd(const gccvae_chain_fwd_args* a, void* stream);

typedef struct {
  int batch, batch_global, supervised, K;
  int rows_per_cta;          /* set by the library */
  int n_partials;
  const void* dg1;           /* bf16 [B,2048] gradient of conv1t's pre-activation */
  const void* g0;            /* bf16 [B,64] fc1 output */
  const void* h5;            /* bf16 [B,256] conv5 output */
  const float* pre;          /* [B,96] from the forward */
  const int* y;              /* [B,18] labels used by the forward (y_out) */
  const float* eps;
  const float* eps_k;
  uint64_t seed, offset;
  const int* step_dev;
  const float* gate_ws;
  const float* terms;        /* [6,B] from the forward */
  const float* log_pxz;      /* [B] */
  const void* w_conv1t_t;    /* bf16 [64][2048]  [ci][(kh,kw,co)] */
  const void* w_fc1_t;       /* bf16 [64][64]  [in][out] */
  const void* w_heads_t;     /* bf16 [256][96] */
  void* dg0;                 /* bf16 [B,64] gradient of fc1's pre-activation */
  void* dpre16;              /* bf16 [B,96] gradient of the heads' pre-activations */
  void* dh5;                 /* bf16 [B,256] gradient of conv5's pre-activation */
  float* partials;           /* [n_partials + 1, GCCVAE_LATENT_PARTIAL_FLOATS] */
  float* db_loc;             /* [45] += (optional, with db_scale) */
  float* db_scale;
  float* db_fc1;             /* [45] += (optional) */
  float* db_conv1t;          /* [128] += (optional) */
  float* db_conv5;           /* [256] += (optional) */
} gccvae_chain_bwd_args;
int gccvae_chain_bwd(const gccvae_chain_bwd_args* a, void* stream);


/* ---- reconstruction log-likelihood (utils.py:101-105) ---------------------------------------------
 * log_pxz[b] = -sum|x - xhat| - 12288 ln2; optionally also the gradient w.r.t. the decoder's
 * pre-sigmoid logits, dlogit = coef[b] * sign(x - xhat) * xhat (1 - xhat). */
int gccvae_recon_f32(const float* x, const float* xhat, int batch, int per_image, const float* coef,
                     float* log_pxz, float* dlogit, void* stream);

/* ---- Keras-2.8 Adam on the flat parameter buffer (gated_ccvae.py:144,310) ---------------------------
 * theta -= lr*sqrt(1-b2^t)/(1-b1^t) * m/(sqrt(v)+eps); `step` is t (1-based).  If `step_dev`
 * (device int) is given it is incremented first and used as t, so a captured CUDA graph of the
 * whole step can be replayed. */
int gccvae_adam_f32(float* param, const float* grad, float* m, float* v, long long n, float lr,
                    float beta1, float beta2, float eps, int step, int* step_dev, void* stream);

/* The same update as ONE launch for the replayed step: t = step_state[0] + 1 is used; grad[i0..n_zero) is cleared
 * behind the read (n_zero >= n), so the next backward pass accumulates into a clean buffer without a memset.  Elements
 * [i0, n) are updated.  publish != 0: step_state[0] = t when the kernel ends.  A step may therefore run the update in
 * two launches over disjoint ranges - the second one publishing - e.g. everything but the first layer while the last
 * dgrad is still running.  step_state: 2 device ints {t, 0}; the second is the block ticket of the publishing launch
 * and must be 0 on entry (it is left at 0).
 * result_ring (optional, with publish): ring_slots rows of GCCVAE_RESULT_SLOT_FLOATS floats; the publishing launch
 * copies {result_loss[0], result_c[0..324)} into row (t - 1) % ring_slots, so that what train_step hands back
 * (gated_ccvae.py:311 returns fresh tensors) is not overwritten by the next replay of the same captured step. */
#define GCCVAE_RESULT_SLOT_FLOATS 328
int gccvae_adam_fused_f32(float* param, float* grad, float* m, float* v, long long i0, long long n, long long n_zero,
                          float lr, float beta1, float beta2, float eps, int* step_state, int publish,
                          const float* result_loss, const float* result_c, float* result_ring, int ring_slots,
                          void* stream);

/* Data parallel: two-shot all-reduce (sum over the ranks of one node) of grad[i0..n) over NVLink peer memory, fused with
 * the same Adam update as gccvae_adam_fused_f32 on the result (csrc/dp.cu).  grad[q] / sync[q] are rank q's gradient
 * buffer and its block of GCCVAE_DP_SYNC_WORDS zero-initialised 32-bit words, both in memory every rank of the node
 * can address (torch.distributed._symmetric_memory); every rank must issue the same sequence of calls.  loss_index >= 0:
 * grad[q][loss_index] is summed over the ranks too (into this rank's slot and, with publish, into the result ring).
 * The range bounds i0, n, n_zero must be multiples of 4 elements. */
#define GCCVAE_DP_MAX_RANKS 16
#define GCCVAE_DP_SYNC_WORDS 32
typedef struct {
  int world, rank;
  float* grad[GCCVAE_DP_MAX_RANKS];
  void* sync[GCCVAE_DP_MAX_RANKS];
  float* param;
  float* m;
  float* v;
  long long i0, n, n_zero;
  long long loss_index;
  float lr, beta1, beta2, eps;
  int* step_state;
  int publish;
  int ring_slots;
  const float* result_loss;
  const float* result_c;
  float* result_ring;
  /* push != 0: the one-barrier variant for a short range - every rank pushes grad[i0..n) (+ the loss) into slot `rank`
   * of every rank's receive buffer recv[q] (world slots of recv_stride >= n - i0 + 4 floats each, peer-addressable like
   * grad) and sums its own slots after the barrier.  Between two push calls every rank must issue a two-barrier call. */
  int push;
  int pad_;
  long long recv_stride;
  float* recv[GCCVAE_DP_MAX_RANKS];
} gccvae_dp_args;
int gccvae_dp_reduce_adam_f32(const gccvae_dp_args* a, void* stream);

/* loss[0] = sum_b(-elbo_b)/batch_global (+ gating_reg*mean|mu| when mu != NULL): the forward-only
 * value of sup_loss / unsup_loss (gated_ccvae.py:225-230, 291-298). */
int gccvae_elbo_loss_f32(const float* terms, const float* log_pxz, int batch, int batch_global,
                         int supervised, const float* mu, float gating_reg, float* loss, void* stream);

/* networks.py:17-18,33-34: loc = relu(loc_pre), scale = clip(softplus(scale_pre), 1e-3, 1e3). */
int gccvae_head_act_f32(const float* loc_pre, const float* scale_pre, long long n, float* loc, float* scale,
                        void* stream);
/* gated_ccvae.py:436-445: out[0] = mean( round(sigmoid(logits)) == y ), y int64, n = B*18. */
int gccvae_accuracy_f32(const float* logits, const long long* y, int n, float* out, void* stream);

/* test/debug aid: write the noise the kernels would draw in Philox mode.
 * kind 0: eps [B,45]; 1: eps_k [K,B,18]; 2: U_y [B,18]; 3: U1|U2 [2,18,18];
 * 4: eps [K,B,45] and 5: U_y [K,B,18] of gccvae_iw_latent. */
int gccvae_draw_noise_f32(int kind, uint64_t seed, uint64_t offset, int batch, int K, float* out, void* stream);

/* ---- tiled module API (networks.py:72-74,83-86,104-106,118-127) --------------------------------------
 * logits[b,j] = sum_i zt[b,i,j]*gates[i,j]*W[i,j] + bias[j];  zt strides allow broadcasting. */
int gccvae_classifier_tiled_f32(const float* zt, long long sb, long long si, long long sj, int batch,
                                const float* gates, const float* W, const float* bias, float* logits,
                                void* stream);
/* (loc,scale)[b,i] from tiled y[b,j,i], c[i,j] and the four [j,i] kernels. */
int gccvae_cond_prior_tiled_f32(const float* yt, long long sb, long long sj, long long si, int batch,
                                const float* c, const float* Wlt, const float* Wlf, const float* Wst,
                                const float* Wsf, float* loc, float* scale, void* stream);
/* sum_d KL(N(lq,sq) || N(lp,sp)) over `dims` (utils.py:108-119); lp/sp may be NULL (0 / 1). */
int gccvae_gaussian_kl_f32(const float* lq, const float* sq, const float* lp, const float* sp, int batch,
                           int dims, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GCCVAE_H */
