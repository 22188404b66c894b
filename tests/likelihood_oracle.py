"""CPU restatement of the importance-weighted log-likelihood (Learner.log_likelihood) over the oracle's networks.
TEST INFRASTRUCTURE ONLY.  The estimate has no counterpart in the reference; it is written here from the oracle's
`encoder`, `decoder`, `classifier` and `cond_prior` (so it runs in fp32 and fp64 and, under `O.bf16_emulation()`,
rounds where the kernels do: `decoder` rounds z through `_w16` like the bf16 engine's z16 operand, while the density
terms use the unrounded z, as the latent kernel does).

Noise is explicit: eps [K,B,45] (style dims 0..26, classify dims 27..44) and, unlabelled, U_y [K,B,18]."""
import math

import torch

import gccvae_oracle as O
import generation_oracle as GO

HALF_LN_2PI = 0.5 * math.log(2.0 * math.pi)


def log_weight_terms(p, x, c, eps, y=None, U_y=None, decode=True):
    """-> dict of [K,B] tensors: every term of log w_k and log_w itself.  y [B,18] (labelled) or None (y_k drawn from
    the classifier with U_y, as unsup_loss draws y).  decode=False leaves log p(x|z) out (log_pxz = 0)."""
    locs, scale = O.encoder(p, x)
    K, B = eps.shape[0], eps.shape[1]
    z = locs.unsqueeze(0) + scale.unsqueeze(0) * eps                        # [K,B,45]
    zs, zc = z[..., :O.Z_STYLE], z[..., O.Z_STYLE:]
    log_q = (-0.5 * eps ** 2 - torch.log(scale).unsqueeze(0)).sum(-1) - O.Z_DIM * HALF_LN_2PI
    log_pzs = (-0.5 * zs ** 2).sum(-1) - O.Z_STYLE * HALF_LN_2PI
    zc_flat = zc.reshape(K * B, O.Z_CLASSIFY)
    logits = O.classifier(p, zc_flat.unsqueeze(-1).repeat(1, 1, O.Y_DIM), c)
    if y is None:
        yk = O.bernoulli_sample(logits, U_y.reshape(K * B, O.Y_DIM)).to(torch.int64)
    else:
        yk = (y != 0).to(torch.int64).repeat(K, 1)
    log_qy = O.bernoulli_logits_log_prob(logits, yk).sum(-1).reshape(K, B)
    loc_p, scale_p = GO.prior(p, yk, c)
    t = (zc_flat - loc_p) / scale_p
    log_pzc = (-0.5 * t ** 2 - torch.log(scale_p)).sum(-1).reshape(K, B) - O.Z_CLASSIFY * HALF_LN_2PI
    log_py = torch.full((K, B), O.Y_DIM * math.log(0.5), dtype=z.dtype, device=z.device)
    if decode:
        xhat = O.decoder(p, z.reshape(K * B, O.Z_DIM))
        log_pxz = O.img_log_likelihood(xhat, x.repeat(K, 1, 1, 1)).reshape(K, B)
    else:
        log_pxz = torch.zeros(K, B, dtype=z.dtype, device=z.device)
    log_w = log_pxz + log_pzs + log_pzc + log_py - log_q - (log_qy if y is None else 0.0)
    return dict(log_w=log_w, log_pxz=log_pxz, log_pzs=log_pzs, log_pzc=log_pzc, log_py=log_py, log_q=log_q,
                log_qy=log_qy, y=yk.reshape(K, B, O.Y_DIM), z=z, logits=logits.reshape(K, B, O.Y_DIM))


def estimate(log_w):
    """[K,B] -> (log p_hat [B], effective sample size [B])."""
    K = log_w.shape[0]
    est = torch.logsumexp(log_w, dim=0) - math.log(K)
    ess = torch.exp(2.0 * torch.logsumexp(log_w, dim=0) - torch.logsumexp(2.0 * log_w, dim=0))
    return est, ess


def log_likelihood(p, x, c, eps, y=None, U_y=None):
    """-> (log p_hat [B], ess [B], log_w [K,B])."""
    lw = log_weight_terms(p, x, c, eps, y, U_y)["log_w"]
    est, ess = estimate(lw)
    return est, ess, lw
