"""CPU restatement of the generation path (Learner.generate / reconstruct / intervene) over the oracle's networks.
TEST INFRASTRUCTURE ONLY.  The three calls have no counterpart in the reference; they are written here from
the oracle's `encoder`, `decoder`, `cond_prior` and `classifier` (so they run in fp32 and fp64 and, under
`O.bf16_emulation()`, round where the kernels do: `decoder` rounds z through `_w16` like the bf16 engine's z16 operand).

Noise is explicit: eps [B,45] (style dims 0..26, classify dims 27..44), or None for the means."""
import numpy as np
import torch

import gccvae_oracle as O


def prior(p, y, c):
    """(loc_p, scale_p) [B,18] of the conditional prior for labels y [B,18] (nonzero = 1) and gate c [18,18]."""
    y_tiled = (y != 0).to(c.dtype).unsqueeze(-1).repeat(1, 1, O.Z_CLASSIFY)
    return O.cond_prior(p, y_tiled, c)


def generate(p, y, c, eps=None):
    """-> (image, z): z_s = eps_s, z_c = loc_p(y,c) + scale_p(y,c) eps_c; eps=None: z_s = 0, z_c = loc_p(y,c)."""
    loc_p, scale_p = prior(p, y, c)
    if eps is None:
        z = torch.cat([torch.zeros(y.shape[0], O.Z_STYLE, dtype=c.dtype), loc_p], dim=-1)
    else:
        z = torch.cat([eps[:, :O.Z_STYLE], loc_p + scale_p * eps[:, O.Z_STYLE:]], dim=-1)
    return O.decoder(p, z), z


def _posterior_z(p, x, eps):
    locs, scale = O.encoder(p, x)
    return locs if eps is None else O.sample_normal(locs, scale, eps)


def reconstruct(p, x, eps=None):
    """-> (image, z): z = posterior mean; with eps: z = loc + scale eps."""
    z = _posterior_z(p, x, eps)
    return O.decoder(p, z), z


def decision(p, zc, c):
    """the classifier's labels for z_c: sigmoid(logit) > 0.5 (and the logits)."""
    logits = O.classifier(p, zc.unsqueeze(-1).repeat(1, 1, O.Y_DIM), c)
    return (torch.sigmoid(logits) > 0.5).to(torch.int64), logits


def intervene(p, x, y_new, c, y=None, eps=None):
    """-> (image, z', y_src): z as in `reconstruct`, classify dims moved from y (default: the classifier's decision) to
    y_new by e = (z_c - loc_p(y)) / scale_p(y), z_c' = z_c + (loc_p(y_new) - loc_p(y)) + (scale_p(y_new) - scale_p(y)) e."""
    z = _posterior_z(p, x, eps)
    zc = z[:, O.Z_STYLE:]
    if y is None:
        y, _ = decision(p, zc, c)
    ls, ss = prior(p, y, c)
    lt, st = prior(p, y_new, c)
    e = (zc - ls) / ss
    z2 = torch.cat([z[:, :O.Z_STYLE], zc + (lt - ls) + (st - ss) * e], dim=-1)
    return O.decoder(p, z2), z2, (y != 0).to(torch.int64)


def to_u8(xhat):
    """min(255, rint(255 x)) with the product and the rounding in fp32 (numpy: half to even)."""
    v = np.float32(255) * np.asarray(xhat, dtype=np.float32)
    return np.minimum(np.float32(255), np.rint(v)).astype(np.uint8)
