"""CPU restatement of the label walk and the characteristic swap (Learner.walk / swap) over the oracle's networks.
TEST INFRASTRUCTURE ONLY.  Like tests/generation_oracle.py, written from the oracle's `encoder`, `decoder`,
`cond_prior` and `classifier`, so it runs in fp32 and fp64 and rounds where the kernels do under `O.bf16_emulation()`.

A walk of label l at value alpha is the conditional prior with y_l replaced by the real number alpha: `O.cond_prior`
takes a continuous tiled y.  Noise is explicit: eps [B,45] (style dims 0..26, classify dims 27..44), shared by every
frame of an image, or None for the means."""
import torch

import generation_oracle as GO
import gccvae_oracle as O

ZS = O.Z_STYLE


def prior_walk(p, y, c, l, alpha):
    """(loc_p, scale_p) [B,18] for the labels y [B,18] (nonzero = 1) with label l at the real value alpha."""
    yt = (y != 0).to(c.dtype)
    yt[:, l] = float(alpha)
    return O.cond_prior(p, yt.unsqueeze(-1).repeat(1, 1, O.Z_CLASSIFY), c)


def walk_z(p, c, labels, alphas, x=None, y=None, eps=None):
    """-> (z [B,L,T,45], y_src [B,18] int64 or None).  x given: the posterior z (or loc + scale eps) moved from y (default:
    the classifier's decision on z_c) to y with y_l = alpha by the counterfactual of `GO.intervene`.  x None: z_s = eps_s,
    z_c = loc_p + scale_p eps_c at the walked labels (eps None: z_s = 0, z_c = loc_p)."""
    y_src = None
    if x is not None:
        z0 = GO._posterior_z(p, x, eps)
        zc = z0[:, ZS:]
        if y is None:
            y, _ = GO.decision(p, zc, c)
        y_src = (y != 0).to(torch.int64)
        ls, ss = GO.prior(p, y, c)
        e = (zc - ls) / ss
    frames = []
    for l in labels:
        row = []
        for a in alphas:
            lt, st = prior_walk(p, y, c, l, a)
            if x is not None:
                z = torch.cat([z0[:, :ZS], zc + (lt - ls) + (st - ss) * e], dim=-1)
            elif eps is None:
                z = torch.cat([torch.zeros(y.shape[0], ZS, dtype=c.dtype), lt], dim=-1)
            else:
                z = torch.cat([eps[:, :ZS], lt + st * eps[:, ZS:]], dim=-1)
            row.append(z)
        frames.append(torch.stack(row, dim=1))
    return torch.stack(frames, dim=1), y_src


def walk(p, c, labels, alphas, x=None, y=None, eps=None):
    """-> (images [B,L,T,64,64,3], z [B,L,T,45], y_src)."""
    z, y_src = walk_z(p, c, labels, alphas, x=x, y=y, eps=eps)
    B, L, T, _ = z.shape
    return O.decoder(p, z.reshape(B * L * T, -1)).reshape(B, L, T, 64, 64, 3), z, y_src


def swap(p, x_style, x_char):
    """-> (images, z): z = [z_s of x_style, z_c of x_char], both posterior means."""
    z = torch.cat([GO._posterior_z(p, x_style, None)[:, :ZS], GO._posterior_z(p, x_char, None)[:, ZS:]], dim=-1)
    return O.decoder(p, z), z
