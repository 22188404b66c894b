"""CPU restatement of the latent traversal and the pair interpolation (Learner.traverse / interpolate) over the oracle's
networks.  TEST INFRASTRUCTURE ONLY.  Like tests/walk_oracle.py, written from the oracle's `encoder`, `decoder` and
`cond_prior`, so it runs in fp32 and fp64 and rounds where the kernels do under `O.bf16_emulation()` (the z of both calls
is an fp32 value the kernel only selects or interpolates; `decoder` rounds it through `_w16` like the bf16 engine's z16).

A traversal sets z_d to an absolute value and keeps every other dim of the base code: the posterior z (`reconstruct`)
from images, the prior z (`generate`) from labels.  An interpolation mixes the posterior means z_a, z_b inside one range
of dims: z_a at t = 0, z_b at t = 1, z_a + t (z_b - z_a) otherwise.  Noise is explicit: eps [B,45] or None (means)."""
import torch

import generation_oracle as GO
import gccvae_oracle as O

ZS = O.Z_STYLE
PARTS = {"all": (0, O.Z_DIM), "style": (0, ZS), "classify": (ZS, O.Z_DIM)}


def base_z(p, c, x=None, y=None, eps=None):
    """z [B,45] of `reconstruct(x)` (x given) or of `generate(y)` (x None), without decoding."""
    if x is not None:
        return GO._posterior_z(p, x, eps)
    loc_p, scale_p = GO.prior(p, y, c)
    if eps is None:
        return torch.cat([torch.zeros(y.shape[0], ZS, dtype=c.dtype), loc_p], dim=-1)
    return torch.cat([eps[:, :ZS], loc_p + scale_p * eps[:, ZS:]], dim=-1)


def traverse_z(p, c, dims, values, x=None, y=None, eps=None):
    """-> z [B,D,T,45]: the base code with z_{dims[d]} = values[t]."""
    z0 = base_z(p, c, x=x, y=y, eps=eps)
    z = z0[:, None, None].repeat(1, len(dims), len(values), 1)
    for di, d in enumerate(dims):
        for t, v in enumerate(values):
            z[:, di, t, d] = float(v)
    return z


def interpolate_z(p, x_a, x_b, ts, part="all"):
    """-> z [B,T,45]: z_a outside PARTS[part]; inside it z_a at t = 0, z_b at t = 1, z_a + t (z_b - z_a) otherwise."""
    lo, hi = PARTS[part]
    za, zb = GO._posterior_z(p, x_a, None), GO._posterior_z(p, x_b, None)
    frames = []
    for t in ts:
        z = za.clone()
        t = float(t)
        z[:, lo:hi] = za[:, lo:hi] if t == 0.0 else zb[:, lo:hi] if t == 1.0 else za[:, lo:hi] + t * (zb - za)[:, lo:hi]
        frames.append(z)
    return torch.stack(frames, dim=1)


def _decode(p, z):
    return O.decoder(p, z.reshape(-1, O.Z_DIM)).reshape(*z.shape[:-1], 64, 64, 3)


def traverse(p, c, dims, values, x=None, y=None, eps=None):
    """-> (images [B,D,T,64,64,3], z [B,D,T,45])."""
    z = traverse_z(p, c, dims, values, x=x, y=y, eps=eps)
    return _decode(p, z), z


def interpolate(p, x_a, x_b, ts, part="all"):
    """-> (images [B,T,64,64,3], z [B,T,45])."""
    z = interpolate_z(p, x_a, x_b, ts, part)
    return _decode(p, z), z
