"""CPU restatement of image completion (Learner.complete) over the oracle's networks.  TEST INFRASTRUCTURE ONLY.  A loop
over tests/generation_oracle.py's `reconstruct` / `intervene` with the mask composite, so it runs in fp32 and fp64 and,
under `O.bf16_emulation()`, rounds where the kernels do.

Iteration t encodes the composite (x's observed pixels, the previous decode elsewhere; x itself at t = 1), takes z as
`reconstruct` does - or moves its classify dims to y_new as `intervene` does - and decodes; the decoder's mean replaces
the unobserved pixels.  Noise is explicit: eps [iters,B,45] or None (posterior means)."""
import torch

import generation_oracle as GO


def step(p, comp, x, mask, y_new=None, c=None, y=None, eps=None):
    """one iteration from the composite `comp` -> (next composite, decode, z, y_src or None); mask [B,64,64] bool."""
    if y_new is None:
        img, z = GO.reconstruct(p, comp, eps)
        y_src = None
    else:
        img, z, y_src = GO.intervene(p, comp, y_new, c, y=y, eps=eps)
    return torch.where(mask.unsqueeze(-1), x, img), img, z, y_src


def complete(p, x, mask, iters, y_new=None, c=None, y=None, eps=None):
    """-> (completed image, z, y_src) of the last iteration: x fp [B,64,64,3], mask [B,64,64] bool (True = observed)."""
    comp, z, y_src = x, None, None
    for t in range(iters):
        comp, _, z, y_src = step(p, comp, x, mask, y_new, c, y, None if eps is None else eps[t])
    return comp, z, y_src
