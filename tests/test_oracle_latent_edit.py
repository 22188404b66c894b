"""CPU: known answers of the traversal's and the interpolation's restatement (tests/latent_edit_oracle.py).
  * interpolation at t = 0 is the reconstruction of x_a, part "all" at t = 1 that of x_b;
  * part "classify" at t = 1 is swap(x_a, x_b), part "style" at t = 1 is swap(x_b, x_a);
  * the style and classify parts split the whole line: "all" is the style part's style dims with the classify part's
    classify dims, at every t; the dims outside a part are x_a's posterior mean;
  * a traversal frame at the base's own z_d is the base (reconstruction or generation), and every other dim of every
    traversal frame is the base code."""
import pytest
import torch

import generation_oracle as GO
import gccvae_oracle as O
import latent_edit_oracle as LO
import walk_oracle as WO
from test_oracle_walk import _setup

DTYPES = [torch.float64, torch.float32]
ZS = O.Z_STYLE
TS = [-0.5, 0.0, 0.3, 1.0, 1.5]


@pytest.mark.parametrize("dtype", DTYPES)
def test_interpolation_ends_are_reconstructions_and_swaps(dtype):
    p, x, _, _, _ = _setup(dtype)
    xb = x.flip(0)
    img_a, z_a = GO.reconstruct(p, x)
    img_b, z_b = GO.reconstruct(p, xb)
    img, z = LO.interpolate(p, x, xb, [0.0, 1.0], "all")
    assert torch.equal(z[:, 0], z_a) and torch.equal(img[:, 0], img_a)
    assert torch.equal(z[:, 1], z_b) and torch.equal(img[:, 1], img_b)
    for part, (first, second) in (("classify", (x, xb)), ("style", (xb, x))):
        img, z = LO.interpolate(p, x, xb, [0.0, 1.0], part)
        img_s, z_s = WO.swap(p, first, second)
        assert torch.equal(z[:, 0], z_a) and torch.equal(img[:, 0], img_a)
        assert torch.equal(z[:, 1], z_s) and torch.equal(img[:, 1], img_s)


@pytest.mark.parametrize("dtype", DTYPES)
def test_style_and_classify_parts_split_the_line(dtype):
    p, x, _, _, _ = _setup(dtype)
    xb = x.flip(0)
    _, z_a = GO.reconstruct(p, x)
    z_all = LO.interpolate_z(p, x, xb, TS, "all")
    z_sty = LO.interpolate_z(p, x, xb, TS, "style")
    z_cls = LO.interpolate_z(p, x, xb, TS, "classify")
    assert torch.equal(z_all, torch.cat([z_sty[..., :ZS], z_cls[..., ZS:]], dim=-1))
    T = len(TS)
    assert torch.equal(z_sty[..., ZS:], z_a[:, None, ZS:].expand(-1, T, -1))
    assert torch.equal(z_cls[..., :ZS], z_a[:, None, :ZS].expand(-1, T, -1))
    # the line is affine in t, also beyond [0, 1]
    _, z_b = GO.reconstruct(p, xb)
    tol = 1e-12 if dtype == torch.float64 else 2e-6
    for t, tv in enumerate(TS):
        assert float((z_all[:, t] - (z_a + tv * (z_b - z_a))).abs().max()) <= tol * max(1.0, abs(tv)) * float(z_a.abs().max())


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("source", ["images", "labels"])
@pytest.mark.parametrize("sample", [False, True])
def test_traversal_at_the_base_value_is_the_base(dtype, source, sample):
    p, x, y, noise, c = _setup(dtype)
    eps = noise["eps"] if sample else None
    if source == "images":
        img0, z0 = GO.reconstruct(p, x, eps)
        kw = dict(x=x, eps=eps)
    else:
        img0, z0 = GO.generate(p, y, c, eps)
        kw = dict(y=y, eps=eps)
    assert torch.equal(LO.base_z(p, c, **kw), z0)
    dims = [0, 26, 27, 44, 5]
    values = [-3.0, 0.5, 2.0]
    z = LO.traverse_z(p, c, dims, values, **kw)
    for di, d in enumerate(dims):
        keep = [k for k in range(O.Z_DIM) if k != d]
        assert torch.equal(z[:, di][..., keep], z0[:, None, keep].expand(-1, len(values), -1))
        assert torch.equal(z[:, di, :, d], torch.tensor(values, dtype=dtype).expand(x.shape[0], -1))
    # one image: the frame at the image's own z_d is the base image
    e1 = None if eps is None else eps[:1]
    img1, z1 = GO.reconstruct(p, x[:1], e1) if source == "images" else GO.generate(p, y[:1], c, e1)
    k1 = dict(x=x[:1], eps=e1) if source == "images" else dict(y=y[:1], eps=e1)
    for d in (3, 30):
        img, zt = LO.traverse(p, c, [d], [float(z1[0, d])], **k1)
        assert torch.equal(zt[0, 0, 0], z1[0]) and torch.equal(img[0, 0, 0], img1[0])
