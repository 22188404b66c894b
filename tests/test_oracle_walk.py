"""CPU: known answers of the label walk's and the swap's restatement (tests/walk_oracle.py).
  * frames at alpha in {0, 1} are `intervene` / `generate` with that label set, bit for bit;
  * the frame at alpha = y_src,l is the reconstruction (per image: the images whose label l is alpha);
  * one-one gates (c = I): walking label l moves classify dim l only;
  * fresh-init prior: every frame is the reconstruction (to rounding: `cond_prior` forms the true and the false sums
    separately, so a fractional alpha rounds them differently);
  * loc_p(alpha) is affine in alpha, also beyond [0, 1];
  * swap(x, x) is the reconstruction."""
import numpy as np
import pytest
import torch

import generation_oracle as GO
import gccvae_oracle as O
import walk_oracle as WO

DTYPES = [torch.float64, torch.float32]
ZS = O.Z_STYLE


def _setup(dtype, B=4, trained_like=True, one_one=False, seed=0):
    import os
    p = {k: v.to(dtype) for k, v in O.init_params(seed, trained_like=trained_like).items()}
    x, y, noise = O.make_inputs(B, k=1, dtype=dtype)
    if one_one:
        c = torch.eye(18, dtype=dtype)
    else:
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "data", "gating_matrix_0.2.npy")
        mu = torch.as_tensor(np.load(path), dtype=dtype)
        c = O.sample_gating_parameter(mu, 0.3, noise["U1"], noise["U2"])
    return p, x, y, noise, c


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sample", [False, True])
def test_frames_at_zero_and_one_are_intervene_and_generate(dtype, sample):
    p, x, y, noise, c = _setup(dtype)
    eps = noise["eps"] if sample else None
    labels = [3, 0, 17]
    img_w, z_w, y_src = WO.walk(p, c, labels, [0.0, 1.0], x=x, y=y, eps=eps)
    assert torch.equal(y_src, y)
    _, z_g, _ = WO.walk(p, c, labels, [0.0, 1.0], y=y, eps=eps)
    for li, l in enumerate(labels):
        for t, a in enumerate((0, 1)):
            y_a = y.clone()
            y_a[:, l] = a
            img_i, z_i, _ = GO.intervene(p, x, y_a, c, y=y, eps=eps)
            assert torch.equal(z_w[:, li, t], z_i) and torch.equal(img_w[:, li, t], img_i)
            _, z_gen = GO.generate(p, y_a, c, eps)
            assert torch.equal(z_g[:, li, t], z_gen)


@pytest.mark.parametrize("dtype", DTYPES)
def test_frame_at_the_source_label_is_the_reconstruction(dtype):
    p, x, y, _, c = _setup(dtype, B=8)
    _, z_r = GO.reconstruct(p, x)
    for y_given in (y, None):
        z_w, y_src = WO.walk_z(p, c, range(18), [0.0, 1.0], x=x, y=y_given)
        for l in range(18):
            for t in (0, 1):
                rows = y_src[:, l] == t
                assert torch.equal(z_w[rows, l, t], z_r[rows])


@pytest.mark.parametrize("dtype", DTYPES)
def test_one_one_gates_move_only_the_walked_label_dim(dtype):
    p, x, y, _, c = _setup(dtype, one_one=True)
    _, z_r = GO.reconstruct(p, x)
    alphas = [-0.5, 0.25, 1.5]
    z_w, _ = WO.walk_z(p, c, [0, 9, 17], alphas, x=x, y=y)
    for li, l in enumerate((0, 9, 17)):
        keep = [d for d in range(O.Z_DIM) if d != ZS + l]
        for t in range(len(alphas)):
            assert torch.equal(z_w[:, li, t][:, keep], z_r[:, keep])
            assert not torch.equal(z_w[:, li, t, ZS + l], z_r[:, ZS + l])


@pytest.mark.parametrize("dtype", DTYPES)
def test_fresh_init_prior_makes_every_frame_the_reconstruction(dtype):
    p, x, y, _, c = _setup(dtype, trained_like=False)
    img_r, z_r = GO.reconstruct(p, x)
    img_w, z_w, _ = WO.walk(p, c, [2, 11], [-0.5, 0.0, 0.4, 1.0, 1.5], x=x, y=y)
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    assert float((z_w - z_r[:, None, None]).abs().max()) <= tol * float(z_r.abs().max())
    assert float((img_w - img_r[:, None, None]).abs().max()) <= tol


@pytest.mark.parametrize("dtype", DTYPES)
def test_prior_loc_is_affine_in_alpha(dtype):
    p, _, y, _, c = _setup(dtype)
    tol = 1e-12 if dtype == torch.float64 else 2e-6
    for l in (0, 8, 17):
        l0, _ = WO.prior_walk(p, y, c, l, 0.0)
        l1, _ = WO.prior_walk(p, y, c, l, 1.0)
        scale = float(torch.cat([l0, l1]).abs().max())
        for a in (-0.5, 0.3, 0.5, 1.5, 3.0):
            la, sa = WO.prior_walk(p, y, c, l, a)
            assert float((la - (l0 + a * (l1 - l0))).abs().max()) <= tol * max(1.0, abs(a)) * scale
            assert bool((sa >= 1e-3).all()) and bool(torch.isfinite(sa).all())
        assert not torch.equal(l0, l1)


@pytest.mark.parametrize("dtype", DTYPES)
def test_swap_of_an_image_with_itself_is_the_reconstruction(dtype):
    p, x, _, _, _ = _setup(dtype)
    img_r, z_r = GO.reconstruct(p, x)
    img_s, z_s = WO.swap(p, x, x)
    assert torch.equal(z_s, z_r) and torch.equal(img_s, img_r)
    x2 = x.flip(0)
    _, z_s2 = WO.swap(p, x, x2)
    _, z_r2 = GO.reconstruct(p, x2)
    assert torch.equal(z_s2[:, :ZS], z_r[:, :ZS]) and torch.equal(z_s2[:, ZS:], z_r2[:, ZS:])
