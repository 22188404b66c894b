"""CPU: known answers of the generation path's restatement (tests/generation_oracle.py) and the uint8 rule of the
generated images.
  * identity: intervening from y to y gives the reconstruction, bit for bit;
  * one-one gates (c = I): changing label j moves classify dim j only, the other 44 dims are bit-identical;
  * fresh-init prior (loc kernels 0, scale kernels 1, SURVEY.md §8c known answer 5): loc_p = 0 and scale_p does not
    depend on y, so any intervention is the identity - here only to rounding, because `cond_prior` forms the true and
    the false sums separately (the kernel's single running sum makes it bitwise, tests/test_gpu_generation.py);
  * Generate with sample=False: z_s = 0 and z_c = loc_p(y, c) exactly."""
import numpy as np
import pytest
import torch

import generation_oracle as GO
import gccvae_oracle as O

DTYPES = [torch.float64, torch.float32]


def _setup(dtype, B=4, trained_like=True, one_one=False, seed=0):
    p = {k: v.to(dtype) for k, v in O.init_params(seed, trained_like=trained_like).items()}
    x, y, noise = O.make_inputs(B, k=1, dtype=dtype)
    if one_one:
        c = torch.eye(18, dtype=dtype)
    else:
        mu = torch.as_tensor(np.load(_gating("0.2")), dtype=dtype)
        c = O.sample_gating_parameter(mu, 0.3, noise["U1"], noise["U2"])
    return p, x, y, noise, c


def _gating(frac):
    import os
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "data", "gating_matrix_{}.npy".format(frac))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sample", [False, True])
def test_intervention_to_the_same_labels_is_the_reconstruction(dtype, sample):
    p, x, y, noise, c = _setup(dtype)
    eps = noise["eps"] if sample else None
    img_r, z_r = GO.reconstruct(p, x, eps)
    img_i, z_i, y_src = GO.intervene(p, x, y, c, y=y, eps=eps)
    assert torch.equal(z_i, z_r) and torch.equal(img_i, img_r) and torch.equal(y_src, y)
    # the classifier's own decision as the source labels, moved to itself: identity as well
    _, z_d, _ = GO.intervene(p, x, GO.decision(p, z_r[:, O.Z_STYLE:], c)[0], c, eps=eps)
    assert torch.equal(z_d, z_r)


@pytest.mark.parametrize("dtype", DTYPES)
def test_one_one_gates_move_only_the_changed_label_dim(dtype):
    p, x, y, _, c = _setup(dtype, one_one=True)
    _, z_r = GO.reconstruct(p, x)
    for j in (0, 7, 17):
        y_new = y.clone()
        y_new[:, j] = 1 - y_new[:, j]
        _, z_i, _ = GO.intervene(p, x, y_new, c, y=y)
        keep = [d for d in range(O.Z_DIM) if d != O.Z_STYLE + j]
        assert torch.equal(z_i[:, keep], z_r[:, keep])
        assert not torch.equal(z_i[:, O.Z_STYLE + j], z_r[:, O.Z_STYLE + j])


@pytest.mark.parametrize("dtype", DTYPES)
def test_fresh_init_prior_makes_every_intervention_the_identity(dtype):
    p, x, y, _, c = _setup(dtype, trained_like=False)
    assert float(p["prior.loc_true"].abs().max()) == 0.0 and float(p["prior.scale_false"].min()) == 1.0
    img_r, z_r = GO.reconstruct(p, x)
    y_new = 1 - y
    img_i, z_i, _ = GO.intervene(p, x, y_new, c, y=y)
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    assert float((z_i - z_r).abs().max()) <= tol * float(z_r.abs().max())
    assert float((img_i - img_r).abs().max()) <= tol
    loc_a, sc_a = GO.prior(p, y, c)
    loc_b, sc_b = GO.prior(p, y_new, c)
    assert float(loc_a.abs().max()) == 0.0 and float(loc_b.abs().max()) == 0.0
    assert float((sc_a - sc_b).abs().max()) <= tol


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("one_one", [True, False])
def test_generate_without_sampling_is_the_prior_mean(dtype, one_one):
    p, _, y, noise, c = _setup(dtype, one_one=one_one)
    img, z = GO.generate(p, y, c)
    loc_p, _ = GO.prior(p, y, c)
    assert torch.equal(z[:, :O.Z_STYLE], torch.zeros_like(z[:, :O.Z_STYLE]))
    assert torch.equal(z[:, O.Z_STYLE:], loc_p)
    assert img.shape == (y.shape[0], 64, 64, 3) and img.dtype == dtype
    # the prior's mean depends on the labels (a trained-like prior), the sampled code on eps as well
    assert not torch.equal(GO.generate(p, 1 - y, c)[1], z)
    _, z_s = GO.generate(p, y, c, noise["eps"])
    assert torch.equal(z_s[:, :O.Z_STYLE], noise["eps"][:, :O.Z_STYLE])


def _half_way_values():
    """fp32 x with 255 * x (in fp32) exactly k + 0.5 for codes k = 0..254."""
    out = []
    for k in range(255):
        x = np.float32((k + 0.5) / 255.0)
        for _ in range(8):
            v = np.float32(255) * x
            if v == np.float32(k + 0.5):
                out.append((k, x))
                break
            x = np.nextafter(x, np.float32(np.inf) if v < k + 0.5 else np.float32(-np.inf), dtype=np.float32)
    return out


def test_uint8_rule_rounds_half_way_values_to_even():
    half = _half_way_values()
    assert len(half) >= 200, len(half)
    ks = np.array([k for k, _ in half])
    xs = np.array([x for _, x in half], dtype=np.float32)
    want = np.where(ks % 2 == 0, ks, ks + 1).astype(np.uint8)
    assert np.array_equal(GO.to_u8(xs), want)
    # the engine's rule (torch, fp32) is the same function
    from gccvae_b200.engine import image_u8
    assert np.array_equal(image_u8(torch.from_numpy(xs)).numpy(), want)
    # ends of the range, and a value whose product rounds past 255 is held at 255
    edge = np.array([0.0, 1.0, np.nextafter(np.float32(1), np.float32(2), dtype=np.float32)], dtype=np.float32)
    assert GO.to_u8(edge).tolist() == [0, 255, 255]
    assert image_u8(torch.from_numpy(edge)).tolist() == [0, 255, 255]
    rnd = np.random.default_rng(0).random(100000, dtype=np.float32)
    assert np.array_equal(image_u8(torch.from_numpy(rnd)).numpy(), GO.to_u8(rnd))
