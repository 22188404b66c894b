"""GPU: the latent traversal and the pair interpolation - Learner.traverse / interpolate (gccvae_gen_latent with its
traversal and pair fields + the chunked forward-only decoder, on the bf16 engine gccvae_convt_image_bf16 into each chunk's
slice of the output) - against the fp64 restatement of tests/latent_edit_oracle.py, their exact known answers against
reconstruct / generate / swap on both engines, chunking, sizes and argument checks."""
import numpy as np
import pytest
import torch

import generation_oracle as GO
import gccvae_oracle as O
import latent_edit_oracle as LO
from helpers import rel_err
from test_gpu_generation import _inputs, _learner, _oracle_params

pytestmark = pytest.mark.gpu
PRECISIONS = ["fp32", "bf16"]
ZS = O.Z_STYLE
PARTS = ["all", "style", "classify"]
TS = [-0.5, 0.0, 0.3, 1.0, 1.5]
VALUES = [-3.0, -0.7, 0.0, 2.5]
# traversal sources: (images or labels, sampling)
SOURCES = [("images", False), ("images", True), ("labels", False), ("labels", True)]


def _traverse(lrn, source, x, y, eps, c, sample, dims, values, **kw):
    noise = {"eps": eps} if sample else None
    if source == "images":
        img = lrn.traverse(x, dims=dims, values=values, sample=sample, c=c, noise=noise, **kw)
    else:
        img = lrn.traverse(y=y, dims=dims, values=values, sample=sample, c=c, noise=noise, **kw)
    torch.cuda.synchronize()
    return img, lrn.last["z"]


def _oracle_traverse(p, source, x, y, eps, c, sample, dims, values):
    e = eps.double() if sample else None
    v = torch.tensor(values, dtype=torch.float32).double().tolist()
    if source == "images":
        return LO.traverse(p, c.double(), dims, v, x=x.double(), eps=e)
    return LO.traverse(p, c.double(), dims, v, y=y, eps=e)


def _interpolate(lrn, xa, xb, ts, part, **kw):
    img = lrn.interpolate(xa, xb, ts=ts, part=part, **kw)
    torch.cuda.synchronize()
    return img, lrn.last["z"]


def _ts64(ts):
    return torch.tensor(ts, dtype=torch.float32).double().tolist()


# (B, dims): every dim, and a reordered subset across the style / classify boundary
CASES = [(4, list(range(45))), (7, [44, 0, 27, 26, 9])]


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
@pytest.mark.parametrize("case", [0, 1])
def test_fp32_engine_matches_fp64_oracle(params, case):
    B, dims = CASES[case]
    values = [-3.0, 2.5] if case == 0 else VALUES
    lrn = _learner(params, "fp32")
    p = _oracle_params(lrn)
    x, y, _, eps, c = _inputs(B)
    for source, sample in SOURCES:
        img, z = _traverse(lrn, source, x, y, eps, c, sample, dims, values)
        img_o, z_o = _oracle_traverse(p, source, x, y, eps, c, sample, dims, values)
        ei, ez = rel_err(img, img_o), rel_err(z, z_o)
        print("fp32 {} B={} traverse {} sample={}: image {:.2e}, z {:.2e}".format(params, B, source, sample, ei, ez))
        assert img.shape == (B, len(dims), len(values), 64, 64, 3) and img.dtype == torch.float32
        assert z.shape == (B, len(dims), len(values), 45) and img.is_contiguous()
        assert ei <= 1e-5 and ez <= 1e-5, (source, sample, ei, ez)
    # Interpolation, judged per frame.  Frame t decodes (1 - t) z_a + t z_b, so the fp32 encoder's own error in z_a and
    # z_b reaches it with the weights |1 - t| and |t|: for t in [0, 1] the frame is held to 1e-5 like a reconstruction,
    # an extrapolated frame to 1e-5 (|1 - t| + |t|).  Measured on B200 (1000 W), shipped checkpoint, B = 4 and 7, all
    # parts: frames in [0, 1] at most 7.6e-6 (t = 0 and 1: 7.2e-6, the reconstruction's error), frames at t = -0.5
    # and 1.5 at most 1.08e-5 (part "all", bound 2e-5); trained-like parameters 1.4e-7.
    xb = x.flip(0)
    for part in PARTS:
        img, z = _interpolate(lrn, x, xb, TS, part)
        img_o, z_o = LO.interpolate(p, x.double(), xb.double(), _ts64(TS), part)
        assert img.shape == (B, len(TS), 64, 64, 3) and z.shape == (B, len(TS), 45) and img.is_contiguous()
        ez = rel_err(z, z_o)
        ei = [rel_err(img[:, t], img_o[:, t]) for t in range(len(TS))]
        print("fp32 {} B={} interpolate {}: z {:.2e}, image per t {}".format(
            params, B, part, ez, ", ".join("{}: {:.2e}".format(tv, e) for tv, e in zip(TS, ei))))
        assert ez <= 1e-5, (part, ez)
        for tv, e in zip(TS, ei):
            assert e <= 1e-5 * max(1.0, abs(1.0 - tv) + abs(tv)), (part, tv, e)


# bf16 engine vs the emulating oracle, judged per stage as tests/test_gpu_walk.py does: z against the oracle's z, the image
# against the emulating decoder applied to the engine's own z.
# Measured on B200 (1000 W), largest over the four traversal cases and the three interpolation parts, B = 7:
#   z: 1.12e-3 (trained-like parameters, interpolation: the encoder's bf16 z), checkpoint 4.3e-5;
#   image from own z: 4.12e-3 (checkpoint, interpolation over all dims, t from -0.5 to 1.5), trained-like 6.3e-5.
# Bounds: ~1.5x those.
BF16_BOUNDS = {"z": 1.7e-3, "image_from_z": 6.2e-3}


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
def test_bf16_engine_matches_emulating_oracle(params):
    lrn = _learner(params, "bf16")
    p = _oracle_params(lrn)
    B, dims = CASES[1]
    x, y, _, eps, c = _inputs(B)
    worst = dict(z=0.0, image_from_z=0.0)
    runs = []
    for source, sample in SOURCES:
        img, z = _traverse(lrn, source, x, y, eps, c, sample, dims, VALUES)
        with O.bf16_emulation():
            _, z_o = _oracle_traverse(p, source, x, y, eps, c, sample, dims, VALUES)
        runs.append(("traverse {} sample={}".format(source, sample), img, z, z_o))
    for part in PARTS:
        img, z = _interpolate(lrn, x, x.flip(0), TS, part)
        with O.bf16_emulation():
            z_o = LO.interpolate_z(p, x.double(), x.flip(0).double(), _ts64(TS), part)
        runs.append(("interpolate " + part, img, z, z_o))
    for what, img, z, z_o in runs:
        with O.bf16_emulation():
            img_z = O.decoder(p, z.reshape(-1, 45).cpu().double()).reshape(img.shape)
        e = dict(z=rel_err(z, z_o), image_from_z=rel_err(img, img_z))
        print("bf16 {} {}: z {:.2e}, image from the engine's z {:.2e}".format(params, what, e["z"], e["image_from_z"]))
        worst = {k: max(worst[k], e[k]) for k in worst}
    print("bf16 {} worst: {}".format(params, worst))
    assert worst["z"] <= BF16_BOUNDS["z"] and worst["image_from_z"] <= BF16_BOUNDS["image_from_z"], worst


@pytest.mark.parametrize("precision", PRECISIONS)
def test_exact_known_answers(precision):
    B = 8
    x, y, _, eps, c = _inputs(B)
    xb = x.flip(0)
    lrn = _learner("trained_like", precision)
    # interpolation: t = 0 is reconstruct(x_a), part "all" at t = 1 is reconstruct(x_b); "classify" at t = 1 is
    # swap(x_a, x_b), "style" at t = 1 is swap(x_b, x_a); the dims outside the part are x_a's posterior mean
    ra = lrn.reconstruct(x)
    za = lrn.last["z"]
    rb = lrn.reconstruct(xb)
    zb = lrn.last["z"]
    s_ab = lrn.swap(x, xb)
    z_ab = lrn.last["z"]
    s_ba = lrn.swap(xb, x)
    z_ba = lrn.last["z"]
    ends = {"all": (rb, zb), "classify": (s_ab, z_ab), "style": (s_ba, z_ba)}
    lo_hi = {"all": (0, 45), "style": (0, ZS), "classify": (ZS, 45)}
    for part in PARTS:
        img, z = _interpolate(lrn, x, xb, TS, part)
        assert torch.equal(z[:, 1], za) and torch.equal(img[:, 1], ra), part
        assert torch.equal(z[:, 3], ends[part][1]) and torch.equal(img[:, 3], ends[part][0]), part
        lo, hi = lo_hi[part]
        outside = [d for d in range(45) if not lo <= d < hi]
        assert torch.equal(z[..., outside], za[:, None, outside].expand(-1, len(TS), -1)), part
    # swap is the one-value classify interpolation, and swap(x, x) is still the reconstruction
    assert torch.equal(lrn.swap(x, x), ra) and torch.equal(lrn.last["z"], za)
    # traversal: every other dim of every frame is the base code; the frame at the base's own z_d is the base
    dims = [3, 30, 44, 0]
    for sample in (False, True):
        noise = {"eps": eps} if sample else None
        for source in ("images", "labels"):
            if source == "images":
                lrn.reconstruct(x, sample=sample, noise=noise)
            else:
                lrn.generate(y, sample=sample, c=c, noise=noise)
            z0 = lrn.last["z"]
            img, z = _traverse(lrn, source, x, y, eps, c, sample, dims, VALUES)
            for di, d in enumerate(dims):
                keep = [k for k in range(45) if k != d]
                assert torch.equal(z[:, di][..., keep], z0[:, None, keep].expand(-1, len(VALUES), -1))
                assert torch.equal(z[:, di, :, d].cpu(), torch.tensor(VALUES).expand(B, -1))
            # values are shared by all images: one image per call, against the base call of that one image
            for b in (0, 5):
                n1 = {"eps": eps[b:b + 1]} if sample else None
                if source == "images":
                    base1 = lrn.reconstruct(x[b:b + 1], sample=sample, noise=n1)
                else:
                    base1 = lrn.generate(y[b:b + 1], sample=sample, c=c, noise=n1)
                z1 = lrn.last["z"]
                for d in (3, 30):
                    img, z = _traverse(lrn, source, x[b:b + 1], y[b:b + 1], eps[b:b + 1], c, sample, [d],
                                       [float(z1[0, d])])
                    assert torch.equal(z[0, 0, 0], z1[0]) and torch.equal(img[0, 0, 0], base1[0]), (source, sample, b, d)
    # uint8 output = to_u8 of the fp32 output; the same noise and c twice give the same bits
    f = lrn.traverse(x, dims=[1, 40], values=VALUES, sample=True, c=c, noise={"eps": eps})
    f2 = lrn.traverse(x, dims=[1, 40], values=VALUES, sample=True, c=c, noise={"eps": eps})
    u = lrn.traverse(x, dims=[1, 40], values=VALUES, sample=True, c=c, noise={"eps": eps}, dtype=torch.uint8)
    torch.cuda.synchronize()
    assert torch.equal(f, f2) and u.dtype == torch.uint8 and u.shape == f.shape and u.is_contiguous()
    assert np.array_equal(u.cpu().numpy(), GO.to_u8(f.cpu().numpy()))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_chunking_changes_no_bit(precision):
    lrn = _learner("trained_like", precision)
    x, y, _, eps, c = _inputs(3)
    dims, values = [40, 2], [-1.0, 0.0, 0.6, 3.0]
    for source, sample in SOURCES:
        outs = []
        for max_rows in (1, 7, 3 * 2 * 4):
            img, z = _traverse(lrn, source, x, y, eps, c, sample, dims, values, max_rows=max_rows)
            outs.append((img, z.clone()))
        for img, z in outs[1:]:
            assert torch.equal(z, outs[0][1]), (source, sample)
            assert torch.equal(img, outs[0][0]), (source, sample)
    for part in PARTS:
        outs = []
        for max_rows in (1, 7, 3 * len(TS)):
            img, z = _interpolate(lrn, x, x.flip(0), TS, part, max_rows=max_rows)
            outs.append((img, z.clone()))
        for img, z in outs[1:]:
            assert torch.equal(z, outs[0][1]) and torch.equal(img, outs[0][0]), part


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B", [1, 7, 256])
def test_batch_sizes(precision, B):
    lrn = _learner("trained_like", precision)
    x, y, _, eps, c = _inputs(B)
    xu8 = (x * 255).round().to(torch.uint8)          # uint8 images are accepted too
    dims, values, ts = [16, 2, 33], [-2.0, 0.5, 1.0], [0.0, 0.5, 1.0]
    max_rows = max(1, B * 9 // 4)                     # several chunks, the last one short
    for dtype in (torch.float32, torch.uint8):
        t = lrn.traverse(xu8, dims=dims, values=values, c=c, dtype=dtype, max_rows=max_rows)
        assert set(lrn.last) == {"z", "c"} and lrn.last["z"].shape == (B, 3, 3, 45)
        g = lrn.traverse(y=y, dims=dims, values=values, c=c, noise={"eps": eps}, sample=True, dtype=dtype,
                         max_rows=max_rows)
        i = lrn.interpolate(xu8, x.flip(0), ts=ts, part="style", dtype=dtype, max_rows=max_rows)
        assert set(lrn.last) == {"z"} and lrn.last["z"].shape == (B, 3, 45)
        torch.cuda.synchronize()
        for r in (t, g):
            assert r.shape == (B, 3, 3, 64, 64, 3) and r.dtype == dtype and r.is_contiguous() and r.is_cuda
        assert i.shape == (B, 3, 64, 64, 3) and i.dtype == dtype and i.is_contiguous()
        if dtype == torch.float32:
            assert all(bool(torch.isfinite(r).all()) and float(r.min()) >= 0.0 and float(r.max()) <= 1.0
                       for r in (t, g, i))
            t32, g32, i32 = t, g, i
        else:
            for r, r32 in ((t, t32), (g, g32), (i, i32)):
                assert np.array_equal(r.cpu().numpy(), GO.to_u8(r32.cpu().numpy()))
    # defaults: all 45 dims at the integers -3..3; 8 points from 0 to 1, both ends exact
    d = lrn.traverse(xu8[:1])
    zd = lrn.last["z"]
    e = lrn.interpolate(xu8[:1], x[:1])
    torch.cuda.synchronize()
    assert d.shape == (1, 45, 7, 64, 64, 3) and e.shape == (1, 8, 64, 64, 3)
    assert torch.equal(zd[0, torch.arange(45), :, torch.arange(45)].cpu(), torch.arange(-3.0, 4.0).expand(45, -1))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_noise_is_fresh_per_call_and_a_given_c_and_eps_are_used_verbatim(precision):
    x, y, _, eps, c = _inputs(4)
    lrn = _learner("trained_like", precision)
    a = lrn.traverse(y=y, dims=[30], values=[0.5], sample=True)
    ca = lrn.last["c"]
    b_ = lrn.traverse(y=y, dims=[30], values=[0.5], sample=True)
    cb = lrn.last["c"]
    torch.cuda.synchronize()
    assert not torch.equal(a, b_) and not torch.equal(ca, cb)
    assert not torch.equal(lrn.traverse(x, dims=[3], values=[0.5], sample=True, c=c),
                           lrn.traverse(x, dims=[3], values=[0.5], sample=True, c=c))
    for call in (lambda: lrn.traverse(y=y, dims=[3], c=c), lambda: lrn.traverse(x, dims=[3], c=c)):
        call()
        torch.cuda.synchronize()
        assert torch.equal(lrn.last["c"].cpu(), c)
    # a given eps is used verbatim: the traversal's base is the sampled reconstruction / generation with that eps
    r = lrn.reconstruct(x, sample=True, noise={"eps": eps})
    zr = lrn.last["z"]
    lrn.traverse(x, dims=[0], values=[0.0], sample=True, noise={"eps": eps})
    assert torch.equal(lrn.last["z"][:, 0, 0, 1:], zr[:, 1:])
    lrn.generate(y, sample=True, c=c, noise={"eps": eps})
    zg = lrn.last["z"]
    lrn.traverse(y=y, dims=[44], values=[0.0], sample=True, c=c, noise={"eps": eps})
    torch.cuda.synchronize()
    assert torch.equal(lrn.last["z"][:, 0, 0, :44], zg[:, :44]) and r.shape == (4, 64, 64, 3)


def test_bad_arguments_raise_value_error():
    lrn = _learner("trained_like", "bf16")
    x, y, _, eps, c = _inputs(4)
    bad = [
        lambda: lrn.traverse(),
        lambda: lrn.traverse(x, y=y),
        lambda: lrn.traverse(y=y[:, :17]),
        lambda: lrn.traverse(x[:, :32]),
        lambda: lrn.traverse(x[:0]),
        lambda: lrn.traverse(x, dims=[]),
        lambda: lrn.traverse(x, dims=[45]),
        lambda: lrn.traverse(x, dims=[-1]),
        lambda: lrn.traverse(x, dims=[2, 2]),
        lambda: lrn.traverse(x, dims=[1.5]),
        lambda: lrn.traverse(x, dims=[[1, 2]]),
        lambda: lrn.traverse(x, values=[]),
        lambda: lrn.traverse(x, values=[[0.0, 1.0]]),
        lambda: lrn.traverse(x, values=[0.0, float("nan")]),
        lambda: lrn.traverse(x, values=[float("-inf")]),
        lambda: lrn.traverse(x, values=[1e39]),
        lambda: lrn.traverse(x, values=["a"]),
        lambda: lrn.traverse(x, dtype=torch.float16),
        lambda: lrn.traverse(x, c=c[:17]),
        lambda: lrn.traverse(x, noise={"eps": eps[:3]}),
        lambda: lrn.traverse(x, max_rows=0),
        lambda: lrn.traverse(x, max_rows=2.5),
        lambda: lrn.traverse(x, dims=list(range(45)), values=torch.zeros(2 ** 31 // 180 + 1)),   # 2^31 rows
        lambda: lrn.interpolate(x, x[:3]),
        lambda: lrn.interpolate(x[:0], x[:0]),
        lambda: lrn.interpolate(x[:, :32], x),
        lambda: lrn.interpolate(x, x, part="labels"),
        lambda: lrn.interpolate(x, x, part=None),
        lambda: lrn.interpolate(x, x, ts=[]),
        lambda: lrn.interpolate(x, x, ts=[0.5, float("nan")]),
        lambda: lrn.interpolate(x, x, ts=[[0.0]]),
        lambda: lrn.interpolate(x, x, dtype=torch.int32),
        lambda: lrn.interpolate(x, x, max_rows=0),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
            pytest.fail("case {} did not raise".format(i))
