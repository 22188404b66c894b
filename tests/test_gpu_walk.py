"""GPU: the label walk and the characteristic swap - Learner.walk / swap (gccvae_gen_latent + the chunked forward-only
decoder, on the bf16 engine gccvae_convt_image_bf16 into each chunk's slice of the output) - against the fp64
restatement of tests/walk_oracle.py, their exact known answers against generate / reconstruct / intervene on both
engines, chunking, sizes and argument checks."""
import numpy as np
import pytest
import torch

import generation_oracle as GO
import gccvae_oracle as O
import walk_oracle as WO
from helpers import rel_err
from test_gpu_generation import _inputs, _learner, _oracle_params

pytestmark = pytest.mark.gpu
PRECISIONS = ["fp32", "bf16"]
ZS = O.Z_STYLE
ALPHAS = [-0.5, 0.0, 0.3, 1.0, 1.5]


def _walk(lrn, mode, x, y, eps, c, sample, labels, alphas, **kw):
    noise = {"eps": eps} if sample else None
    if mode == "images":
        img = lrn.walk(x, y=y, labels=labels, alphas=alphas, sample=sample, c=c, noise=noise, **kw)
    else:
        img = lrn.walk(y=y, labels=labels, alphas=alphas, sample=sample, c=c, noise=noise, **kw)
    torch.cuda.synchronize()
    return img, lrn.last["z"]


def _oracle(p, mode, x, y, eps, c, sample, labels, alphas):
    e = eps.double() if sample else None
    a = torch.tensor(alphas, dtype=torch.float32).double().tolist()
    if mode == "images":
        img, z, _ = WO.walk(p, c.double(), labels, a, x=x.double(), y=y, eps=e)
    else:
        img, z, _ = WO.walk(p, c.double(), labels, a, y=y, eps=e)
    return img, z


MODES = [("images", False), ("images", True), ("labels", False), ("labels", True)]
# (B, labels, alphas): every label at the two extrapolated values, and a reordered subset at five values
CASES = [(4, list(range(18)), [-0.5, 1.5]), (7, [17, 3, 9], ALPHAS)]


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
@pytest.mark.parametrize("case", [0, 1])
def test_fp32_engine_matches_fp64_oracle(params, case):
    B, labels, alphas = CASES[case]
    lrn = _learner(params, "fp32")
    p = _oracle_params(lrn)
    x, y, _, eps, c = _inputs(B)
    for mode, sample in MODES:
        img, z = _walk(lrn, mode, x, y, eps, c, sample, labels, alphas)
        img_o, z_o = _oracle(p, mode, x, y, eps, c, sample, labels, alphas)
        ei, ez = rel_err(img, img_o), rel_err(z, z_o)
        print("fp32 {} B={} {} sample={}: image {:.2e}, z {:.2e}".format(params, B, mode, sample, ei, ez))
        assert img.shape == (B, len(labels), len(alphas), 64, 64, 3) and img.dtype == torch.float32
        assert z.shape == (B, len(labels), len(alphas), 45) and img.is_contiguous()
        assert ei <= 1e-5 and ez <= 1e-5, (mode, sample, ei, ez)
    img = lrn.swap(x, x.flip(0))
    torch.cuda.synchronize()
    img_o, z_o = WO.swap(p, x.double(), x.flip(0).double())
    assert rel_err(img, img_o) <= 1e-5 and rel_err(lrn.last["z"], z_o) <= 1e-5


# bf16 engine vs the emulating oracle, judged per stage as tests/test_gpu_generation.py does: z against the oracle's z,
# the image against the emulating decoder applied to the engine's own z.
# Measured on B200 (1000 W), largest over the four mode / sampling cases and the swap, B = 7:
#   z: 7.7e-4 (trained-like parameters), checkpoint 3.2e-5;
#   image from own z: 2.89e-3 (checkpoint, from images with sampling), trained-like 6.0e-5.
# Bounds: ~1.5x those.
BF16_BOUNDS = {"z": 1.2e-3, "image_from_z": 4.4e-3}


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
def test_bf16_engine_matches_emulating_oracle(params):
    lrn = _learner(params, "bf16")
    p = _oracle_params(lrn)
    B, labels, alphas = 7, [17, 3, 9], ALPHAS
    x, y, _, eps, c = _inputs(B)
    worst = dict(z=0.0, image_from_z=0.0)
    for mode, sample in MODES:
        img, z = _walk(lrn, mode, x, y, eps, c, sample, labels, alphas)
        with O.bf16_emulation():
            _, z_o = _oracle(p, mode, x, y, eps, c, sample, labels, alphas)
            img_z = O.decoder(p, z.reshape(-1, 45).cpu().double()).reshape(img.shape)
        e = dict(z=rel_err(z, z_o), image_from_z=rel_err(img, img_z))
        print("bf16 {} {} sample={}: z {:.2e}, image from the engine's z {:.2e}".format(params, mode, sample, e["z"],
                                                                                       e["image_from_z"]))
        worst = {k: max(worst[k], e[k]) for k in worst}
    img = lrn.swap(x, x.flip(0))
    torch.cuda.synchronize()
    with O.bf16_emulation():
        _, z_o = WO.swap(p, x.double(), x.flip(0).double())
        img_z = O.decoder(p, lrn.last["z"].cpu().double())
    worst["z"] = max(worst["z"], rel_err(lrn.last["z"], z_o))
    worst["image_from_z"] = max(worst["image_from_z"], rel_err(img, img_z))
    print("bf16 {} worst: {}".format(params, worst))
    assert worst["z"] <= BF16_BOUNDS["z"] and worst["image_from_z"] <= BF16_BOUNDS["image_from_z"], worst


@pytest.mark.parametrize("precision", PRECISIONS)
def test_exact_known_answers(precision):
    x, y, _, eps, c = _inputs(8)
    lrn = _learner("trained_like", precision)
    for sample in (False, True):
        noise = {"eps": eps} if sample else None
        for l, v in ((0, 0), (7, 1), (17, 0)):
            # label l is v in every image: the one frame at alpha = 1 - v is `intervene` with label l flipped
            yl = y.clone()
            yl[:, l] = v
            w = lrn.walk(x, y=yl, labels=[l], alphas=[1.0 - v], sample=sample, c=c, noise=noise)
            zw = lrn.last["z"]
            assert torch.equal(lrn.last["y_src"].cpu().long(), yl) and w.shape == (8, 1, 1, 64, 64, 3)
            yf = yl.clone()
            yf[:, l] = 1 - v
            i = lrn.intervene(x, yf, y=yl, sample=sample, c=c, noise=noise)
            assert torch.equal(zw[:, 0, 0], lrn.last["z"]) and torch.equal(w[:, 0, 0], i)
            # from labels, alpha in {0, 1} is `generate` with y_l = alpha
            for a in (0, 1):
                ya = y.clone()
                ya[:, l] = a
                g = lrn.generate(ya, sample=sample, c=c, noise=noise)
                zg = lrn.last["z"]
                wg = lrn.walk(y=y, labels=[l], alphas=[float(a)], sample=sample, c=c, noise=noise)
                assert torch.equal(lrn.last["z"][:, 0, 0], zg) and torch.equal(wg[:, 0, 0], g)
        # the frame at alpha = y_src,l is the reconstruction, also with y defaulting to the classifier's decision
        r = lrn.reconstruct(x, sample=sample, noise=noise)
        zr = lrn.last["z"]
        for y_given in (y, None):
            w = lrn.walk(x, y=y_given, labels=[4, 12], alphas=[0.0, 1.0], sample=sample, c=c, noise=noise)
            zw, ys = lrn.last["z"], lrn.last["y_src"].long()
            ar = torch.arange(8, device="cuda")
            for li, l in enumerate((4, 12)):
                assert torch.equal(zw[ar, li, ys[:, l]], zr) and torch.equal(w[ar, li, ys[:, l]], r)
    # uint8 output = to_u8 of the fp32 output; the same noise and c twice give the same bits
    f = lrn.walk(x, labels=[1, 5], alphas=ALPHAS, sample=True, c=c, noise={"eps": eps})
    f2 = lrn.walk(x, labels=[1, 5], alphas=ALPHAS, sample=True, c=c, noise={"eps": eps})
    u = lrn.walk(x, labels=[1, 5], alphas=ALPHAS, sample=True, c=c, noise={"eps": eps}, dtype=torch.uint8)
    torch.cuda.synchronize()
    assert torch.equal(f, f2) and u.dtype == torch.uint8 and u.shape == f.shape and u.is_contiguous()
    assert np.array_equal(u.cpu().numpy(), GO.to_u8(f.cpu().numpy()))
    # swap(x, x) is the reconstruction; swap's z halves are those of the two reconstructions
    r = lrn.reconstruct(x)
    zr = lrn.last["z"]
    assert torch.equal(lrn.swap(x, x), r) and torch.equal(lrn.last["z"], zr)
    x2 = x.flip(0)
    lrn.reconstruct(x2)
    zr2 = lrn.last["z"]
    lrn.swap(x, x2)
    assert torch.equal(lrn.last["z"][:, :ZS], zr[:, :ZS]) and torch.equal(lrn.last["z"][:, ZS:], zr2[:, ZS:])
    # one-one gates: c = I exactly, walking label l moves classify dim l only
    oo = _learner("trained_like", precision, mode="one-one")
    oo.reconstruct(x)
    zr = oo.last["z"]
    oo.walk(x, y=y, labels=[0, 9, 17], alphas=[-0.5, 0.3, 1.5])
    torch.cuda.synchronize()
    assert torch.equal(oo.last["c"], torch.eye(18, device="cuda"))
    for li, l in enumerate((0, 9, 17)):
        keep = [d for d in range(45) if d != ZS + l]
        zl = oo.last["z"][:, li]
        assert torch.equal(zl[..., keep], zr[:, None, keep].expand(-1, 3, -1))
        assert not torch.equal(zl[..., ZS + l], zr[:, None, ZS + l].expand(-1, 3))
    # fresh-init prior: every frame is the reconstruction, bitwise at the image level
    fr = _learner("fresh", precision)
    r = fr.reconstruct(x)
    w = fr.walk(x, labels=[2, 11], alphas=ALPHAS, c=c)
    torch.cuda.synchronize()
    assert torch.equal(w, r[:, None, None].expand_as(w))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_chunking_changes_no_bit(precision):
    lrn = _learner("trained_like", precision)
    x, y, _, eps, c = _inputs(3)
    labels, alphas = [5, 0], [-0.5, 0.0, 0.6, 1.0]
    for mode, sample in MODES:
        outs = []
        for max_rows in (1, 7, 3 * 2 * 4):
            img, z = _walk(lrn, mode, x, y, eps, c, sample, labels, alphas, max_rows=max_rows)
            outs.append((img, z.clone()))
        for img, z in outs[1:]:
            assert torch.equal(z, outs[0][1]), (mode, sample)
            assert torch.equal(img, outs[0][0]), (mode, sample)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B", [1, 7, 256])
def test_batch_sizes(precision, B):
    lrn = _learner("trained_like", precision)
    x, y, _, eps, c = _inputs(B)
    xu8 = (x * 255).round().to(torch.uint8)          # uint8 images are accepted too
    labels, alphas = [16, 2, 8], [0.0, 0.5, 1.0]
    max_rows = max(1, B * 9 // 4)                     # several chunks, the last one short
    for dtype in (torch.float32, torch.uint8):
        w = lrn.walk(xu8, y=y, labels=labels, alphas=alphas, c=c, dtype=dtype, max_rows=max_rows)
        assert lrn.last["y_src"].dtype == torch.int32 and torch.equal(lrn.last["y_src"].cpu().long(), y)
        g = lrn.walk(y=y, labels=labels, alphas=alphas, c=c, noise={"eps": eps}, dtype=dtype, max_rows=max_rows)
        assert lrn.last["y_src"] is None and lrn.last["z"].shape == (B, 3, 3, 45)
        s = lrn.swap(xu8, x.flip(0), dtype=dtype)
        torch.cuda.synchronize()
        for t in (w, g):
            assert t.shape == (B, 3, 3, 64, 64, 3) and t.dtype == dtype and t.is_contiguous() and t.is_cuda
        assert s.shape == (B, 64, 64, 3) and s.dtype == dtype and s.is_contiguous()
        if dtype == torch.float32:
            assert all(bool(torch.isfinite(t).all()) and float(t.min()) >= 0.0 and float(t.max()) <= 1.0
                       for t in (w, g, s))
            w32, g32, s32 = w, g, s
        else:
            for t, t32 in ((w, w32), (g, g32), (s, s32)):
                assert np.array_equal(t.cpu().numpy(), GO.to_u8(t32.cpu().numpy()))
    # default labels and alphas: all 18 labels, 8 points from 0 to 1
    d = lrn.walk(xu8[:1])
    torch.cuda.synchronize()
    assert d.shape == (1, 18, 8, 64, 64, 3)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_noise_is_fresh_per_call_and_a_given_c_is_used_verbatim(precision):
    x, y, _, eps, c = _inputs(4)
    lrn = _learner("trained_like", precision)
    a = lrn.walk(y=y, labels=[3], alphas=[0.5])
    ca = lrn.last["c"]
    b_ = lrn.walk(y=y, labels=[3], alphas=[0.5])
    cb = lrn.last["c"]
    torch.cuda.synchronize()
    assert not torch.equal(a, b_) and not torch.equal(ca, cb)
    assert not torch.equal(lrn.walk(x, labels=[3], alphas=[0.5], sample=True, c=c),
                           lrn.walk(x, labels=[3], alphas=[0.5], sample=True, c=c))
    for call in (lambda: lrn.walk(y=y, labels=[3], c=c), lambda: lrn.walk(x, labels=[3], c=c)):
        call()
        torch.cuda.synchronize()
        assert torch.equal(lrn.last["c"].cpu(), c)


def test_bad_arguments_raise_value_error():
    lrn = _learner("trained_like", "bf16")
    x, y, _, eps, c = _inputs(4)
    bad = [
        lambda: lrn.walk(),
        lambda: lrn.walk(y=y[:, :17]),
        lambda: lrn.walk(x, y=y[:3]),
        lambda: lrn.walk(x[:, :32]),
        lambda: lrn.walk(x, labels=[]),
        lambda: lrn.walk(x, labels=[18]),
        lambda: lrn.walk(x, labels=[-1]),
        lambda: lrn.walk(x, labels=[2, 2]),
        lambda: lrn.walk(x, labels=[1.5]),
        lambda: lrn.walk(x, labels=[[1, 2]]),
        lambda: lrn.walk(x, alphas=[]),
        lambda: lrn.walk(x, alphas=[[0.0, 1.0]]),
        lambda: lrn.walk(x, alphas=[0.0, float("nan")]),
        lambda: lrn.walk(x, alphas=[float("inf")]),
        lambda: lrn.walk(x, alphas=[1e39]),
        lambda: lrn.walk(x, alphas=["a"]),
        lambda: lrn.walk(x, dtype=torch.float16),
        lambda: lrn.walk(x, c=c[:17]),
        lambda: lrn.walk(x, noise={"eps": eps[:3]}),
        lambda: lrn.walk(x, noise={"U1": eps}),
        lambda: lrn.walk(x, max_rows=0),
        lambda: lrn.walk(x, max_rows=2.5),
        lambda: lrn.swap(x, x[:3]),
        lambda: lrn.swap(x[:, :32], x),
        lambda: lrn.swap(x[:0], x[:0]),
        lambda: lrn.swap(x, x, dtype=torch.int32),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
            pytest.fail("case {} did not raise".format(i))
