"""GPU: image completion - Learner.complete (the per-call body of the image calls once per iteration; on the bf16 engine
gccvae_convt_complete_bf16 writes each iteration's composite into the encoder's input blocks) - against the hand-written
loop of `reconstruct` / `intervene` calls with torch.where compositing, bit for bit on both engines; its exact identities;
the kernel alone against gccvae_convt_image_bf16 + where + gccvae_prep_x2_bf16; accuracy against the fp64 restatement of
tests/completion_oracle.py; argument checks."""
import numpy as np
import pytest
import torch

import completion_oracle as CO
import gccvae_oracle as O
from helpers import rel_err
from test_gpu_generation import BF16_BOUNDS, PRECISIONS, _inputs, _learner, _oracle_params

pytestmark = pytest.mark.gpu


def _mask(B, seed=3, p_obs=0.6):
    """random per-pixel mask [B,64,64] bool (True = observed), with a centred 24 x 24 hole in every image."""
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(B, 64, 64, generator=g) < p_obs
    m[:, 20:44, 20:44] = False
    return m


def _as(x, dtype):
    """x (fp32 in [0,1] or uint8) converted to dtype by the rules of the image calls."""
    if dtype == torch.uint8:
        return x if x.dtype == torch.uint8 else torch.clamp(torch.round(x * 255.0), max=255.0).to(torch.uint8)
    return x.to(torch.float32) / 255.0 if x.dtype == torch.uint8 else x


def _loop(lrn, x, m, T, y_new, y, sample, eps, c, dtype):
    """the completion written with the public calls: T reconstruct / intervene calls on the fp32 composite."""
    m4 = m.unsqueeze(-1)
    comp, xf = x, _as(x, torch.float32)
    for t in range(T):
        noise = {"eps": eps[t]} if eps is not None else None
        dt = dtype if t == T - 1 else torch.float32
        if y_new is None:
            img = lrn.reconstruct(comp, sample=sample, noise=noise, dtype=dt)
        else:
            img = lrn.intervene(comp, y_new, y=y, sample=sample, c=c, noise=noise, dtype=dt)
        comp = torch.where(m4, xf, img)
    return torch.where(m4, _as(x, dtype), img)


def _device_inputs(B, u8):
    x, y, y_new, _, c = _inputs(B)
    x = x.cuda()
    if u8:
        x = (x * 255).round().to(torch.uint8)
    return x, y.cuda(), y_new.cuda(), c.cuda()


LABELS = ["none", "y_new", "y_new_and_y"]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("T", [1, 3])
@pytest.mark.parametrize("labels", LABELS)
def test_matches_the_loop_of_public_calls_bitwise(precision, T, labels):
    lrn = _learner("trained_like", precision)
    B = 5
    m = _mask(B).cuda()
    eps = torch.randn(T, B, 45, generator=torch.Generator().manual_seed(9)).cuda()
    for u8 in (False, True):
        x, y, y_new, c = _device_inputs(B, u8)
        yn = None if labels == "none" else y_new
        ys = y if labels == "y_new_and_y" else None
        for sample in (False, True):
            e = eps if sample else None
            for dtype in (torch.float32, torch.uint8):
                got = lrn.complete(x, m, y_new=yn, y=ys, iters=T, sample=sample, c=c,
                                   noise=None if e is None else {"eps": e}, dtype=dtype)
                last = dict(lrn.last)
                want = _loop(lrn, x, m, T, yn, ys, sample, e, c, dtype)
                torch.cuda.synchronize()
                case = (u8, sample, dtype)
                assert got.shape == (B, 64, 64, 3) and got.dtype == dtype and got.is_contiguous(), case
                assert torch.equal(got, want), case
                assert torch.equal(last["z"], lrn.last["z"]), case
                assert torch.equal(last["c"], c), case
                if yn is None:
                    assert last["y_src"] is None
                else:
                    assert torch.equal(last["y_src"], lrn.last["y_src"]), case
                m4 = m.unsqueeze(-1).expand_as(got)
                assert torch.equal(got[m4], _as(x, dtype)[m4]), case


@pytest.mark.parametrize("precision", PRECISIONS)
def test_fresh_noise_matches_the_loop_bitwise(precision):
    lrn = _learner("trained_like", precision)
    B, T = 4, 3
    m = _mask(B).cuda()
    x, y, y_new, _ = _device_inputs(B, True)
    for yn in (None, y_new):
        e0 = lrn._eval_calls
        got = lrn.complete(x, m, y_new=yn, iters=T, sample=True)
        z, c = lrn.last["z"].clone(), lrn.last["c"].clone()
        lrn._eval_calls = e0
        # the loop's first call draws the gate; the others get it, as `complete` shares it
        comp, xf = x, _as(x, torch.float32)
        for t in range(T):
            if yn is None:
                img = lrn.reconstruct(comp, sample=True)
            else:
                img = lrn.intervene(comp, yn, sample=True, c=None if t == 0 else c)
            if t == 0:
                assert torch.equal(lrn.last["c"], c)
            comp = torch.where(m.unsqueeze(-1), xf, img)
        torch.cuda.synchronize()
        assert torch.equal(got, comp) and torch.equal(z, lrn.last["z"])
        assert lrn._eval_calls == e0 + T
    # and the noise differs between calls
    a = lrn.complete(x, m, iters=2, sample=True)
    b = lrn.complete(x, m, iters=2, sample=True)
    assert not torch.equal(a, b)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("u8", [False, True])
def test_exact_identities(precision, u8):
    lrn = _learner("trained_like", precision)
    B = 6
    x, y, y_new, c = _device_inputs(B, u8)
    ones = torch.ones(B, 64, 64, dtype=torch.bool)
    zeros = torch.zeros(B, 64, 64, dtype=torch.bool)
    r = lrn.reconstruct(x)
    z_r = lrn.last["z"].clone()
    for dtype in (torch.float32, torch.uint8):
        # all observed: x itself, and every iteration encodes x
        out = lrn.complete(x, ones, iters=3, dtype=dtype)
        assert torch.equal(out, _as(x, dtype)) and torch.equal(lrn.last["z"], z_r)
        # nothing observed, one iteration: reconstruct / intervene
        assert torch.equal(lrn.complete(x, zeros, iters=1, dtype=dtype), lrn.reconstruct(x, dtype=dtype))
        assert torch.equal(lrn.complete(x, zeros.numpy(), y_new=y_new, y=y, iters=1, c=c, dtype=dtype),
                           lrn.intervene(x, y_new, y=y, c=c, dtype=dtype))
    assert torch.equal(lrn.complete(x, zeros, iters=1), r)
    # a [64,64] mask is its expansion over the batch; integer masks are nonzero = observed
    m2 = _mask(1)[0]
    a = lrn.complete(x, m2, iters=2)
    b = lrn.complete(x, m2.expand(B, 64, 64).to(torch.int32) * 7, iters=2)
    assert torch.equal(a, b)


@pytest.mark.parametrize("B", [1, 3, 256])
def test_kernel_alone_against_image_where_and_prep_x2(B):
    import gccvae_b200._lib as L
    lrn = _learner("trained_like", "bf16")
    eng = lrn.engine
    eng.pack_weights()
    g = torch.Generator().manual_seed(B)
    g4 = torch.relu(torch.randn(B, 32, 32, 32, generator=g)).to(torch.bfloat16).cuda()
    m = torch.rand(B, 64, 64, generator=g) < 0.5
    m[0] = True                   # an image with nothing to rewrite
    if B > 1:
        m[1] = False              # and one with every pixel
    m = m.cuda()
    st = torch.cuda.current_stream().cuda_stream
    wp, bias = L.ptr(eng.wp["dec.conv5t.x2t"]), L.ptr(lrn.store.view("dec.conv5t.b"))
    img = torch.empty(B, 64, 64, 3, dtype=torch.float32, device="cuda")
    L.check(eng.lib.gccvae_convt_image_bf16(B, L.ptr(g4), wp, bias, L.ptr(img), 0, st), "convt_image")
    mb = eng.complete_begin(None, m)["mask_blocks"]
    n16 = B * 1089 * 16
    for u8 in (False, True):
        x = torch.rand(B, 64, 64, 3, generator=g)
        x = (x * 255).round().to(torch.uint8).cuda() if u8 else x.cuda()
        X2 = torch.full((B * 1089 * 24,), float("nan"), dtype=torch.bfloat16, device="cuda")
        L.check(eng.prep_x2(x, X2, st), "prep_x2")
        before = X2.clone()
        L.check(eng.lib.gccvae_convt_complete_bf16(B, L.ptr(g4), wp, bias, L.ptr(mb), L.ptr(X2), st), "convt_complete")
        want = torch.full_like(X2, float("nan"))
        comp = torch.where(m.unsqueeze(-1), _as(x, torch.float32), img)
        L.check(eng.prep_x2(comp, want, st), "prep_x2")
        torch.cuda.synchronize()
        v = lambda t: t.view(torch.int16)
        assert torch.equal(v(X2[:n16]), v(want[:n16])), u8
        # the raw-byte blocks of uint8 images (or, for fp32 images, the untouched tail) keep their bytes
        assert torch.equal(v(X2[n16:]), v(before[n16:])), u8
        # the all-observed image's blocks are untouched
        assert torch.equal(v(X2[:1089 * 16]), v(before[:1089 * 16]))


# fp32 engine vs the fp64 restatement.  Measured on B200 (1000 W), largest over reconstruct / intervene (with given y),
# sample False / True, B = 4 and 7, T = 1 and 3: image 5.75e-6 and z 1.90e-6 with the shipped checkpoint, 7.1e-8 and
# 2.2e-7 with the trained-like parameters (the image calls' 1e-5, which holds with ~1.7x margin).
FP32_BOUND = 1e-5


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
@pytest.mark.parametrize("B", [4, 7])
@pytest.mark.parametrize("T", [1, 3])
def test_fp32_engine_matches_fp64_oracle(params, B, T):
    lrn = _learner(params, "fp32")
    p = _oracle_params(lrn)
    x, y, y_new, _, c = _inputs(B)
    m = _mask(B)
    eps = torch.randn(T, B, 45, generator=torch.Generator().manual_seed(4))
    worst = 0.0
    for yn in (None, y_new):
        for sample in (False, True):
            e = eps if sample else None
            out = lrn.complete(x, m, y_new=yn, y=None if yn is None else y, iters=T, sample=sample, c=c,
                               noise=None if e is None else {"eps": e})
            z = lrn.last["z"]
            out_o, z_o, _ = CO.complete(p, x.double(), m, T, y_new=yn, c=c.double(), y=None if yn is None else y,
                                        eps=None if e is None else e.double())
            ei, ez = rel_err(out, out_o), rel_err(z, z_o)
            print("fp32 {} B={} T={} labels={} sample={}: image {:.2e}, z {:.2e}".format(
                params, B, T, yn is not None, sample, ei, ez))
            worst = max(worst, ei, ez)
    assert worst <= FP32_BOUND, worst


# Judged per iteration, as tests/test_gpu_generation.py judges one call (BF16_BOUNDS): measured on B200 (1000 W), largest
# over reconstruct / intervene, sample False / True and t = 1..3: z 1.30e-3 (trained-like, reconstruct without sampling),
# image from the engine's z 3.29e-3 (checkpoint, t = 1).
@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
def test_bf16_engine_matches_emulating_oracle_per_iteration(params):
    lrn = _learner(params, "bf16")
    p = _oracle_params(lrn)
    B, T = 16, 3
    x, y, y_new, _, c = _inputs(B)
    m = _mask(B)
    eps = torch.randn(T, B, 45, generator=torch.Generator().manual_seed(4))
    worst = dict(z=0.0, image_from_z=0.0)
    for yn in (None, y_new):
        for sample in (False, True):
            prev = x
            for t in range(1, T + 1):
                e = eps[:t] if sample else None
                out = lrn.complete(x, m, y_new=yn, y=None if yn is None else y, iters=t, sample=sample, c=c,
                                   noise=None if e is None else {"eps": e})
                z = lrn.last["z"].cpu().double()
                with O.bf16_emulation():
                    _, _, z_o, _ = CO.step(p, prev.cpu().double(), x.double(), m, y_new=yn, c=c.double(),
                                           y=None if yn is None else y, eps=None if e is None else e[t - 1].double())
                    img_z = torch.where(m.unsqueeze(-1), x.double(), O.decoder(p, z))
                err = dict(z=rel_err(z, z_o), image_from_z=rel_err(out, img_z))
                print("bf16 {} labels={} sample={} t={}: z {:.2e}, image from the engine's z {:.2e}".format(
                    params, yn is not None, sample, t, err["z"], err["image_from_z"]))
                worst = {k: max(worst[k], err[k]) for k in worst}
                prev = out
    assert worst["z"] <= BF16_BOUNDS["z"] and worst["image_from_z"] <= BF16_BOUNDS["image_from_z"], worst


def test_bad_arguments_raise_value_error():
    lrn = _learner("trained_like", "bf16")
    x, y, y_new, eps, c = _inputs(4)
    m = _mask(4)
    bad = [
        lambda: lrn.complete(x, m[:3]),
        lambda: lrn.complete(x, m[:, :32]),
        lambda: lrn.complete(x, m[0, 0]),
        lambda: lrn.complete(x, m[None]),
        lambda: lrn.complete(x, m.float()),
        lambda: lrn.complete(x, m, iters=0),
        lambda: lrn.complete(x, m, iters=2.0),
        lambda: lrn.complete(x, m, iters=True),
        lambda: lrn.complete(x, m, y=y),
        lambda: lrn.complete(x, m, y_new=y_new[:3]),
        lambda: lrn.complete(x, m, iters=2, sample=True, noise={"eps": eps}),
        lambda: lrn.complete(x, m, iters=2, sample=True, noise={"eps": eps[None].expand(3, -1, -1)}),
        lambda: lrn.complete(x, m, noise={"U1": eps}),
        lambda: lrn.complete(x, m, c=c[:17]),
        lambda: lrn.complete(x, m, dtype=torch.float16),
        lambda: lrn.complete(x[:, :32], m),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
            pytest.fail("case {} did not raise".format(i))
