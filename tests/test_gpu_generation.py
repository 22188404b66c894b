"""GPU: the generation path - Learner.generate / reconstruct / intervene (gccvae_gen_latent + the decoder + on the bf16
engine gccvae_convt_image_bf16) - against the fp64 restatement of tests/generation_oracle.py, its exact known answers
on both engines, its noise handling and argument checks, and a consistency check on the shipped trained checkpoint."""
import os

import numpy as np
import pytest
import torch

import generation_oracle as GO
import gccvae_oracle as O
from helpers import GOLDEN, cfg_for, make_learner, rel_err

pytestmark = pytest.mark.gpu
CKPT = os.path.join(GOLDEN, "models", "params_0.2_learnable")
PRECISIONS = ["fp32", "bf16"]


def _learner(params, precision, mode="inferred", **kw):
    """params: 'trained_like' (O.init_params(0, trained_like=True)), 'fresh' (Keras initialisers) or 'checkpoint'."""
    import gccvae_b200 as G
    if params == "checkpoint":
        lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 0.2, cfg_for("learnable", "0.2"), precision=precision, **kw)
        lrn.load_model(CKPT, "best")
        return lrn
    return make_learner(cfg_for(mode, "0.2"), O.init_params(0, trained_like=params == "trained_like"),
                        precision=precision, **kw)


def _oracle_params(lrn):
    p = {k: v.detach().cpu().double() for k, v in lrn.store.to_dict().items()}
    p.pop("mu")
    return p


def _inputs(B, seed=5):
    x, y, noise = O.make_inputs(B, k=1, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    y_new = y.clone()
    flip = torch.rand(B, 18, generator=g) < 0.3
    y_new[flip] = 1 - y_new[flip]
    mu = torch.as_tensor(np.load(os.path.join(GOLDEN, "data", "gating_matrix_0.2.npy")))
    c = O.sample_gating_parameter(mu.float(), 0.3, noise["U1"], noise["U2"])   # fp32 c, passed verbatim
    return x, y, y_new, noise["eps"], c


def _run(lrn, mode, x, y, y_new, eps, c, sample, dtype=torch.float32):
    noise = {"eps": eps} if sample else None
    if mode == "generate":
        img = lrn.generate(y_new, sample=sample, c=c, noise=noise, dtype=dtype)
    elif mode == "reconstruct":
        img = lrn.reconstruct(x, sample=sample, noise=noise, dtype=dtype)
    else:
        img = lrn.intervene(x, y_new, y=y, sample=sample, c=c, noise=noise, dtype=dtype)
    torch.cuda.synchronize()
    return img, lrn.last["z"]


def _oracle(p, mode, x, y, y_new, eps, c, sample):
    e = eps.double() if sample else None
    if mode == "generate":
        return GO.generate(p, y_new, c.double(), e)
    if mode == "reconstruct":
        return GO.reconstruct(p, x.double(), e)
    img, z, _ = GO.intervene(p, x.double(), y_new, c.double(), y=y, eps=e)
    return img, z


MODES = [("generate", True), ("generate", False), ("reconstruct", False), ("reconstruct", True), ("intervene", False),
         ("intervene", True)]


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
@pytest.mark.parametrize("B", [8, 32])
def test_fp32_engine_matches_fp64_oracle(params, B):
    lrn = _learner(params, "fp32")
    p = _oracle_params(lrn)
    x, y, y_new, eps, c = _inputs(B)
    for mode, sample in MODES:
        img, z = _run(lrn, mode, x, y, y_new, eps, c, sample)
        img_o, z_o = _oracle(p, mode, x, y, y_new, eps, c, sample)
        ei, ez = rel_err(img, img_o), rel_err(z, z_o)
        print("fp32 {} B={} {} sample={}: image {:.2e}, z {:.2e}".format(params, B, mode, sample, ei, ez))
        assert img.shape == (B, 64, 64, 3) and img.dtype == torch.float32 and img.is_contiguous()
        assert ei <= 1e-5 and ez <= 1e-5, (mode, sample, ei, ez)
    # default source labels: the classifier's decision on z_c (compared where the fp64 logit is not at the threshold)
    img = lrn.intervene(x, y_new, c=c)
    torch.cuda.synchronize()
    y_src = lrn.last["y_src"].cpu().long()
    _, z_o = GO.reconstruct(p, x.double())
    y_o, logits = GO.decision(p, z_o[:, 27:], c.double())
    clear = logits.abs() > 1e-4
    assert torch.equal(y_src[clear], y_o[clear])
    img_o, z_o, _ = GO.intervene(p, x.double(), y_new, c.double(), y=y_src)
    assert rel_err(img, img_o) <= 1e-5 and rel_err(lrn.last["z"], z_o) <= 1e-5


# bf16 engine vs the oracle that rounds where the kernels do (activations between the layers, bf16 weights, z -> the bf16
# operand of fc1), judged per stage: z against the oracle's z, the image against the emulating decoder applied to the
# engine's own z.  End to end the two stages compose through z's bf16 rounding: where the device's fp32 z and the
# oracle's z round to different bf16 values (a 2^-8 step; 1-5 % of the elements when an encoder produced z, none for
# generate), the trained checkpoint's decoder amplifies the step - end to end 1.4e-2 .. 1.9e-2 there (checkpoint,
# reconstruct / intervene), 4.4e-4 for generate; 8.2e-5 at most with the trained-like parameters.
# Measured on B200 (1000 W), largest over the six mode / sampling cases:
#   z:                    1.65e-3 (trained-like reconstruct without sampling, where max|z| is smallest), checkpoint 7.9e-5
#   image from own z:     2.63e-3 (checkpoint intervene without sampling), trained-like 6.7e-5
#   end to end, trained-like parameters: 8.17e-5
# Bounds: ~1.5x those.
BF16_BOUNDS = {"z": 2.5e-3, "image_from_z": 4e-3, "end_to_end_trained_like": 1.3e-4}


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
def test_bf16_engine_matches_emulating_oracle(params):
    lrn = _learner(params, "bf16")
    p = _oracle_params(lrn)
    B = 16
    x, y, y_new, eps, c = _inputs(B)
    worst = dict(z=0.0, image_from_z=0.0, end_to_end=0.0)
    for mode, sample in MODES:
        img, z = _run(lrn, mode, x, y, y_new, eps, c, sample)
        with O.bf16_emulation():
            img_o, z_o = _oracle(p, mode, x, y, y_new, eps, c, sample)
            img_z = O.decoder(p, z.cpu().double())
        e = dict(z=rel_err(z, z_o), image_from_z=rel_err(img, img_z), end_to_end=rel_err(img, img_o))
        flips = float((z.cpu().to(torch.bfloat16) != z_o.to(torch.bfloat16)).double().mean())
        print("bf16 {} {} sample={}: z {:.2e} (bf16 roundings that differ: {:.2%}), image from the engine's z {:.2e}, "
              "end to end {:.2e}".format(params, mode, sample, e["z"], flips, e["image_from_z"], e["end_to_end"]))
        worst = {k: max(worst[k], e[k]) for k in worst}
    assert worst["z"] <= BF16_BOUNDS["z"] and worst["image_from_z"] <= BF16_BOUNDS["image_from_z"], worst
    if params == "trained_like":
        assert worst["end_to_end"] <= BF16_BOUNDS["end_to_end_trained_like"], worst


def test_image_kernel_alone_against_fp64_and_the_decoder():
    import gccvae_b200._lib as L
    lrn = _learner("trained_like", "bf16")
    eng = lrn.engine
    B = 8
    z = torch.randn(B, 45, generator=torch.Generator().manual_seed(3)).cuda()
    eng.pack_weights()
    ref_dec = lrn.model.decoder(z)              # the generic conv5t path (gccvae_sl_bf16 family, fp32 out)
    b = eng.bufs(B)
    g4 = b["dec.conv4t.out"].clone()
    outs = {}
    for u8 in (0, 1):
        out = torch.empty(B, 64, 64, 3, dtype=torch.uint8 if u8 else torch.float32, device="cuda")
        L.check(eng.lib.gccvae_convt_image_bf16(B, L.ptr(g4), L.ptr(eng.wp["dec.conv5t.x2t"]),
                                                L.ptr(lrn.store.view("dec.conv5t.b")), L.ptr(out), u8,
                                                torch.cuda.current_stream().cuda_stream), "convt_image")
        outs[u8] = out
    torch.cuda.synchronize()
    w16 = lrn.store.view("dec.conv5t.w").detach().cpu().to(torch.bfloat16).double()
    bias = lrn.store.view("dec.conv5t.b").detach().cpu().double()
    want = torch.sigmoid(O._convT(g4.cpu().double(), w16, bias, 2, 1))
    d64 = float((outs[0].cpu().double() - want).abs().max())
    ddec = float((outs[0] - ref_dec).abs().max())
    print("image kernel: max|.| vs fp64 {:.3e}, vs Decoder(z) {:.3e}".format(d64, ddec))
    # measured on B200: 8.2e-8 and 1.2e-7 (about one ulp at 1.0: fp32 accumulation of 128 terms, approximate sigmoid)
    assert d64 <= 2e-7 and ddec <= 2e-7, (d64, ddec)
    assert np.array_equal(outs[1].cpu().numpy(), GO.to_u8(outs[0].cpu().numpy()))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_exact_known_answers(precision):
    x, y, y_new, eps, c = _inputs(8)
    lrn = _learner("trained_like", precision)
    # uint8 output = rint(255 * fp32 output) of the same engine, for every mode
    for mode, sample in MODES:
        f, _ = _run(lrn, mode, x, y, y_new, eps, c, sample)
        u, _ = _run(lrn, mode, x, y, y_new, eps, c, sample, dtype=torch.uint8)
        assert u.dtype == torch.uint8 and u.shape == f.shape and u.is_contiguous()
        assert np.array_equal(u.cpu().numpy(), GO.to_u8(f.cpu().numpy())), mode
        # same explicit noise and c twice: the same bits
        f2, _ = _run(lrn, mode, x, y, y_new, eps, c, sample)
        assert torch.equal(f, f2), mode
    # identity: intervening from y to y is the reconstruction (also with y defaulting to the classifier's decision)
    for sample in (False, True):
        r, zr = _run(lrn, "reconstruct", x, y, y_new, eps, c, sample)
        i, zi = _run(lrn, "intervene", x, y, y, eps, c, sample)
        assert torch.equal(zi, zr) and torch.equal(i, r)
        noise = {"eps": eps} if sample else None
        lrn.intervene(x, y, sample=sample, c=c, noise=noise)
        y_dec = lrn.last["y_src"].clone()
        i2 = lrn.intervene(x, y_dec, sample=sample, c=c, noise=noise)
        assert torch.equal(lrn.last["y_src"], y_dec) and torch.equal(i2, r)
    # one-one gates: c = I exactly, label j moves classify dim j only
    oo = _learner("trained_like", precision, mode="one-one")
    _, zr = _run(oo, "reconstruct", x, y, y_new, eps, None, False)
    for j in (0, 9, 17):
        yj = y.clone()
        yj[:, j] = 1 - yj[:, j]
        oo.intervene(x, yj, y=y)
        torch.cuda.synchronize()
        assert torch.equal(oo.last["c"], torch.eye(18, device="cuda"))
        keep = [d for d in range(45) if d != 27 + j]
        assert torch.equal(oo.last["z"][:, keep], zr[:, keep]) and not torch.equal(oo.last["z"][:, 27 + j], zr[:, 27 + j])
    # fresh-init prior: every intervention is the identity, bitwise at the image level
    fr = _learner("fresh", precision)
    r, _ = _run(fr, "reconstruct", x, y, y_new, eps, c, False)
    i, _ = _run(fr, "intervene", x, y, 1 - y, eps, None, False)
    assert torch.equal(i, r)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_noise_is_fresh_per_call_and_a_given_c_is_used_verbatim(precision):
    x, y, y_new, eps, c = _inputs(4)
    lrn = _learner("trained_like", precision)
    a = lrn.generate(y)
    ca = lrn.last["c"]
    b_ = lrn.generate(y)
    cb = lrn.last["c"]
    torch.cuda.synchronize()
    assert not torch.equal(a, b_) and not torch.equal(ca, cb)
    assert not torch.equal(lrn.reconstruct(x, sample=True), lrn.reconstruct(x, sample=True))
    for call in (lambda: lrn.generate(y, c=c), lambda: lrn.intervene(x, y_new, c=c)):
        call()
        torch.cuda.synchronize()
        assert torch.equal(lrn.last["c"].cpu(), c)
    # means do not depend on the noise: reconstruct(sample=False) is deterministic without `noise`
    assert torch.equal(lrn.reconstruct(x), lrn.reconstruct(x))


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B", [1, 7, 1024])
def test_batch_sizes(precision, B):
    lrn = _learner("trained_like", precision)
    x, y, y_new, eps, c = _inputs(B)
    xu8 = (x * 255).round().to(torch.uint8)          # uint8 images are accepted too
    for dtype in (torch.float32, torch.uint8):
        g = lrn.generate(y_new, c=c, noise={"eps": eps}, dtype=dtype)
        r = lrn.reconstruct(xu8, dtype=dtype)
        i = lrn.intervene(xu8, y_new, y=y, c=c, dtype=dtype)
        assert lrn.last["y_src"].dtype == torch.int32 and torch.equal(lrn.last["y_src"].cpu().long(), y)
        torch.cuda.synchronize()
        for t in (g, r, i):
            assert t.shape == (B, 64, 64, 3) and t.dtype == dtype and t.is_contiguous() and t.is_cuda
        if dtype == torch.float32:
            assert all(bool(torch.isfinite(t).all()) and float(t.min()) >= 0.0 and float(t.max()) <= 1.0 for t in (g, r, i))
            g32, r32 = g, r
        else:
            assert np.array_equal(g.cpu().numpy(), GO.to_u8(g32.cpu().numpy()))
            assert np.array_equal(r.cpu().numpy(), GO.to_u8(r32.cpu().numpy()))
    if B <= 7:      # against the (emulating, for bf16) fp64 oracle
        p = _oracle_params(lrn)
        with O.bf16_emulation(precision == "bf16"):
            want, _ = GO.generate(p, y_new, c.double(), eps.double())
        assert rel_err(g32, want) <= (1e-5 if precision == "fp32" else BF16_BOUNDS["end_to_end_trained_like"])


def test_bad_arguments_raise_value_error():
    lrn = _learner("trained_like", "bf16")
    x, y, y_new, eps, c = _inputs(4)
    bad = [
        lambda: lrn.generate(y[:, :17]),
        lambda: lrn.generate(y[0]),
        lambda: lrn.generate(y[:0]),
        lambda: lrn.generate(y, noise={"eps": eps[:3]}),
        lambda: lrn.generate(y, c=c[:17]),
        lambda: lrn.generate(y, dtype=torch.float16),
        lambda: lrn.reconstruct(x[:, :32]),
        lambda: lrn.intervene(x, y_new[:3]),
        lambda: lrn.intervene(x, y_new, y=y[:, :5]),
        lambda: lrn.intervene(x, y_new, noise={"U1": eps}),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
            pytest.fail("case {} did not raise".format(i))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_trained_model_generates_images_its_classifier_reads_as_the_target_labels(precision):
    lrn = _learner("checkpoint", precision)
    g = torch.Generator().manual_seed(11)
    y = (torch.rand(256, 18, generator=g) < 0.5).long().cuda()
    img = lrn.generate(y, sample=False)
    acc_y = float(lrn.classifier_accuracy(img, y))
    acc_not = float(lrn.classifier_accuracy(img, 1 - y))
    print("{}: classifier accuracy of generate(y) against y {:.4f}, against 1 - y {:.4f}".format(precision, acc_y, acc_not))
    # measured on B200: fp32 0.5098 / 0.4798, bf16 0.5098 / 0.4787
    assert acc_y > acc_not
