"""GPU: the importance-weighted log-likelihood - Learner.log_likelihood / test_log_likelihood (gccvae_iw_latent, the
decoder, gccvae_convt_ll_bf16 on the bf16 engine, gccvae_iw_accumulate) - against the fp64 restatement of
tests/likelihood_oracle.py, the likelihood kernel alone, invariances, noise handling, argument checks and a consistency
check on the shipped trained checkpoint."""
import os

import numpy as np
import pytest
import torch

import gccvae_oracle as O
import likelihood_oracle as LO
from helpers import GOLDEN, cfg_for, make_learner, rel_err

pytestmark = pytest.mark.gpu
CKPT = os.path.join(GOLDEN, "models", "params_0.2_learnable")
PRECISIONS = ["fp32", "bf16"]


def _learner(params, precision, mode="inferred"):
    """params: 'trained_like' (O.init_params(0, trained_like=True)) or 'checkpoint' (run under gate mode `mode`)."""
    import gccvae_b200 as G
    if params == "checkpoint":
        cfg = cfg_for(mode, "0.2")
        lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 0.2, cfg, precision=precision)
        lrn.load_model(CKPT, "best")
        return lrn
    return make_learner(cfg_for(mode, "0.2"), O.init_params(0, trained_like=True), precision=precision)


def _oracle_params(lrn):
    p = {k: v.detach().double() for k, v in lrn.store.to_dict().items()}
    p.pop("mu")
    return p


def _inputs(B, K, seed=5):
    x, y, noise = O.make_inputs(B, k=1, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    eps = torch.randn(K, B, 45, generator=g)
    U_y = torch.rand(K, B, 18, generator=g)
    mu = torch.as_tensor(np.load(os.path.join(GOLDEN, "data", "gating_matrix_0.2.npy")))
    c = O.sample_gating_parameter(mu.float(), 0.3, noise["U1"], noise["U2"])   # fp32 c, passed verbatim
    return x, y, eps, U_y, c


def _oracle(p, x, y, eps, U_y, c, labelled):
    """fp64 oracle on the device (the decoder over K x B rows is too slow for the host at these sizes)."""
    d = lambda t: t.cuda().double()
    return LO.log_likelihood(p, d(x), d(c), d(eps), y.cuda() if labelled else None, d(U_y))


def _safe_uy(p, x, eps, U_y, c):
    """U_y moved 2e-3 away from the classifier's probability where it lies within 1e-3 of it, so that fp32 and fp64
    draw the same labels (a label on the threshold flips between precisions and changes log w by nats)."""
    d = lambda t: t.cuda().double()
    t = LO.log_weight_terms(p, d(x), d(c), d(eps), None, d(U_y), decode=False)
    s = torch.sigmoid(t["logits"]).float().cpu()
    near = (U_y - s).abs() < 1e-3
    moved = torch.where(U_y < s, s - 2e-3, s + 2e-3).clamp(0.0, 0.999)
    return torch.where(near, moved, U_y)


def _call(lrn, x, y, eps, U_y, c, labelled, **kw):
    est = lrn.log_likelihood(x, y if labelled else None, k=eps.shape[0], c=c, noise={"eps": eps, "U_y": U_y}, **kw)
    torch.cuda.synchronize()
    return est


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
@pytest.mark.parametrize("B", [8, 32])
def test_fp32_engine_matches_fp64_oracle(params, B):
    lrn = _learner(params, "fp32")
    p = _oracle_params(lrn)
    for K in (1, 7, 64):
        x, y, eps, U_y, c = _inputs(B, K)
        U_y = _safe_uy(p, x, eps, U_y, c)
        for labelled in (True, False):
            est = _call(lrn, x, y, eps, U_y, c, labelled, keep_log_w=True)
            est_o, ess_o, lw_o = _oracle(p, x, y, eps, U_y, c, labelled)
            e, ew, es = rel_err(est, est_o), rel_err(lrn.last["log_w"], lw_o), rel_err(lrn.last["ess"], ess_o)
            print("fp32 {} B={} K={} labelled={}: estimate {:.2e}, log_w {:.2e}, ess {:.2e}".format(
                params, B, K, labelled, e, ew, es))
            assert est.shape == (B,) and est.dtype == torch.float32 and est.is_cuda
            assert e <= 1e-5 and ew <= 1e-5, (K, labelled, e, ew)


# bf16 engine vs the oracle that rounds where the kernels do.  One known cause of difference: the decoder's operand is z
# rounded to bf16, while the density terms use the fp32 z; where the device's z and the oracle's z round to different
# bf16 values the trained decoder amplifies the step (tests/test_gpu_generation.py: images up to 1.9e-2 on the
# checkpoint) and log p(x|z), a sum over 12288 pixels, moves with it.
# Measured on B200 (1000 W), B = 16, K = 7, largest over labelled / unlabelled of the estimate and log w:
#   trained-like parameters 3.1e-7 (0.004 nats at most), shipped checkpoint 1.71e-4 (log w up to 2.0 nats apart,
#   the estimate 8.2e-5).  Bounds: ~1.5x those.
BF16_BOUNDS = {"trained_like": 5e-7, "checkpoint": 2.6e-4}


@pytest.mark.parametrize("params", ["trained_like", "checkpoint"])
def test_bf16_engine_matches_emulating_oracle(params):
    lrn = _learner(params, "bf16")
    p = _oracle_params(lrn)
    B, K = 16, 7
    x, y, eps, U_y, c = _inputs(B, K)
    U_y = _safe_uy(p, x, eps, U_y, c)
    worst = 0.0
    for labelled in (True, False):
        est = _call(lrn, x, y, eps, U_y, c, labelled, keep_log_w=True)
        with O.bf16_emulation():
            est_o, _, lw_o = _oracle(p, x, y, eps, U_y, c, labelled)
        e, ew = rel_err(est, est_o), rel_err(lrn.last["log_w"], lw_o)
        print("bf16 {} labelled={}: estimate {:.2e}, log_w {:.2e} (max |diff| {:.3f} nats)".format(
            params, labelled, e, ew, float((lrn.last["log_w"].double() - lw_o).abs().max())))
        worst = max(worst, e, ew)
    assert worst <= BF16_BOUNDS[params], worst


def test_likelihood_kernel_alone_against_fp64_and_the_recon_kernel():
    import gccvae_b200._lib as L
    lrn = _learner("trained_like", "bf16")
    eng = lrn.engine
    eng.pack_weights()
    B, kc = 4, 3
    rows = B * kc
    g = torch.Generator().manual_seed(7)
    g4 = (torch.rand(rows, 32, 32, 32, generator=g) * 0.5).to(torch.bfloat16).cuda()
    x = torch.rand(B, 64, 64, 3, generator=g).cuda()
    xu8 = (x * 255).round().to(torch.uint8)
    st = torch.cuda.current_stream().cuda_stream
    w, bias = L.ptr(eng.wp["dec.conv5t.x2t"]), L.ptr(lrn.store.view("dec.conv5t.b"))
    ln2 = -12288.0 * 0.6931471805599453

    def prep(img):    # x2 blocks + raw-byte blocks of uint8 images
        n = img.shape[0]
        x2 = torch.zeros(n * 33 * 33 * 24, dtype=torch.bfloat16, device="cuda")
        L.check(eng.lib.gccvae_prep_x2_bf16(L.ptr(img), 1, n, L.ptr(x2), eng.xb_ptr(x2, n), st), "prep_x2")
        return x2

    def ll(img, form):
        out = torch.full((rows,), ln2, dtype=torch.float32, device="cuda")
        src = eng.xb_ptr(prep(img), B) if form == 2 else L.ptr(img)
        L.check(eng.lib.gccvae_convt_ll_bf16(rows, kc, L.ptr(g4), w, bias, src, form, L.ptr(out), st), "convt_ll")
        return out

    def recon(img, form):
        rep = img.repeat_interleave(kc, 0).contiguous()
        out = torch.empty(rows, dtype=torch.float32, device="cuda")
        src = eng.xb_ptr(prep(rep), rows) if form == 2 else L.ptr(rep)
        L.check(eng.lib.gccvae_convt_recon_bf16(rows, L.ptr(g4), w, bias, src, form, None, L.ptr(out), None, None, None,
                                                0, st), "convt_recon")
        torch.cuda.synchronize()     # (`rep` and its blocks live until here)
        return out

    w16 = lrn.store.view("dec.conv5t.w").detach().cpu().to(torch.bfloat16).double()
    xhat = torch.sigmoid(O._convT(g4.cpu().double(), w16, lrn.store.view("dec.conv5t.b").detach().cpu().double(), 2, 1))
    for img, form in ((x, 0), (xu8, 1), (xu8, 2)):
        got = ll(img, form)
        want_rec = recon(img, form)
        xr = (img.cpu().double() / 255.0 if img.dtype == torch.uint8 else img.cpu().double()).repeat_interleave(kc, 0)
        want64 = O.img_log_likelihood(xhat, xr)
        e64, erec = rel_err(got, want64), rel_err(got, want_rec)
        print("likelihood kernel, image form {}: vs fp64 {:.2e}, vs convt_recon {:.2e}".format(form, e64, erec))
        # measured on B200: 3.1e-7 .. 3.6e-7 vs fp64 and 8.4e-8 vs convt_recon for the three forms (fp32 accumulation of
        # 12288 terms with the approximate sigmoid of convt_recon; float atomics across CTAs)
        assert e64 <= 1e-6 and erec <= 1e-6, (form, e64, erec)


def test_chunking_and_batch_do_not_change_the_estimate():
    lrn = _learner("trained_like", "bf16")
    B, K = 8, 100
    x, y, eps, U_y, c = _inputs(B, K)
    for labelled in (True, False):
        big = _call(lrn, x, y, eps, U_y, c, labelled)
        small = _call(lrn, x, y, eps, U_y, c, labelled, max_rows=64)        # 8 samples per image and chunk: 13 chunks
        assert rel_err(small, big) <= 1e-6, rel_err(small, big)
        # an image's estimate does not depend on the batch it is in (explicit noise sliced along B)
        part = lrn.log_likelihood(x[2:5], y[2:5] if labelled else None, k=K, c=c,
                                  noise={"eps": eps[:, 2:5], "U_y": U_y[:, 2:5]})
        assert rel_err(part, big[2:5]) <= 1e-6, rel_err(part, big[2:5])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_philox_mode_equals_explicit_mode_and_noise_is_fresh(precision):
    import gccvae_b200._lib as L
    from gccvae_b200 import dp
    lrn = _learner("trained_like", precision)
    B, K = 6, 9
    x, y, eps, U_y, c = _inputs(B, K)
    # the next call's Philox counter offset (gated_ccvae.Learner._fresh_noise; the step counter is 0)
    offset = (lrn._eval_calls + 1) << 32
    philox = lrn.log_likelihood(x, k=K, c=c)
    seed = dp.data_seed(lrn.seed, lrn.rank)
    draws = {}
    for kind, name, w in ((4, "eps", 45), (5, "U_y", 18)):
        t = torch.empty(K, B, w, dtype=torch.float32, device="cuda")
        L.check(lrn.lib.gccvae_draw_noise_f32(kind, seed, offset, B, K, L.ptr(t), torch.cuda.current_stream().cuda_stream),
                "draw_noise")
        draws[name] = t
    explicit = lrn.log_likelihood(x, k=K, c=c, noise=draws)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(draws["eps"]).all()) and float(draws["U_y"].min()) >= 0 and float(draws["U_y"].max()) < 1
    assert rel_err(explicit, philox) <= 1e-6, rel_err(explicit, philox)
    # without noise two calls differ; with the same noise and c they agree (up to the order of float atomics)
    a, b = lrn.log_likelihood(x, k=K), lrn.log_likelihood(x, k=K)
    assert not torch.equal(a, b)
    a = lrn.log_likelihood(x, k=K, c=c, noise={"eps": eps, "U_y": U_y})
    b = lrn.log_likelihood(x, k=K, c=c, noise={"eps": eps, "U_y": U_y})
    assert rel_err(a, b) <= 1e-6
    assert torch.equal(lrn.last["c"].cpu(), c) and lrn.last["log_w"] is None and lrn.last["ess"].shape == (B,)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B", [1, 7, 1024])
def test_batch_sizes(precision, B):
    lrn = _learner("trained_like", precision)
    x, y, _, _, _ = _inputs(B, 1)
    xu8 = (x * 255).round().to(torch.uint8)
    for xin, lab in ((x, None), (xu8, y)):
        est = lrn.log_likelihood(xin, lab, k=100)
        ess = lrn.last["ess"]
        torch.cuda.synchronize()
        assert est.shape == (B,) and est.dtype == torch.float32 and est.is_cuda and est.is_contiguous()
        assert bool(torch.isfinite(est).all()) and bool(((ess >= 1.0 - 1e-4) & (ess <= 100.0 + 1e-3)).all())


def test_bad_arguments_raise_value_error():
    lrn = _learner("trained_like", "bf16")
    x, y, eps, U_y, c = _inputs(4, 3)
    bad = [
        lambda: lrn.log_likelihood(x, k=0),
        lambda: lrn.log_likelihood(x, k=2.5),
        lambda: lrn.log_likelihood(x, max_rows=0),
        lambda: lrn.log_likelihood(x[:0]),
        lambda: lrn.log_likelihood(x[:, :32]),
        lambda: lrn.log_likelihood(x, y[:3]),
        lambda: lrn.log_likelihood(x, y[:, :17]),
        lambda: lrn.log_likelihood(x, k=3, noise={"eps": eps[:2]}),
        lambda: lrn.log_likelihood(x, k=3, noise={"eps": eps[..., :18]}),
        lambda: lrn.log_likelihood(x, k=3, noise={"U_y": U_y[:, :3]}),
        lambda: lrn.log_likelihood(x, k=3, noise={"U1": eps}),
        lambda: lrn.log_likelihood(x, c=c[:17]),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
            pytest.fail("case {} did not raise".format(i))


class _Loader:
    """in-memory stand-in for the reader: `.n_s` samples, `.step()` yields (xs, ys) batches, the last one short."""

    def __init__(self, x, y, batch_size):
        self.x, self.y, self.n_s, self.bs = x, y, x.shape[0], batch_size

    def step(self):
        for i in range(0, self.n_s, self.bs):
            yield self.x[i:i + self.bs], self.y[i:i + self.bs]


@pytest.mark.parametrize("mode", ["one-one", "learnable"])
def test_checkpoint_scores_its_own_images_above_noise(mode):
    lrn = _learner("checkpoint", "bf16", mode=mode)
    B = 256
    g = torch.Generator().manual_seed(11)
    y = (torch.rand(B, 18, generator=g) < 0.5).long().cuda()
    own = lrn.generate(y, dtype=torch.uint8)
    noise_img = torch.randint(0, 256, (B, 64, 64, 3), generator=g, dtype=torch.uint8).cuda()
    ll_own = lrn.log_likelihood(own, k=100)
    ll_noise = lrn.log_likelihood(noise_img, k=100)
    ll_own_y = lrn.log_likelihood(own, y, k=100)
    m_own, m_noise, m_own_y = float(ll_own.mean()), float(ll_noise.mean()), float(ll_own_y.mean())
    # measured on B200: one-one -9281.5 (own) vs -12105.2 (noise), learnable -9285.2 vs -11746.1 nats per image
    print("{}: mean log p(x) of generate(y) {:.1f} nats, of uniform noise {:.1f}; mean log p(x, y) of generate(y) "
          "{:.1f}; mean ESS {:.2f}".format(mode, m_own, m_noise, m_own_y, float(lrn.last["ess"].mean())))
    assert m_own > m_noise + 100.0 and bool((ll_own > ll_noise.max()).float().mean() > 0.9)
    if mode == "one-one":
        assert torch.equal(lrn.last["c"], torch.eye(18, device="cuda"))
    # test_log_likelihood over a two-batch loader (256 + 128 images) = the image-weighted mean of the two calls
    xs = torch.cat([own, noise_img[:128]])
    ys = torch.cat([y, y[:128]])
    lrn.train_config["batch_size"] = 256
    calls0 = lrn._eval_calls
    mean, per_px, c = lrn.test_log_likelihood(_Loader(xs, ys, 256), k=100, labelled=True)
    # the same per-call Philox offsets again: skip the gate draw's, then the two batches in order
    lrn._eval_calls = calls0 + 1
    a = lrn.log_likelihood(xs[:256], ys[:256], k=100, c=c)
    b = lrn.log_likelihood(xs[256:], ys[256:], k=100, c=c)
    want = (float(a.double().sum()) + float(b.double().sum())) / 384
    print("{}: test_log_likelihood {:.3f} nats per image, {:.5f} per pixel value".format(mode, mean, per_px))
    assert abs(mean - want) <= 1e-6 * abs(want) and abs(per_px - mean / 12288) <= 1e-12 * abs(mean)
