"""CPU checks of tests/launch_reference.py: each reference, fed a launch snapshot built with the layout helpers from small
random tensors, agrees with the oracle's convolutions / autograd on the plain NHWC tensors; and the per-element check
catches the mistakes a subtly wrong kernel makes (one element a few bf16 ulps off, one weight-gradient split missing,
two s2d slots swapped, a NaN in a pad column) while an exactly rounded result passes."""
import math

import pytest
import torch

import gccvae_oracle as O
import launch_reference as R

B = 2
NAMES = [n for n, _ in O.PARAM_SHAPES]
SHAPES = dict(O.PARAM_SHAPES)


def bf(t):
    return t.to(torch.bfloat16)


def _flat_view(flat):
    out, off = {}, 0
    for n in NAMES:
        k = math.prod(SHAPES[n])
        out[n] = flat[off:off + k].view(SHAPES[n])
        off += k
    return out


def _ctx(**kw):
    p = O.init_params(0, trained_like=True)
    W = {k: v.to(torch.bfloat16).double() for k, v in p.items() if k.endswith(".w")}
    P = {k: v.double() for k, v in p.items()}
    return R.Ctx(W, P, _flat_view, **kw), p


def _act(g, *shape):
    return bf(torch.relu(torch.randn(*shape, generator=g)))


def _grad_buf(g):
    return torch.randn(sum(math.prod(s) for s in SHAPES.values()), generator=g) * 0.01


def _ok(op, pre, post, ctx, rows=B):
    res = R.check_launch(op, pre, post, ctx, rows)
    assert res, op
    return max(r for _, r in res), res


# ---- every reference against the oracle, through the layout helpers -----------------------------------------------
def _conv_case(op, g, ctx, p):
    """(pre, post) of a conv-type launch computed with the oracle on NHWC tensors (bf16 outputs rounded once)."""
    W = {k: v.double() for k, v in ctx.W.items()}
    name, kind = op.rsplit(" ", 1)
    s, pd = R.GEOM[name]
    b = p[name + ".b"].double()
    if op == "enc.conv2 fwd":
        h = _act(g, B, 32, 32, 32)
        want = torch.relu(O._conv(h.double(), W[name + ".w"], b, s, pd))
        return {"enc.conv1.out": R.s2d_blocks(h)}, {"enc.conv2.out": R.s2d_blocks(bf(want))}
    if op == "enc.conv4 fwd":
        h = _act(g, B, 8, 8, 64)
        want = torch.relu(O._conv(h.double(), W[name + ".w"], b, s, pd))
        return {"enc.conv3.out": R.s2d_blocks(h)}, {"enc.conv4.out": bf(want)}
    if op == "dec.conv3t fwd":
        h = _act(g, B, 8, 8, 64)
        want = torch.relu(O._convT(h.double(), W[name + ".w"], b, s, pd))
        return {"dec.conv2t.out": h}, {"dec.conv3t.out": bf(want)}
    if op == "enc.conv3 dgrad":
        h = _act(g, B, 16, 16, 32)
        d = bf(torch.randn(B, 8, 8, 64, generator=g))
        L = torch.zeros(B, 16, 16, 32, dtype=torch.float64, requires_grad=True)
        (O._conv(L, W[name + ".w"], None, s, pd) * d.double()).sum().backward()
        return ({"enc.conv3.dout": d, "enc.conv2.out": R.s2d_blocks(h)},
                {"enc.conv2.dout": bf(L.grad * (h.double() > 0))})
    if op == "dec.conv4t dgrad":
        h = _act(g, B, 16, 16, 32)
        d = bf(torch.randn(B, 32, 32, 32, generator=g))
        S = torch.zeros(B, 16, 16, 32, dtype=torch.float64, requires_grad=True)
        (O._convT(S, W[name + ".w"], None, s, pd) * d.double()).sum().backward()
        return ({"dec.conv4t.dout": R.s2d_blocks(d), "dec.conv3t.out": h},
                {"dec.conv3t.dout": R.s2d_blocks(bf(S.grad * (h.double() > 0)))})
    gbuf = _grad_buf(g)
    post = gbuf.clone()
    Wg = torch.zeros(SHAPES[name + ".w"], dtype=torch.float64, requires_grad=True)
    if op == "enc.conv2 wgrad":
        h = _act(g, B, 32, 32, 32)
        d = bf(torch.randn(B, 16, 16, 32, generator=g))
        (O._conv(h.double(), Wg, None, s, pd) * d.double()).sum().backward()
        pre = {"enc.conv1.out": R.s2d_blocks(h), "enc.conv2.dout": d, "grad": gbuf}
    elif op == "dec.conv3t wgrad":
        h = _act(g, B, 8, 8, 64)
        d = bf(torch.randn(B, 16, 16, 32, generator=g))
        (O._convT(h.double(), Wg, None, s, pd) * d.double()).sum().backward()
        pre = {"dec.conv3t.dout": R.s2d_blocks(d), "dec.conv2t.out": h, "grad": gbuf}
    elif op == "dec.conv4t bgrad":
        d = bf(torch.randn(B, 32, 32, 32, generator=g))
        _flat_view(post)[name + ".b"].add_(d.double().sum((0, 1, 2)).float())
        return {"dec.conv4t.dout": R.s2d_blocks(d), "grad": gbuf}, {"grad": post}
    else:
        raise KeyError(op)
    _flat_view(post)[name + ".w"].add_(Wg.grad.float())
    return pre, {"grad": post}


CONV_OPS = ["enc.conv2 fwd", "enc.conv4 fwd", "dec.conv3t fwd", "enc.conv3 dgrad", "dec.conv4t dgrad", "enc.conv2 wgrad",
            "dec.conv3t wgrad", "dec.conv4t bgrad"]


@pytest.mark.parametrize("op", CONV_OPS)
def test_conv_reference_equals_oracle(op):
    g = torch.Generator().manual_seed(1)
    ctx, p = _ctx()
    pre, post = _conv_case(op, g, ctx, p)
    worst, res = _ok(op, pre, post, ctx)
    assert worst <= 1.0, res


def _chain_fwd_case(supervised, K=5):
    """a chain forward snapshot computed with the oracle's network, classifier, prior and KL."""
    g = torch.Generator().manual_seed(4)
    c = torch.rand(18, 18, generator=g)
    x, y, noise = O.make_inputs(B, k=K)
    ctx, p = _ctx(c=c, supervised=supervised, K=K, y=y, eps=noise["eps"], eps_k=noise["eps_k"], U_y=noise["U_y"])
    P, W = ctx.P, ctx.W
    h5 = _act(g, B, 1, 1, 256)
    hf = h5.double().reshape(B, 256)
    pre96 = torch.zeros(B, 96, dtype=torch.float64)
    pre96[:, :45] = hf @ W["enc.locs.w"] + P["enc.locs.b"]
    pre96[:, 48:93] = hf @ W["enc.std.w"] + P["enc.std.b"]
    pre96 = pre96.float()
    loc = torch.relu(pre96[:, :45].double()).float()
    scale = O.clipped_softplus(pre96[:, 48:93].double()).float()
    z = (loc.double() + scale.double() * noise["eps"].double()).float()
    L, S, Z = loc.double(), scale.double(), z.double()
    logits = O.classifier(P, Z[:, O.Z_STYLE:].unsqueeze(-1).repeat(1, 1, 18), c.double())
    yy = y if supervised else O.bernoulli_sample(logits, noise["U_y"].double()).long()
    kl, _, _ = O._prior_and_kl(P, yy, c.double(), L, S)
    lq = O.bernoulli_logits_log_prob(logits, yy).sum(-1)
    terms = torch.zeros(6, B, dtype=torch.float64)
    terms[0], terms[1], terms[4] = kl, lq, 18 * math.log(0.5)
    if supervised:
        rows = []
        for k in range(K):
            zk = L + S * noise["eps_k"][k].double()
            lk = O.classifier(P, zk[:, O.Z_STYLE:].unsqueeze(-1).repeat(1, 1, 18), c.double())
            rows.append(O.bernoulli_logits_log_prob(lk, yy).sum(-1))
        terms[2] = torch.logsumexp(torch.stack(rows), 0) - math.log(K)
        terms[3] = torch.exp(lq - terms[2])
    else:
        terms[3] = 1.0
    terms[5] = -terms[3] / B
    z16 = torch.zeros(B, 64, dtype=torch.bfloat16)
    z16[:, :45] = bf(z)
    g0 = torch.zeros(B, 64, dtype=torch.bfloat16)
    g0[:, :45] = bf(torch.relu(z16[:, :45].double() @ W["dec.fc1.w"] + P["dec.fc1.b"]))
    g1 = bf(torch.relu(O._convT(g0[:, :45].double().reshape(B, 1, 1, 45), W["dec.conv1t.w"], P["dec.conv1t.b"], 1, 0)))
    post = {"pre96": pre96, "z16": z16, "dec.fc1.out": g0, "dec.conv1t.out": g1, "lb:loc": loc, "lb:scale": scale,
            "lb:z": z, "lb:terms": terms.float(), "lb:logits": logits.float(), "lb:y_i32": yy.int()}
    return {"enc.conv5.out": h5}, post, ctx


@pytest.mark.parametrize("supervised", [True, False])
def test_chain_fwd_reference_equals_oracle(supervised):
    pre, post, ctx = _chain_fwd_case(supervised)
    worst, res = _ok("chain fwd", pre, post, ctx)
    assert worst <= 1.0, res
    labels = {label for label, _ in res}
    assert {"kl", "log_qy_zc", "w", "coef", "log_py", "logits", "z", "dec.conv1t.out"} <= labels
    assert ("log_qy_x" in labels) == supervised


def test_recon_reference_equals_oracle():
    g = torch.Generator().manual_seed(5)
    x, _, _ = O.make_inputs(B, k=1)
    ctx, p = _ctx(x=x)
    g4 = _act(g, B, 32, 32, 32)
    terms = torch.randn(6, B, generator=g)
    logit = O._convT(g4.double(), ctx.W["dec.conv5t.w"], ctx.P["dec.conv5t.b"], 2, 1)
    xh = torch.sigmoid(logit).float()
    e = x.double() - xh.double()
    d = terms[5].double().view(B, 1, 1, 1) * torch.sign(e) * xh.double() * (1 - xh.double())
    gbuf = _grad_buf(g)
    post_g = gbuf.clone()
    _flat_view(post_g)["dec.conv5t.b"].add_(d.sum((0, 1, 2)).float())
    pre = {"dec.conv4t.out": g4, "lb:terms": terms, "grad": gbuf}
    post = {"xhat3": xh, "lb:log_pxz": O.img_log_likelihood(xh.double(), x.double()).float(),
            "D2": R.x2_blocks(bf(d)), "grad": post_g}
    worst, res = _ok("dec.conv5t fwd+recon", pre, post, ctx)
    assert worst <= 1.0, res
    # conv5t's dgrad / wgrad from those blocks
    D2 = post["D2"]
    Wg = torch.zeros(4, 4, 3, 32, dtype=torch.float64, requires_grad=True)
    (O._convT(g4.double(), Wg, None, 2, 1) * bf(d).double()).sum().backward()
    post_w = gbuf.clone()
    _flat_view(post_w)["dec.conv5t.w"].add_(Wg.grad.float())
    worst, res = _ok("dec.conv5t wgrad", {"D2": D2, "dec.conv4t.out": g4, "grad": gbuf}, {"grad": post_w}, ctx)
    assert worst <= 1.0, res
    dg4 = O._conv(bf(d).double(), ctx.W["dec.conv5t.w"], None, 2, 1) * (g4.double() > 0)
    worst, res = _ok("dec.conv5t dgrad", {"D2": D2, "dec.conv4t.out": g4},
                     {"dec.conv4t.dout": R.s2d_blocks(bf(dg4))}, ctx)
    assert worst <= 1.0, res


# ---- every reference runs on a snapshot of the right shapes -----------------------------------------------------------
def _buffer(key, rows, g):
    shapes = {"X2": (rows * 1089 * 24,), "D2": (rows, 33, 33, 16), "pre96": (rows, 96), "dpre16": (rows, 96),
              "z16": (rows, 64), "dz64": (rows, 64), "dec.fc1.out": (rows, 64), "dec.fc1.dout": (rows, 64),
              "xhat3": (rows, 64, 64, 3), "lb:loc": (rows, 45), "lb:scale": (rows, 45), "lb:z": (rows, 45),
              "lb:terms": (6, rows), "lb:logits": (rows, 18), "lb:y_i32": (rows, 18), "lb:log_pxz": (rows,),
              "ll:log_pxz": (rows,), "grad": (sum(math.prod(s) for s in SHAPES.values()),)}
    maps = {"enc.conv1": (32, 32, 32), "enc.conv2": (16, 16, 32), "enc.conv3": (8, 8, 64), "enc.conv4": (4, 4, 128),
            "enc.conv5": (1, 1, 256), "dec.conv1t": (4, 4, 128), "dec.conv2t": (8, 8, 64), "dec.conv3t": (16, 16, 32),
            "dec.conv4t": (32, 32, 32)}
    if key in shapes:
        shape = shapes[key]
    else:
        H, W, C = maps[key.rsplit(".", 1)[0]]
        shape = (rows, H // 2 + 1, W // 2 + 1, 4 * C) if key in R.S2D else (rows, H, W, C)
    t = torch.rand(*shape, generator=g)
    if key == "lb:y_i32":
        return (t < 0.5).int()
    if key in ("grad", "xhat3") or key.startswith("lb:") or key.startswith("ll:") or key in ("pre96", "dz64"):
        return t
    return bf(t)


@pytest.mark.parametrize("op", sorted(R.OPS))
def test_every_reference_runs(op):
    g = torch.Generator().manual_seed(2)
    rows = 2 if op != "dec.conv5t fwd ll" else 4
    x, y, noise = O.make_inputs(2, k=3)
    ctx, _ = _ctx(x=x, x_raw=(x * 255).to(torch.uint8), c=torch.rand(18, 18, generator=g), supervised=True, K=3, y=y,
                  eps=noise["eps"], eps_k=noise["eps_k"], U_y=noise["U_y"])
    reads, writes, _ = R.OPS[op]
    pre = {k: _buffer(k, rows, g) for k in reads}
    post = {k: _buffer(k, rows, g) for k in writes}
    res = R.check_launch(op, pre, post, ctx, rows)
    assert res and all(r >= 0 for _, r in res)


# ---- the check catches subtly wrong results ---------------------------------------------------------------------------
def test_one_element_four_ulps_off_fails():
    g = torch.Generator().manual_seed(1)
    ctx, p = _ctx()
    pre, post = _conv_case("enc.conv4 fwd", g, ctx, p)
    out = post["enc.conv4.out"].clone()
    i = int(out.float().abs().argmax())
    out.view(-1).view(torch.int16)[i] += 4
    worst, _ = _ok("enc.conv4 fwd", pre, {"enc.conv4.out": out}, ctx)
    assert worst > 1.0


def test_missing_weight_gradient_split_fails():
    """one of 74 K-splits of conv2's weight gradient lost: the other 73 are exact"""
    g = torch.Generator().manual_seed(1)
    ctx, p = _ctx()
    pre, post = _conv_case("enc.conv2 wgrad", g, ctx, p)
    h = R.s2d_pixels(pre["enc.conv1.out"].double())
    d = pre["enc.conv2.dout"].double().clone()
    rows = d.reshape(-1, 32)
    n = rows.shape[0]
    rows[n - (n + 73) // 74:] = 0                      # the last split's output pixels
    lost = R.wg(h, d, "enc.conv2")
    post_bad = pre["grad"].clone()
    _flat_view(post_bad)["enc.conv2.w"].add_(lost.float())
    worst, _ = _ok("enc.conv2 wgrad", pre, {"grad": post_bad}, ctx)
    assert worst > 1.0


def test_swapped_s2d_slots_fail():
    g = torch.Generator().manual_seed(1)
    ctx, p = _ctx()
    pre, post = _conv_case("enc.conv2 fwd", g, ctx, p)
    out = post["enc.conv2.out"].clone()
    C = 32
    a, b_ = out[0, 4, 4, 0:C].clone(), out[0, 4, 4, C:2 * C].clone()
    out[0, 4, 4, 0:C], out[0, 4, 4, C:2 * C] = b_, a
    worst, _ = _ok("enc.conv2 fwd", pre, {"enc.conv2.out": out}, ctx)
    assert worst > 1.0
    # a value in a border slot (the next layer's zero padding) fails as well
    out = post["enc.conv2.out"].clone()
    out[1, 0, 3, 0] = 1.0
    worst, res = _ok("enc.conv2 fwd", pre, {"enc.conv2.out": out}, ctx)
    assert worst > 1.0 and dict(res)["enc.conv2.out border slots"] > 1.0


def test_nan_in_a_pad_column_fails():
    g = torch.Generator().manual_seed(3)
    ctx, p = _ctx()
    z16 = torch.zeros(B, 64, dtype=torch.bfloat16)
    z16[:, :45] = bf(torch.randn(B, 45, generator=g))
    want = torch.relu(z16[:, :45].double() @ ctx.W["dec.fc1.w"] + ctx.P["dec.fc1.b"])
    g0 = torch.zeros(B, 64, dtype=torch.bfloat16)
    g0[:, :45] = bf(want)
    worst, _ = _ok("dec.fc1 fwd", {"z16": z16}, {"dec.fc1.out": g0}, ctx)
    assert worst <= 1.0
    g0[1, 50] = float("nan")
    worst, res = _ok("dec.fc1 fwd", {"z16": z16}, {"dec.fc1.out": g0}, ctx)
    assert worst == math.inf and dict(res)["dec.fc1.out pad columns finite"] == math.inf


def test_exact_result_passes_and_bound_is_tight():
    want = torch.tensor([1.0, -3.0, 0.0, 1e-3], dtype=torch.float64)
    scale = want.abs()
    got = bf(want).double()
    assert R.worst_ratio(got, want, scale, "bf16") <= 1.0
    assert R.worst_ratio(want, want, scale, "f32") == 0.0
    # half a bf16 ulp of 1.0 more than the rounding allows
    assert R.worst_ratio(want + torch.tensor([2.0 ** -7, 0, 0, 0]), want, scale, "bf16") > 1.0
    # a zero that should be exact
    assert R.worst_ratio(torch.tensor([0.0, 1e-30]), torch.zeros(2), torch.zeros(2), "f32") == math.inf
