"""fp64 references of the single launches of the bf16 step, one per op kind, and the per-element check they are held to.

Every reference takes one launch's snapshot - the engine buffers it reads before the launch (`pre`) and the buffers it
writes after it (`post`) - and the master weights (fp32 master rounded to bf16 as the pack kernels round, in fp64). It
recomputes the launch's outputs in fp64 from the launch's own inputs, never from an earlier reference, and returns
(label, got, want, scale, kind) tuples:

  kind "bf16"   bf16 output:                 |got - want| <= 2^-8 |want| + 1e-5 scale  (rounding of the output + fp32 sums)
  kind "f32"    fp32 output / accumulation:  |got - want| <= 1e-5 scale                (after subtracting the pre-launch value)
  kind "exact"  layouts, integer outputs:    got == want

`scale` is the same operation applied to the absolute values of its operands (conv(|x|, |W|), |A|^T |B|, ...), element by
element: a single wrong element fails however small it is against the tensor's maximum.  Every reference is built from
the master weights, not from the packed operands, so a packing error shows in the launch that reads the packed operand.

Layout helpers (s2d blocks of the stride-2 layers' L tensors, x2 blocks of the 3-channel images) live here too."""
import math

import torch
import torch.nn.functional as F

import gccvae_oracle as O

BF16_REL = 2.0 ** -8
F32_REL = 1e-5
LN2 = math.log(2.0)

# stride and padding of the k4 layers (weights [4,4,CL,CS]: CL = the large-map side, CS = the small-map side)
GEOM = {"enc.conv1": (2, 1), "enc.conv2": (2, 1), "enc.conv3": (2, 1), "enc.conv4": (2, 1), "enc.conv5": (1, 0),
        "dec.conv1t": (1, 0), "dec.conv2t": (2, 1), "dec.conv3t": (2, 1), "dec.conv4t": (2, 1), "dec.conv5t": (2, 1)}
# tensors the bf16 engine stores in s2d block form
S2D = ("enc.conv1.out", "enc.conv2.out", "enc.conv3.out", "dec.conv4t.dout", "dec.conv3t.dout", "dec.conv2t.dout")
ENC = ["enc.conv1", "enc.conv2", "enc.conv3", "enc.conv4", "enc.conv5"]
DEC = ["dec.conv1t", "dec.conv2t", "dec.conv3t", "dec.conv4t", "dec.conv5t"]


# ---- layouts ---------------------------------------------------------------------------------------------------------
def s2d_blocks(t):
    """[B,H,W,C] -> [B,H/2+1,W/2+1,4C]: block (i,j) slot dy*2+dx = pixel (2i-1+dy, 2j-1+dx), zero outside."""
    B, H, W, Cc = t.shape
    pad = torch.zeros(B, H + 2, W + 2, Cc, dtype=t.dtype, device=t.device)
    pad[:, 1:H + 1, 1:W + 1] = t
    return pad.view(B, H // 2 + 1, 2, W // 2 + 1, 2, Cc).permute(0, 1, 3, 2, 4, 5).reshape(B, H // 2 + 1, W // 2 + 1, 4 * Cc)


def s2d_pixels(blk):
    """inverse of s2d_blocks: [B,Hb,Wb,4C] -> [B,2Hb-2,2Wb-2,C] (the border slots are dropped)."""
    B, Hb, Wb, C4 = blk.shape
    Cc = C4 // 4
    pad = blk.reshape(B, Hb, Wb, 2, 2, Cc).permute(0, 1, 3, 2, 4, 5).reshape(B, 2 * Hb, 2 * Wb, Cc)
    return pad[:, 1:2 * Hb - 1, 1:2 * Wb - 1]


def x2_blocks(img, ones=False):
    """[B,64,64,3] -> [B,33,33,16] with X2[n,i,j,(dy,dx,c4)] = img[n,2i-1+dy,2j-1+dx,c] (zero outside / pad).
    ones=True: as gccvae_prep_x2_bf16 writes the blocks - element 15 (pad channel of the last pixel slot) is 1.0, the
    constant row that turns conv1's weight gradient into its bias gradient as well."""
    B = img.shape[0]
    pad = torch.zeros(B, 66, 66, 4, dtype=img.dtype, device=img.device)
    pad[:, 1:65, 1:65, :3] = img
    blk = pad.view(B, 33, 2, 33, 2, 4).permute(0, 1, 3, 2, 4, 5).reshape(B, 33, 33, 16)
    if ones:
        blk = blk.clone()
        blk[..., 15] = 1
    return blk


def x2_pixels(blk):
    """inverse of x2_blocks: [B,33,33,16] -> [B,64,64,3]."""
    B = blk.shape[0]
    return blk.reshape(B, 33, 33, 2, 2, 4).permute(0, 1, 3, 2, 4, 5).reshape(B, 66, 66, 4)[:, 1:65, 1:65, :3]


def _raw_byte_blocks(xi):
    """[B,64,64,3] uint8 -> [B,33,33,16] uint8: block (i, j) = pixels (2i-1+dy, 2j-1+dx) x 3 channels, 4 zero bytes."""
    B = xi.shape[0]
    pad = torch.zeros(B, 66, 66, 3, dtype=torch.uint8, device=xi.device)
    pad[:, 1:65, 1:65] = xi
    out = torch.zeros(B, 33, 33, 16, dtype=torch.uint8, device=xi.device)
    for dy in range(2):
        for dx in range(2):
            q = dy * 2 + dx
            out[..., 3 * q:3 * q + 3] = pad[:, dy:dy + 65:2, dx:dx + 65:2][:, :33, :33]
    return out


# ---- the check -------------------------------------------------------------------------------------------------------
def bound(want, scale, kind):
    if kind == "bf16":
        return BF16_REL * want.abs() + F32_REL * scale
    if kind == "f32":
        return F32_REL * scale
    raise KeyError(kind)


def worst_ratio(got, want, scale, kind):
    """max over elements of |got - want| / bound (0 where both agree exactly, inf for a NaN or an excess over a zero
    bound); kind "exact": 0 if equal everywhere, else inf."""
    got, want = got.double(), want.double()
    assert got.shape == want.shape, (got.shape, want.shape)
    if got.numel() == 0:
        return 0.0
    if kind == "exact":
        return 0.0 if bool((got == want).all()) else math.inf
    d = (got - want).abs()
    if not bool(torch.isfinite(d).all()):
        return math.inf
    b = bound(want, scale.double(), kind)
    r = torch.where(d == 0, torch.zeros_like(d), d / b)      # d > 0 over b == 0 -> inf
    return float(r.max())


# ---- layer maths (NHWC fp64; W [4,4,CL,CS]) ---------------------------------------------------------------------------
def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def ls(Lt, W, name):
    """L -> S: the convolution (encoder forward, decoder dgrad)."""
    s, p = GEOM[name]
    return _nhwc(F.conv2d(_nchw(Lt), W.permute(3, 2, 0, 1), stride=s, padding=p))


def sl(St, W, name):
    """S -> L: the transposed convolution (decoder forward, encoder dgrad)."""
    s, p = GEOM[name]
    return _nhwc(F.conv_transpose2d(_nchw(St), W.permute(3, 2, 0, 1), stride=s, padding=p))


def wg(Lt, St, name):
    """weight gradient [4,4,CL,CS] of the relation between an L tensor and an S tensor: sum over images and positions."""
    s, p = GEOM[name]
    CL, CS = Lt.shape[-1], St.shape[-1]
    w = torch.nn.grad.conv2d_weight(_nchw(Lt), (CS, CL, 4, 4), _nchw(St), stride=s, padding=p)
    return w.permute(2, 3, 1, 0)


def _with_scale(fn, *args):
    """(fn(args), fn(|args|)) for a function bilinear in its tensor arguments."""
    return fn(*args), fn(*[a.abs() if torch.is_tensor(a) else a for a in args])


# ---- snapshot access ---------------------------------------------------------------------------------------------------
def pixels(key, t):
    """an engine buffer as NHWC (or [rows, cols]) fp64: s2d blocks and x2 blocks unpacked."""
    t = t.double()
    if key in S2D:
        return s2d_pixels(t)
    if key in ("X2", "D2"):
        return x2_pixels(t)
    return t


def invariants(key, t):
    """(label, got, want, scale, kind) checks of what later launches rely on in a buffer that was just written: the
    border slots of block tensors stay zero, pad columns stay finite (or zero where the writer zeroes them)."""
    out = []
    if key in S2D:
        out.append((key + " border slots", t.float(), s2d_blocks(s2d_pixels(t.float())), None, "exact"))
    elif key == "D2":
        out.append((key + " border / pad lanes", t.float(), x2_blocks(x2_pixels(t.float())), None, "exact"))
    elif key in ("pre96", "dpre16"):
        pad = torch.cat([t[:, 45:48], t[:, 93:96]], 1).float()
        out.append((key + " pad columns finite", torch.isfinite(pad), torch.ones_like(pad, dtype=torch.bool), None, "exact"))
    elif key in ("z16", "dec.fc1.out", "dec.fc1.dout"):
        pad = t[:, 45:64].float()
        out.append((key + " pad columns finite", torch.isfinite(pad), torch.ones_like(pad, dtype=torch.bool), None, "exact"))
    return out


def zero_pads(key, t):
    """pad columns a writer sets to exactly zero."""
    pad = (torch.cat([t[:, 45:48], t[:, 93:96]], 1) if key in ("pre96", "dpre16") else t[:, 45:64]).float()
    return [(key + " pad columns zero", pad, torch.zeros_like(pad), None, "exact")]


# ---- the references, by op ---------------------------------------------------------------------------------------------
class Ctx:
    """what a reference needs besides the snapshot: W (bf16-rounded masters, fp64), P (fp32 masters in fp64: biases and
    the latent-stage parameters, which the kernels read unrounded), the images x (fp32 in [0,1], device), and for the
    latent stage the gate sample c, the explicit noise, the labels, K and `supervised`; `grads(flat)` maps a flat gradient
    buffer to {name: tensor}."""

    def __init__(self, W, P, grads, x=None, **kw):
        self.W, self.P, self.grads, self.x = W, P, grads, x
        self.__dict__.update(kw)


def _dgrad_mask(v):
    return (v > 0).double()


def _grad_delta(ctx, pre, post, name):
    return ctx.grads(post["grad"])[name].double() - ctx.grads(pre["grad"])[name].double()


def ref_prep_x2(pre, post, ctx, rows):
    x = ctx.x_raw
    B = x.shape[0]
    xc = x.cpu()       # the host's IEEE division: the kernel's u / 255 is correctly rounded
    xf = (xc.float() / 255.0 if x.dtype == torch.uint8 else xc.float()).to(x.device)
    X2 = post["X2"]
    got = X2[:B * 1089 * 16].view(B, 33, 33, 16)
    out = [("x2 blocks", got.view(torch.int16), x2_blocks(xf, ones=True).to(torch.bfloat16).view(torch.int16), None, "exact")]
    if x.dtype == torch.uint8:
        raw = X2.view(torch.uint8)[B * 1089 * 32:B * 1089 * 48].view(B, 33, 33, 16)
        out.append(("raw-byte blocks", raw, _raw_byte_blocks(x), None, "exact"))
    return out


def _fwd_conv(pre, post, ctx, name, src, dst, transposed, relu=True):
    W, b = ctx.W[name + ".w"], ctx.P[name + ".b"]
    h = pixels(src, pre[src])
    want, scale = _with_scale(sl if transposed else ls, h, W, name)
    want, scale = want + b, scale + b.abs()
    if relu:
        want = want.clamp_min(0)
    return [(dst, pixels(dst, post[dst]), want, scale, "bf16")] + invariants(dst, post[dst])


def _dgrad(pre, post, ctx, name, dout, mask, dst, transposed):
    """gradient of the layer's input from the gradient of its (pre-activation) output, times the ReLU mask of the input"""
    W = ctx.W[name + ".w"]
    g = pixels(dout, pre[dout])
    want, scale = _with_scale(ls if transposed else sl, g, W, name)
    m = _dgrad_mask(pixels(mask, pre[mask]))
    return [(dst, pixels(dst, post[dst]), want * m, scale * m, "bf16")] + invariants(dst, post[dst])


def _wgrad(pre, post, ctx, name, Lkey, Skey):
    Lt, St = pixels(Lkey, pre[Lkey]), pixels(Skey, pre[Skey])
    want, scale = _with_scale(wg, Lt, St, name)
    return [(name + ".w grad", _grad_delta(ctx, pre, post, name + ".w"), want, scale, "f32")]


def _bgrad(pre, post, ctx, name, key, n=None):
    g = pixels(key, pre[key])
    g = g.reshape(-1, g.shape[-1])[:, :n]
    return [(name + ".b grad", _grad_delta(ctx, pre, post, name + ".b"), g.sum(0), g.abs().sum(0), "f32")]


def _fc(A, Wm):
    return _with_scale(lambda a, w: a @ w, A, Wm)


def ref_heads_fwd(pre, post, ctx, h5, out="pre96"):
    P, W = ctx.P, ctx.W
    got = post[out].double()
    checks = []
    for c0, nm in ((0, "enc.locs"), (48, "enc.std")):
        want, scale = _fc(h5, W[nm + ".w"])
        checks.append((out + "[" + nm + "]", got[:, c0:c0 + 45], want + P[nm + ".b"], scale + P[nm + ".b"].abs(), "f32"))
    return checks + invariants(out, post[out])


def _fc1_fwd(z16, ctx):
    want, scale = _fc(z16[:, :45], ctx.W["dec.fc1.w"])
    b = ctx.P["dec.fc1.b"]
    return (want + b).clamp_min(0), scale + b.abs()


def _conv1t_fwd(g0, ctx):
    want, scale = _with_scale(sl, g0[:, :45].reshape(-1, 1, 1, 45), ctx.W["dec.conv1t.w"], "dec.conv1t")
    b = ctx.P["dec.conv1t.b"]
    return (want + b).clamp_min(0).reshape(-1, 2048), (scale + b.abs()).reshape(-1, 2048)


def _latent_terms(pre96, loc, scale, z, logits, y_got, ctx):
    """the latent stage of the chain forward from the kernel's own pre-activations / posterior / logits."""
    P, B = ctx.P, pre96.shape[0]
    out = []
    pl, ps = pre96[:, :45], pre96[:, 48:93]
    want_loc = pl.clamp_min(0)
    want_sc = torch.clamp(F.softplus(ps), 1e-3, 1e3)
    out.append(("loc", loc, want_loc, want_loc.abs(), "f32"))
    # clipped softplus: d softplus / d pre < 1, the fp32 result rounds relative to itself
    out.append(("scale", scale, want_sc, want_sc.abs() + ps.abs() * (want_sc > 1e-3), "f32"))
    eps = ctx.eps[:B].double()
    out.append(("z", z, loc + scale * eps, loc.abs() + (scale * eps).abs(), "f32"))
    c = ctx.c.double()
    zc = z[:, O.Z_STYLE:]
    want_logits = O.classifier(P, zc.unsqueeze(-1).repeat(1, 1, O.Y_DIM), c)
    sc_logits = O.classifier({"cls.w": P["cls.w"].abs(), "cls.b": P["cls.b"].abs()},
                             zc.abs().unsqueeze(-1).repeat(1, 1, O.Y_DIM), c.abs())
    out.append(("logits", logits, want_logits, sc_logits, "f32"))
    if ctx.supervised:
        y = ctx.y[:B].to(y_got.device)
        out.append(("y", y_got.long(), y.long(), None, "exact"))
    else:
        u = ctx.U_y[:B].double()
        pr = torch.sigmoid(logits)
        want_y = (u < pr).long()
        # a label may differ only where U_y is within the fp32 rounding of sigmoid(logit)
        close = (u - pr).abs() <= 1e-6
        out.append(("y (sampled)", torch.where(close, want_y, y_got.long()), want_y, None, "exact"))
        y = y_got.long()
    return out, y


def _terms(terms, loc, scale, logits, y, ctx):
    """the six per-image terms: kl, log q(y|z_c), log q(y|x), w, log p(y), the likelihood's coefficient."""
    P, B = ctx.P, loc.shape[0]
    out = []
    c = ctx.c.double()
    yt = y.unsqueeze(-1).repeat(1, 1, O.Z_CLASSIFY).double()
    prior_l, prior_s = O.cond_prior(P, yt, c)
    mp = torch.cat([torch.zeros(B, O.Z_STYLE, dtype=loc.dtype, device=loc.device), prior_l], 1)
    sp = torch.cat([torch.ones(B, O.Z_STYLE, dtype=loc.dtype, device=loc.device), prior_s], 1)
    dls = torch.log(scale) - torch.log(sp)
    parts = (0.5 * ((loc - mp) / sp) ** 2, 0.5 * torch.expm1(2.0 * dls), -dls)
    kl = sum(parts).sum(-1)
    kl_scale = (sum(p_.abs() for p_ in parts) + (loc.abs() + mp.abs()) / sp).sum(-1)
    out.append(("kl", terms[0], kl, kl_scale, "f32"))
    lp = O.bernoulli_logits_log_prob(logits, y)
    lq, lq_scale = lp.sum(-1), (lp.abs() + logits.abs()).sum(-1)
    out.append(("log_qy_zc", terms[1], lq, lq_scale, "f32"))
    out.append(("log_py", terms[4], torch.full_like(lq, O.Y_DIM * math.log(0.5)), torch.full_like(lq, O.Y_DIM * LN2), "f32"))
    if ctx.supervised:
        K = ctx.K
        ek = ctx.eps_k[:, :B, O.Z_STYLE:].double()                        # [K,B,18]
        zk = loc[:, O.Z_STYLE:] + scale[:, O.Z_STYLE:] * ek
        zk_scale = loc[:, O.Z_STYLE:].abs() + (scale[:, O.Z_STYLE:] * ek).abs()
        lk = torch.einsum("kbi,ij->kbj", zk, c * P["cls.w"]) + P["cls.b"]
        lk_scale = torch.einsum("kbi,ij->kbj", zk_scale, (c * P["cls.w"]).abs()) + P["cls.b"].abs()
        lpk = O.bernoulli_logits_log_prob(lk, y.unsqueeze(0).expand_as(lk))
        s = lpk.sum(-1)                                                   # [K,B]
        lqx = torch.logsumexp(s, 0) - math.log(K)
        lqx_scale = (lpk.abs() + lk_scale).sum(-1).max(0).values + math.log(K)
        out.append(("log_qy_x", terms[2], lqx, lqx_scale, "f32"))
        w = torch.exp(lq - lqx)
        w_scale = w * (lq_scale + lqx_scale)
    else:
        w, w_scale = torch.ones_like(lq), torch.ones_like(lq)
    out.append(("w", terms[3], w, w_scale, "f32"))
    out.append(("coef", terms[5], -w / B, w_scale / B, "f32"))
    return out


def ref_chain_fwd(pre, post, ctx, rows):
    h5 = pre["enc.conv5.out"].double().reshape(rows, 256)
    out = ref_heads_fwd(pre, post, ctx, h5)
    pre96 = post["pre96"].double()
    lat, y = _latent_terms(pre96, post["lb:loc"].double(), post["lb:scale"].double(), post["lb:z"].double(),
                           post["lb:logits"].double(), post["lb:y_i32"], ctx)
    out += lat
    out += _terms(post["lb:terms"].double(), post["lb:loc"].double(), post["lb:scale"].double(),
                  post["lb:logits"].double(), y, ctx)
    z16 = post["z16"]
    out.append(("z16 == bf16(z)", z16[:, :45].view(torch.int16), post["lb:z"].to(torch.bfloat16).view(torch.int16), None,
                "exact"))
    out += zero_pads("z16", z16)
    want, scale = _fc1_fwd(z16.double(), ctx)
    out.append(("dec.fc1.out", post["dec.fc1.out"][:, :45].double(), want, scale, "bf16"))
    out += zero_pads("dec.fc1.out", post["dec.fc1.out"])
    want, scale = _conv1t_fwd(post["dec.fc1.out"].double(), ctx)
    out.append(("dec.conv1t.out", post["dec.conv1t.out"].double().reshape(rows, 2048), want, scale, "bf16"))
    return out


def ref_fc1_fwd(pre, post, ctx, rows):
    want, scale = _fc1_fwd(pre["z16"].double(), ctx)
    got = post["dec.fc1.out"]
    return [("dec.fc1.out", got[:, :45].double(), want, scale, "bf16")] + invariants("dec.fc1.out", got)


def ref_conv1t_fwd(pre, post, ctx, rows):
    want, scale = _conv1t_fwd(pre["dec.fc1.out"].double(), ctx)
    return [("dec.conv1t.out", post["dec.conv1t.out"].double().reshape(rows, 2048), want, scale, "bf16")]


def _recon_logits(g4, ctx):
    W, b = ctx.W["dec.conv5t.w"], ctx.P["dec.conv5t.b"]
    want, scale = _with_scale(sl, g4, W, "dec.conv5t")
    return want + b, scale + b.abs()


def ref_conv5t_recon(pre, post, ctx, rows):
    g4 = pre["dec.conv4t.out"].double()
    logit, lscale = _recon_logits(g4, ctx)
    xh_want = torch.sigmoid(logit)
    xh = post["xhat3"].double()
    x = ctx.x[:rows].double()
    out = [("xhat", xh, xh_want, 0.25 * lscale + xh_want, "f32")]
    # likelihood and its gradient from the kernel's own reconstruction: sign(x - xhat) is discontinuous
    e = x - xh
    ll = -e.abs().sum((1, 2, 3)) - 12288 * LN2
    out.append(("log_pxz", post["lb:log_pxz"].double(), ll, e.abs().sum((1, 2, 3)) + 12288 * LN2, "f32"))
    coef = pre["lb:terms"][5].double().view(-1, 1, 1, 1)
    d = coef * torch.sign(e) * xh * (1 - xh)
    out.append(("D2", pixels("D2", post["D2"]), d, d.abs(), "bf16"))
    out += invariants("D2", post["D2"])
    out.append(("dec.conv5t.b grad", _grad_delta(ctx, pre, post, "dec.conv5t.b"), d.sum((0, 1, 2)),
                d.abs().sum((0, 1, 2)), "f32"))
    return out


def ref_conv5t_ll(pre, post, ctx, rows):
    g4 = pre["dec.conv4t.out"].double()
    logit, lscale = _recon_logits(g4, ctx)
    xh = torch.sigmoid(logit)
    kc = rows // ctx.x.shape[0]
    x = ctx.x.double().repeat_interleave(kc, 0)
    e = (x - xh).abs()
    want = -e.sum((1, 2, 3)) - 12288 * LN2
    scale = (e + 0.25 * lscale).sum((1, 2, 3)) + 12288 * LN2
    return [("log_pxz", post["ll:log_pxz"].double(), want, scale, "f32")]


def ref_conv1t_wgrad(pre, post, ctx, rows):
    dg1 = pre["dec.conv1t.dout"].double().reshape(rows, 2048)
    g0 = pre["dec.fc1.out"].double()[:, :45]
    want, scale = _fc(dg1.t(), g0)
    return [("dec.conv1t.w grad", _grad_delta(ctx, pre, post, "dec.conv1t.w").reshape(2048, 45), want, scale, "f32")]


def ref_conv1t_dgrad(pre, post, ctx, rows):
    dg1 = pre["dec.conv1t.dout"].double().reshape(rows, 2048)
    want, scale = _fc(dg1, ctx.W["dec.conv1t.w"].reshape(2048, 45))
    m = _dgrad_mask(pre["dec.fc1.out"].double()[:, :45])
    got = post["dec.fc1.dout"]
    return [("dec.fc1.dout", got[:, :45].double(), want * m, scale * m, "bf16")] + invariants("dec.fc1.dout", got)


def ref_fc1_wgrad(pre, post, ctx, rows):
    want, scale = _fc(pre["z16"].double()[:, :45].t(), pre["dec.fc1.dout"].double()[:, :45])
    return [("dec.fc1.w grad", _grad_delta(ctx, pre, post, "dec.fc1.w"), want, scale, "f32")]


def ref_fc1_dgrad(pre, post, ctx, rows):
    want, scale = _fc(pre["dec.fc1.dout"].double()[:, :45], ctx.W["dec.fc1.w"].t())
    return [("dz", post["dz64"].double()[:, :45], want, scale, "f32")]


def ref_heads_wgrad(pre, post, ctx, rows):
    h5 = pre["enc.conv5.out"].double().reshape(rows, 256)
    dp = pre["dpre16"].double()
    out = []
    for c0, nm in ((0, "enc.locs"), (48, "enc.std")):
        want, scale = _fc(h5.t(), dp[:, c0:c0 + 45])
        out.append((nm + ".w grad", _grad_delta(ctx, pre, post, nm + ".w"), want, scale, "f32"))
    return out


def _heads_dgrad(dp, h5, ctx):
    W = ctx.W
    want = dp[:, :45] @ W["enc.locs.w"].t() + dp[:, 48:93] @ W["enc.std.w"].t()
    scale = dp[:, :45].abs() @ W["enc.locs.w"].abs().t() + dp[:, 48:93].abs() @ W["enc.std.w"].abs().t()
    m = _dgrad_mask(h5)
    return want * m, scale * m


def ref_heads_dgrad(pre, post, ctx, rows):
    want, scale = _heads_dgrad(pre["dpre16"].double(), pre["enc.conv5.out"].double().reshape(rows, 256), ctx)
    return [("enc.conv5.dout", post["enc.conv5.dout"].double().reshape(rows, 256), want, scale, "bf16")]


def ref_chain_bwd(pre, post, ctx, rows):
    """the dense backward around the latent stage, each part from the kernel's own input to it (dpre16 itself is the
    latent stage's, checked by the fp32 parity tests)."""
    out = ref_conv1t_dgrad(pre, post, ctx, rows)
    dg0 = post["dec.fc1.dout"]
    out += zero_pads("dec.fc1.dout", dg0)
    dp = post["dpre16"]
    out += invariants("dpre16", dp) + zero_pads("dpre16", dp)
    want, scale = _heads_dgrad(dp.double(), pre["enc.conv5.out"].double().reshape(rows, 256), ctx)
    dh5 = post["enc.conv5.dout"].double().reshape(rows, 256)
    out.append(("enc.conv5.dout", dh5, want, scale, "bf16"))
    dg1 = pre["dec.conv1t.dout"].double().reshape(-1, 128)
    gd = lambda n: _grad_delta(ctx, pre, post, n)
    out.append(("dec.conv1t.b grad", gd("dec.conv1t.b"), dg1.sum(0), dg1.abs().sum(0), "f32"))
    g0 = dg0.double()[:, :45]
    out.append(("dec.fc1.b grad", gd("dec.fc1.b"), g0.sum(0), g0.abs().sum(0), "f32"))
    out.append(("enc.conv5.b grad", gd("enc.conv5.b"), dh5.sum(0), dh5.abs().sum(0), "f32"))
    # the heads' bias gradients sum the fp32 values that dpre16 stores rounded: at most 2^-9 relative apart each
    for c0, nm in ((0, "enc.locs"), (48, "enc.std")):
        d = dp.double()[:, c0:c0 + 45]
        want, a = d.sum(0), d.abs().sum(0)
        out.append((nm + ".b grad", gd(nm + ".b"), want, a + (BF16_REL / F32_REL) * a, "f32"))
    return out


def ref_conv1_wgrad(pre, post, ctx, rows):
    x = pixels("X2", pre["X2"][:rows * 1089 * 16].view(rows, 33, 33, 16))
    dh1 = pre["enc.conv1.dout"].double()
    out = _wgrad({"x": x, "d": dh1, "grad": pre["grad"]}, post, ctx, "enc.conv1", "x", "d")
    # the bias gradient comes out of the same launch (the constant 1.0 of every block)
    out.append(("enc.conv1.b grad", _grad_delta(ctx, pre, post, "enc.conv1.b"), dh1.sum((0, 1, 2)),
                dh1.abs().sum((0, 1, 2)), "f32"))
    return out


def _ops():
    """op name -> (buffers read, buffers written, reference(pre, post, ctx, rows)).  Keys: engine buffers (b[...]),
    "grad" (the flat gradient buffer), "lb:<key>" (the latent buffers), "xhat3", "ll:log_pxz" (the likelihood's output)."""
    ops = {"prep_x2": ([], ["X2"], ref_prep_x2)}
    ops["enc.conv1 fwd"] = (["X2"], ["enc.conv1.out"],
                            lambda pre, post, ctx, rows: _fwd_conv(
                                {"X2": pre["X2"][:rows * 1089 * 16].view(rows, 33, 33, 16)}, post, ctx, "enc.conv1", "X2",
                                "enc.conv1.out", False))
    for i in range(1, 5):
        name, src, dst = ENC[i], ENC[i - 1] + ".out", ENC[i] + ".out"
        ops[name + " fwd"] = ([src], [dst], lambda pre, post, ctx, rows, n=name, s=src, d=dst: _fwd_conv(
            pre, post, ctx, n, s, d, False))
    for i in range(1, 4):
        name, src, dst = DEC[i], DEC[i - 1] + ".out", DEC[i] + ".out"
        ops[name + " fwd"] = ([src], [dst], lambda pre, post, ctx, rows, n=name, s=src, d=dst: _fwd_conv(
            pre, post, ctx, n, s, d, True))
    # encoder backward: conv5 .. conv2 (dgrad into the previous layer's output gradient, masked by its output)
    for i in range(1, 5):
        name, dout, xin, dx = ENC[i], ENC[i] + ".dout", ENC[i - 1] + ".out", ENC[i - 1] + ".dout"
        ops[name + " wgrad"] = ([xin, dout, "grad"], ["grad"], lambda pre, post, ctx, rows, n=name, L=xin, S=dout: _wgrad(
            pre, post, ctx, n, L, S))
        ops[name + " bgrad"] = ([dout, "grad"], ["grad"], lambda pre, post, ctx, rows, n=name, k=dout: _bgrad(
            pre, post, ctx, n, k))
        ops[name + " dgrad"] = ([dout, xin], [dx], lambda pre, post, ctx, rows, n=name, g=dout, m=xin, d=dx: _dgrad(
            pre, post, ctx, n, g, m, d, False))
    ops["enc.conv1 wgrad"] = (["X2", "enc.conv1.dout", "grad"], ["grad"], ref_conv1_wgrad)
    # decoder backward: conv4t .. conv2t (their output gradients are L tensors)
    for i in range(1, 4):
        name, dout, xin, dx = DEC[i], DEC[i] + ".dout", DEC[i - 1] + ".out", DEC[i - 1] + ".dout"
        ops[name + " wgrad"] = ([dout, xin, "grad"], ["grad"], lambda pre, post, ctx, rows, n=name, L=dout, S=xin: _wgrad(
            pre, post, ctx, n, L, S))
        ops[name + " bgrad"] = ([dout, "grad"], ["grad"], lambda pre, post, ctx, rows, n=name, k=dout: _bgrad(
            pre, post, ctx, n, k))
        ops[name + " dgrad"] = ([dout, xin], [dx], lambda pre, post, ctx, rows, n=name, g=dout, m=xin, d=dx: _dgrad(
            pre, post, ctx, n, g, m, d, True))

    def conv5t_wgrad(pre, post, ctx, rows):
        d = pixels("D2", pre["D2"][:rows])
        return _wgrad({"d": d, "g": pre["dec.conv4t.out"], "grad": pre["grad"]}, post, ctx, "dec.conv5t", "d", "g")

    def conv5t_dgrad(pre, post, ctx, rows):
        return _dgrad({"d": pixels("D2", pre["D2"][:rows]), "m": pre["dec.conv4t.out"]}, post, ctx, "dec.conv5t", "d", "m",
                      "dec.conv4t.dout", True)

    ops["dec.conv5t fwd+recon"] = (["dec.conv4t.out", "lb:terms", "grad"], ["xhat3", "lb:log_pxz", "D2", "grad"],
                                   ref_conv5t_recon)
    ops["dec.conv5t fwd ll"] = (["dec.conv4t.out"], ["ll:log_pxz"], ref_conv5t_ll)
    ops["dec.conv5t wgrad"] = (["D2", "dec.conv4t.out", "grad"], ["grad"], conv5t_wgrad)
    ops["dec.conv5t dgrad"] = (["D2", "dec.conv4t.out"], ["dec.conv4t.dout"], conv5t_dgrad)
    ops["enc.heads fwd"] = (["enc.conv5.out"], ["pre96"],
                            lambda pre, post, ctx, rows: ref_heads_fwd(pre, post, ctx,
                                                                       pre["enc.conv5.out"].double().reshape(rows, 256)))
    ops["chain fwd"] = (["enc.conv5.out"], ["pre96", "z16", "dec.fc1.out", "dec.conv1t.out", "lb:loc", "lb:scale", "lb:z",
                                            "lb:terms", "lb:logits", "lb:y_i32"], ref_chain_fwd)
    ops["dec.fc1 fwd"] = (["z16"], ["dec.fc1.out"], ref_fc1_fwd)
    ops["dec.conv1t fwd"] = (["dec.fc1.out"], ["dec.conv1t.out"], ref_conv1t_fwd)
    ops["dec.conv1t wgrad"] = (["dec.conv1t.dout", "dec.fc1.out", "grad"], ["grad"], ref_conv1t_wgrad)
    ops["dec.conv1t bgrad"] = (["dec.conv1t.dout", "grad"], ["grad"],
                               lambda pre, post, ctx, rows: _bgrad(pre, post, ctx, "dec.conv1t", "dec.conv1t.dout"))
    ops["dec.conv1t dgrad"] = (["dec.conv1t.dout", "dec.fc1.out"], ["dec.fc1.dout"], ref_conv1t_dgrad)
    ops["dec.fc1 bgrad"] = (["dec.fc1.dout", "grad"], ["grad"],
                            lambda pre, post, ctx, rows: _bgrad(pre, post, ctx, "dec.fc1", "dec.fc1.dout", 45))
    ops["dec.fc1 wgrad"] = (["z16", "dec.fc1.dout", "grad"], ["grad"], ref_fc1_wgrad)
    ops["dec.fc1 dgrad"] = (["dec.fc1.dout"], ["dz64"], ref_fc1_dgrad)
    ops["chain bwd"] = (["dec.conv1t.dout", "dec.fc1.out", "enc.conv5.out", "grad"],
                        ["dec.fc1.dout", "dpre16", "enc.conv5.dout", "grad"], ref_chain_bwd)
    ops["enc.heads wgrad"] = (["enc.conv5.out", "dpre16", "grad"], ["grad"], ref_heads_wgrad)
    ops["enc.heads dgrad"] = (["dpre16", "enc.conv5.out"], ["enc.conv5.dout"], ref_heads_dgrad)
    return ops


OPS = _ops()
# launches without a reference of their own: every packed operand is checked through the launch that reads it
UNCHECKED = {"pack_weights"}


def check_launch(op, pre, post, ctx, rows):
    """[(label, worst |got - want| / bound)] of one recorded launch."""
    _, _, ref = OPS[op]
    return [(label, worst_ratio(got, want, scale, kind)) for label, got, want, scale, kind in ref(pre, post, ctx, rows)]
