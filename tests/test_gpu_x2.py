"""GPU tests of the space-to-depth ("x2") end layers at the C-ABI level: the block transform of the input
(fp32 and uint8), conv1 forward / weight gradient as 4-tap GEMMs over the blocks, and the fused
conv5t + sigmoid + Laplace log-likelihood kernel with its gradient in block form, each against the oracle's
fp64 convolutions on the same bf16-rounded operands."""
import ctypes as C

import numpy as np
import pytest
import torch

import gccvae_oracle as O
from launch_reference import _raw_byte_blocks, x2_blocks

pytestmark = pytest.mark.gpu


def _lib():
    import gccvae_b200._lib as L
    return L, L.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def bf(t):
    return t.to(torch.bfloat16).to(torch.float32)


def pack(lib, L, kind, W, n_out):
    d = W.device
    out = torch.zeros(n_out, dtype=torch.bfloat16, device=d)
    job = (L.PackJob * 1)(L.PackJob(kind, 16, 3, 32, L.ptr(W), L.ptr(out), 0, 0, 0, 0, 0, 0))
    L.check(lib.gccvae_pack_jobs_bf16(job, 1, _stream()))
    return out


@pytest.mark.parametrize("u8", [False, True])
def test_prep_x2(u8):
    L, lib = _lib()
    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(3)
    B = 5
    if u8:
        xi = torch.randint(0, 256, (B, 64, 64, 3), generator=g, dtype=torch.uint8)
        x = torch.from_numpy(xi.numpy().astype(np.float32) / 255.0)      # utils_data.py:56-59
        xin = xi.to(d)
    else:
        x = torch.rand(B, 64, 64, 3, generator=g)
        xin = x.to(d)
    X2 = torch.full((B, 33, 33, 16), float("nan"), dtype=torch.bfloat16, device=d)
    L.check(lib.gccvae_prep_x2_bf16(L.ptr(xin), int(u8), B, L.ptr(X2), None, _stream()))
    torch.cuda.synchronize()
    want = x2_blocks(x, ones=True).to(torch.bfloat16)
    assert torch.equal(X2.cpu().view(torch.int16), want.view(torch.int16)), "x2 block transform must be bit-exact"
    if u8:
        # the raw-byte blocks (image operand of the fused likelihood kernel): staged kernel (16-byte aligned image) and
        # the per-block kernel (unaligned image) must both give the block's 12 bytes + 4 zero bytes, zero outside the image
        want_b = _raw_byte_blocks(xi)
        for shift in (0, 1):
            buf = torch.zeros(xi.numel() + 16, dtype=torch.uint8, device=d)
            buf[shift:shift + xi.numel()] = xi.reshape(-1).to(d)
            XB = torch.full((B, 33, 33, 16), 0xAB, dtype=torch.uint8, device=d)
            X2.fill_(float("nan"))
            L.check(lib.gccvae_prep_x2_bf16(L.ptr(buf) + shift, 1, B, L.ptr(X2), L.ptr(XB), _stream()))
            torch.cuda.synchronize()
            assert torch.equal(XB.cpu(), want_b), ("raw-byte blocks", shift)
            assert torch.equal(X2.cpu().view(torch.int16), want.view(torch.int16))
    else:
        assert lib.gccvae_prep_x2_bf16(L.ptr(xin), 0, B, L.ptr(X2), L.ptr(X2), _stream()) != 0   # fp32 images have no raw bytes


def test_u8_normalisation_is_bit_exact_for_all_256_values():
    """device: __fdiv_rn(float(u), 255.0f) == numpy float32(u) / 255.0 for every byte value."""
    L, lib = _lib()
    d = torch.device("cuda", 0)
    vals = torch.arange(256, dtype=torch.uint8)
    xi = vals.repeat(48)[:64 * 64 * 3].reshape(1, 64, 64, 3).contiguous()
    want = torch.from_numpy(xi.numpy().astype(np.float32) / 255.0)
    # through the fused likelihood kernel: with the decoder output forced to 0.5 (zero weights and bias),
    # log_pxz = -sum |x - 0.5| - 12288 ln 2 in fp32 -> compare against the same sum of the host-normalised image
    g4 = torch.zeros(1, 32, 32, 32, dtype=torch.bfloat16, device=d)
    w8 = torch.zeros(16 * 128, dtype=torch.bfloat16, device=d)
    b3 = torch.zeros(3, device=d)
    lp = torch.zeros(1, device=d)
    xh = torch.zeros(1, 64, 64, 3, device=d)
    L.check(lib.gccvae_convt_recon_bf16(1, L.ptr(g4), L.ptr(w8), L.ptr(b3), L.ptr(xi.to(d)), 1, None, L.ptr(lp), None,
                                        L.ptr(xh), None, 0, _stream()))
    torch.cuda.synchronize()
    ref = -(want.double() - 0.5).abs().sum() - 12288 * np.log(2.0)
    assert abs(float(lp[0]) - float(ref)) / abs(float(ref)) < 1e-6
    assert float((xh - 0.5).abs().max()) == 0.0


@pytest.mark.parametrize("impl", ["tma", "threads"])
def test_conv1_x2_forward_and_wgrad(impl):
    L, lib = _lib()

    def ls(X2, wp, bias, act, mask, out):
        if impl == "tma":
            return lib.gccvae_tap4_ls_bf16(B, 33, 33, 16, L.ptr(X2), L.ptr(wp), 32, L.ptr(bias), act, L.ptr(mask),
                                           L.ptr(out), _stream())
        return lib.gccvae_c3conv_bf16(B, L.ptr(X2), L.ptr(wp), 32, L.ptr(bias), act, L.ptr(mask), L.ptr(out), _stream())

    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(5)
    B = 6
    x = torch.rand(B, 64, 64, 3, generator=g)
    W = torch.randn(4, 4, 3, 32, generator=g) * 0.2
    bias = torch.randn(32, generator=g) * 0.1
    xd, Wd, bd = x.to(d), W.to(d), bias.to(d)
    X2 = torch.empty(B, 33, 33, 16, dtype=torch.bfloat16, device=d)
    L.check(lib.gccvae_prep_x2_bf16(L.ptr(xd), 0, B, L.ptr(X2), None, _stream()))
    wp = pack(lib, L, 7, Wd, 32 * 64)
    h1 = torch.full((B, 32, 32, 32), float("nan"), dtype=torch.bfloat16, device=d)
    L.check(ls(X2, wp, bd, L.ACT_RELU, None, h1))
    torch.cuda.synchronize()
    want = torch.relu(O._conv(bf(x).double(), bf(W).double(), bias.double(), 2, 1))
    err = float((h1.float().cpu().double() - want).abs().max() / want.abs().max())
    assert err < 6e-3, ("conv1 x2 fwd", err)
    # masked variant (the form conv5t's dgrad uses)
    mask = (torch.rand(B, 32, 32, 32, generator=g) < 0.5).float()
    md = mask.to(d).to(torch.bfloat16)
    L.check(ls(X2, wp, None, L.ACT_NONE, md, h1))
    torch.cuda.synchronize()
    want = O._conv(bf(x).double(), bf(W).double(), None, 2, 1) * mask.double()
    err = float((h1.float().cpu().double() - want).abs().max() / want.abs().max())
    assert err < 6e-3, ("conv1 x2 masked", err)
    # weight gradient
    dh1 = torch.randn(B, 32, 32, 32, generator=g)
    dh1d = dh1.to(d).to(torch.bfloat16).contiguous()
    dW = torch.zeros(4, 4, 3, 32, device=d)
    db = torch.full((32,), 0.25, device=d)      # the kernel ADDS the bias gradient (ones slot of prep_x2's blocks)
    L.check(lib.gccvae_tap4_wg_bf16(B, L.ptr(X2), L.ptr(dh1d), 32, L.ptr(dW), L.ptr(db), _stream()))
    torch.cuda.synchronize()
    Wg = torch.zeros(4, 4, 3, 32, dtype=torch.float64, requires_grad=True)
    (O._conv(bf(x).double(), Wg, None, 2, 1) * bf(dh1).double()).sum().backward()
    err = float((dW.cpu().double() - Wg.grad).abs().max() / Wg.grad.abs().max())
    assert err < 1e-4, ("conv1 x2 wgrad", err)
    want_db = bf(dh1).double().sum((0, 1, 2))
    err = float((db.cpu().double() - 0.25 - want_db).abs().max() / want_db.abs().max())
    assert err < 1e-5, ("conv1 bias gradient from the ones row", err)
    # without db the ones row is dropped like the other pad rows
    dW2 = torch.zeros(4, 4, 3, 32, device=d)
    L.check(lib.gccvae_tap4_wg_bf16(B, L.ptr(X2), L.ptr(dh1d), 32, L.ptr(dW2), None, _stream()))
    torch.cuda.synchronize()
    assert float((dW2 - dW).abs().max()) <= 1e-5 * float(dW.abs().max())


@pytest.mark.parametrize("B", [5, 1, 70])
@pytest.mark.parametrize("u8", [0, 1, 2])
def test_fused_conv5t_recon(u8, B):
    """u8 = form of the image operand: 0 fp32 image, 1 uint8 image, 2 the raw-byte blocks of prep_x2.  Batch 70 (630 tiles,
    more than the 592 resident CTAs) gives every CTA a range of two tiles, some of which cross an image boundary."""
    L, lib = _lib()
    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(7)
    if u8:
        xi = torch.randint(0, 256, (B, 64, 64, 3), generator=g, dtype=torch.uint8)
        x = torch.from_numpy(xi.numpy().astype(np.float32) / 255.0)
        xin = xi.to(d)
        if u8 == 2:
            xin = _raw_byte_blocks(xi).to(d)
    else:
        x = torch.rand(B, 64, 64, 3, generator=g)
        xin = x.to(d)
    g4 = torch.relu(torch.randn(B, 32, 32, 32, generator=g))
    W5 = torch.randn(4, 4, 3, 32, generator=g) * 0.1
    b5 = torch.randn(3, generator=g) * 0.1
    coef = -(torch.rand(B, generator=g) + 0.5) / B
    g4d, W5d, b5d, coefd = g4.to(d).to(torch.bfloat16).contiguous(), W5.to(d), b5.to(d), coef.to(d)
    w8 = pack(lib, L, 8, W5d, 16 * 128)
    lpx = torch.empty(B, device=d)
    D2 = torch.full((B, 33, 33, 16), float("nan"), dtype=torch.bfloat16, device=d)
    xhat = torch.full((B, 64, 64, 3), float("nan"), device=d)
    db = torch.zeros(3, device=d)
    L.check(lib.gccvae_convt_recon_bf16(B, L.ptr(g4d), L.ptr(w8), L.ptr(b5d), L.ptr(xin), u8, L.ptr(coefd), L.ptr(lpx),
                                        L.ptr(D2), L.ptr(xhat), L.ptr(db), 0, _stream()))
    torch.cuda.synchronize()
    want_xh = torch.sigmoid(O._convT(bf(g4).double(), bf(W5).double(), b5.double(), 2, 1))
    got_xh = xhat.cpu().double()
    assert torch.isfinite(xhat).all()
    assert float((got_xh - want_xh).abs().max()) < 1e-4, "fused conv5t forward"
    want_ll = O.img_log_likelihood(got_xh, x.double())
    assert float(((lpx.cpu().double() - want_ll) / want_ll).abs().max()) < 1e-5, "log_pxz"
    dlogit = coef.double().view(B, 1, 1, 1) * torch.sign(x.double() - got_xh) * got_xh * (1 - got_xh)
    want_D2 = x2_blocks(dlogit.float()).to(torch.bfloat16)
    assert torch.isfinite(D2.float()).all()
    assert float((D2.float().cpu() - want_D2.float()).abs().max()) <= float(want_D2.float().abs().max()) * 2 ** -7
    assert float((db.cpu().double() - dlogit.sum((0, 1, 2))).abs().max() / dlogit.sum((0, 1, 2)).abs().max()) < 1e-3
    # forward-only form: no gradient outputs
    lp2 = torch.empty(B, device=d)
    L.check(lib.gccvae_convt_recon_bf16(B, L.ptr(g4d), L.ptr(w8), L.ptr(b5d), L.ptr(xin), u8, None, L.ptr(lp2), None,
                                        None, None, 0, _stream()))
    torch.cuda.synchronize()
    assert float((lp2 - lpx).abs().max() / lpx.abs().max()) < 1e-6
    # dgrad and wgrad of conv5t from D2
    wp7 = pack(lib, L, 7, W5d, 32 * 64)
    dg4 = torch.empty(B, 32, 32, 32, dtype=torch.bfloat16, device=d)
    L.check(lib.gccvae_c3conv_bf16(B, L.ptr(D2), L.ptr(wp7), 32, None, L.ACT_NONE, L.ptr(g4d), L.ptr(dg4), _stream()))
    dW5 = torch.zeros(4, 4, 3, 32, device=d)
    L.check(lib.gccvae_tap4_wg_bf16(B, L.ptr(D2), L.ptr(g4d), 32, L.ptr(dW5), None, _stream()))
    torch.cuda.synchronize()
    want = O._conv(bf(dlogit.float()).double(), bf(W5).double(), None, 2, 1) * (bf(g4).double() > 0)
    err = float((dg4.float().cpu().double() - want).abs().max() / want.abs().max())
    assert err < 1e-2, ("conv5t dgrad from D2", err)
    Wg = torch.zeros(4, 4, 3, 32, dtype=torch.float64, requires_grad=True)
    (O._conv(bf(dlogit.float()).double(), Wg, None, 2, 1) * bf(g4).double()).sum().backward()
    err = float((dW5.cpu().double() - Wg.grad).abs().max() / Wg.grad.abs().max())
    assert err < 1e-3, ("conv5t wgrad from D2", err)
