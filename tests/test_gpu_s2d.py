"""GPU tests of the s2d (space-to-depth) storage of the stride-2 layers' L tensors at the C-ABI level: the 4-tap
L->S GEMM over blocks (Conv2D forward / Conv2DTranspose dgrad), s2d outputs and masks, and the weight gradient
with an s2d L operand, against the oracle's fp64 convolutions on the same bf16-rounded operands."""
import ctypes as C

import pytest
import torch

import gccvae_oracle as O
from launch_reference import s2d_blocks

pytestmark = pytest.mark.gpu


def _lib():
    import gccvae_b200._lib as L
    return L, L.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def bf(t):
    return t.to(torch.bfloat16).to(torch.float32)


def pack9(lib, L, W, CL, CS):
    d = W.device
    out = torch.zeros(((CS + 15) // 16 * 16) * 16 * CL, dtype=torch.bfloat16, device=d)
    job = (L.PackJob * 1)(L.PackJob(9, 16, CL, CS, L.ptr(W), L.ptr(out), 0, 0, 0, 0, 0, 0))
    L.check(lib.gccvae_pack_jobs_bf16(job, 1, _stream()))
    return out


@pytest.mark.parametrize("HL,CL,CS,B", [(32, 32, 32, 5), (16, 32, 64, 9), (8, 64, 128, 17)])
def test_s2d_ls_forward_wgrad_and_mask(HL, CL, CS, B):
    L, lib = _lib()
    from gccvae_b200._lib import Geom
    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(HL + CL)
    HS = HL // 2
    Lt = torch.relu(torch.randn(B, HL, HL, CL, generator=g))          # forward activation (also a ReLU mask)
    W = torch.randn(4, 4, CL, CS, generator=g) * 0.1
    bias = torch.randn(CS, generator=g) * 0.1
    Wd, bd = W.to(d), bias.to(d)
    L2 = s2d_blocks(bf(Lt)).to(d).to(torch.bfloat16).contiguous()
    wp = pack9(lib, L, Wd, CL, CS)
    # ---- forward, NHWC output
    S = torch.full((B, HS, HS, CS), float("nan"), dtype=torch.bfloat16, device=d)
    L.check(lib.gccvae_tap4_ls_bf16(B, HS + 1, HS + 1, 4 * CL, L.ptr(L2), L.ptr(wp), CS, L.ptr(bd), L.ACT_RELU, None,
                                    L.ptr(S), _stream()))
    torch.cuda.synchronize()
    want = torch.relu(O._conv(bf(Lt).double(), bf(W).double(), bias.double(), 2, 1))
    err = float((S.float().cpu().double() - want).abs().max() / want.abs().max())
    assert err < 6e-3, ("s2d ls fwd", err)
    # ---- the same through the halo form (two column-shifted boxes with a halo row; where the geometry does not allow
    # it the flag is ignored): same operands, same MMAs in another order -> the same bits up to fp32 summation order
    Sh = torch.full((B, HS, HS, CS), float("nan"), dtype=torch.bfloat16, device=d)
    L.check(lib.gccvae_tap4_ls_bf16(B, HS + 1, HS + 1, 4 * CL, L.ptr(L2), L.ptr(wp), CS, L.ptr(bd),
                                    L.ACT_RELU | L.TAP_HALO, None, L.ptr(Sh), _stream()))
    torch.cuda.synchronize()
    errh = float((Sh.float().cpu().double() - want).abs().max() / want.abs().max())
    assert errh < 6e-3, ("s2d ls fwd, halo form", errh)
    assert float((Sh.float() - S.float()).abs().max()) <= 2e-2 * float(S.float().abs().max())
    # ---- forward, s2d output (what the next stride-2 layer consumes)
    if HS >= 2:
        S2 = torch.zeros(B, HS // 2 + 1, HS // 2 + 1, 4 * CS, dtype=torch.bfloat16, device=d)
        L.check(lib.gccvae_tap4_ls_bf16(B, HS + 1, HS + 1, 4 * CL, L.ptr(L2), L.ptr(wp), CS, L.ptr(bd),
                                        L.ACT_RELU | L.OUT_S2D, None, L.ptr(S2), _stream()))
        torch.cuda.synchronize()
        assert torch.equal(S2.cpu().view(torch.int16), s2d_blocks(S.cpu()).view(torch.int16)), "s2d output layout"
    # ---- weight gradient with the s2d L operand
    dS = torch.randn(B, HS, HS, CS, generator=g)
    dSd = dS.to(d).to(torch.bfloat16).contiguous()
    dW = torch.zeros(4, 4, CL, CS, device=d)
    L.check(lib.gccvae_wg_s2d_bf16(B, HS, HS, CL, L.ptr(L2), L.ptr(dSd), CS, L.ptr(dW), _stream()))
    torch.cuda.synchronize()
    Wg = torch.zeros(4, 4, CL, CS, dtype=torch.float64, requires_grad=True)
    (O._conv(bf(Lt).double(), Wg, None, 2, 1) * bf(dS).double()).sum().backward()
    err = float((dW.cpu().double() - Wg.grad).abs().max() / Wg.grad.abs().max())
    assert err < 1e-4, ("s2d wgrad", err)
    # ---- dgrad of the same layer (S -> L) with the ReLU mask read from the s2d tensor == mask read from NHWC
    geom = Geom(B, HL, HL, CL, HS, HS, CS, 4, 4, 2, 1)
    Ld = bf(Lt).to(d).to(torch.bfloat16).contiguous()
    outs = []
    for mask, flag in ((Ld, 0), (L2, L.MASK_S2D)):
        dL = torch.full((B, HL, HL, CL), float("nan"), dtype=torch.bfloat16, device=d)
        if lib.gccvae_sl_halo_supported(C.byref(geom)):
            w9 = torch.zeros(lib.gccvae_packed_weight_elems(C.byref(geom), 2), dtype=torch.bfloat16, device=d)
            job = (L.PackJob * 1)(L.PackJob(6, 16, CL, CS, L.ptr(Wd), L.ptr(w9), 0, 0, 0, 0, 0, 0))
            L.check(lib.gccvae_pack_jobs_bf16(job, 1, _stream()))
            L.check(lib.gccvae_sl_halo_bf16(C.byref(geom), L.ptr(dSd), L.ptr(w9), None, L.ACT_NONE | flag, L.ptr(mask),
                                            L.ptr(dL), 0, _stream()))
        else:
            wsl = torch.empty(lib.gccvae_packed_weight_elems(C.byref(geom), 1), dtype=torch.bfloat16, device=d)
            L.check(lib.gccvae_pack_weights_bf16(C.byref(geom), L.ptr(Wd), None, L.ptr(wsl), _stream()))
            L.check(lib.gccvae_sl_bf16(C.byref(geom), L.ptr(dSd), L.ptr(wsl), None, L.ACT_NONE | flag, L.ptr(mask), L.ptr(dL),
                                       0, _stream()))
        torch.cuda.synchronize()
        outs.append(dL.cpu())
    assert torch.isfinite(outs[0].float()).all()
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16)), "s2d mask != NHWC mask"


def test_c3conv_s2d_output():
    L, lib = _lib()
    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(9)
    B = 4
    x = torch.rand(B, 64, 64, 3, generator=g).to(d)
    W = (torch.randn(4, 4, 3, 32, generator=g) * 0.2).to(d)
    bias = (torch.randn(32, generator=g) * 0.1).to(d)
    X2 = torch.empty(B, 33, 33, 16, dtype=torch.bfloat16, device=d)
    L.check(lib.gccvae_prep_x2_bf16(L.ptr(x), 0, B, L.ptr(X2), None, _stream()))
    wp = torch.zeros(32 * 64, dtype=torch.bfloat16, device=d)
    job = (L.PackJob * 1)(L.PackJob(7, 16, 3, 32, L.ptr(W), L.ptr(wp), 0, 0, 0, 0, 0, 0))
    L.check(lib.gccvae_pack_jobs_bf16(job, 1, _stream()))
    h1 = torch.empty(B, 32, 32, 32, dtype=torch.bfloat16, device=d)
    h1s = torch.zeros(B, 17, 17, 128, dtype=torch.bfloat16, device=d)
    L.check(lib.gccvae_c3conv_bf16(B, L.ptr(X2), L.ptr(wp), 32, L.ptr(bias), L.ACT_RELU, None, L.ptr(h1), _stream()))
    L.check(lib.gccvae_c3conv_bf16(B, L.ptr(X2), L.ptr(wp), 32, L.ptr(bias), L.ACT_RELU | L.OUT_S2D, None, L.ptr(h1s),
                                   _stream()))
    torch.cuda.synchronize()
    assert torch.equal(h1s.cpu().view(torch.int16), s2d_blocks(h1.cpu()).view(torch.int16))
