"""GPU tests of the bf16 tensor-core path (tcgen05 / TMEM / TMA) at the C-ABI level: TMA box semantics,
then every tap-GEMM configuration against torch's fp64 convolution on the same bf16-rounded operands.
Tolerance: the only differences are fp32 accumulation order and the final bf16 rounding of the
output (2^-9 relative), so 6e-3 of the tensor's max."""
import ctypes as C

import numpy as np
import pytest
import torch

import gccvae_oracle as O

pytestmark = pytest.mark.gpu
TOL = 6e-3


def _lib():
    import gccvae_b200._lib as L
    return L, L.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _swz(off, row_bytes):
    """byte offset inside a TMA/UMMA swizzled tile (swizzle span = row_bytes in {32,64,128})."""
    bits = {128: 7, 64: 3, 32: 1, 16: 0}[row_bytes]
    return off ^ (((off >> 7) & bits) << 4)


@pytest.mark.parametrize("C_,kc,es", [(32, 32, 2), (64, 64, 2), (32, 32, 1), (128, 64, 1), (16, 16, 2)])
def test_tma_box_layout(C_, kc, es):
    """Strided 4-D box: element (dn,dy,dx,c) of the box is src[n0+dn, h0+es*dy, w0+es*dx, c0+c], zero when
    out of the image, and lands at row (dn*BH+dy)*BW+dx of a 128-row K-major swizzled tile."""
    L, lib = _lib()
    d = torch.device("cuda", 0)
    N, H, W = 3, 16, 16
    bw, bh, bn = 8, 8, 2
    src = torch.arange(N * H * W * C_, dtype=torch.float32).reshape(N, H, W, C_) % 251 + 1
    src_d = src.to(d).to(torch.bfloat16).contiguous()
    nbytes = kc * bw * bh * bn * 2
    out = torch.zeros(nbytes, dtype=torch.uint8, device=d)
    c0, w0, h0, n0 = (C_ - kc), -1, -1, 1
    L.check(lib.gccvae_debug_tma4d(L.ptr(src_d), N, H, W, C_, kc, bw, bh, bn, es, c0, w0, h0, n0, L.ptr(out), nbytes,
                                   _stream()))
    torch.cuda.synchronize()
    raw = out.cpu().numpy().view(np.uint16)
    got = torch.from_numpy(raw.astype(np.int32) << 16).view(torch.float32)  # bf16 bits -> f32
    row_bytes = kc * 2
    bad = 0
    for dn in range(bn):
        for dy in range(bh):
            for dx in range(bw):
                r = (dn * bh + dy) * bw + dx
                n, y, x = n0 + dn, h0 + es * dy, w0 + es * dx
                for c in range(0, kc, 8):
                    off = _swz(r * row_bytes + c * 2, row_bytes)
                    want = src[n, y, x, c0 + c:c0 + c + 8] if (0 <= n < N and 0 <= y < H and 0 <= x < W) else torch.zeros(8)
                    g = got[off // 2: off // 2 + 8]
                    if not torch.equal(g, want.to(torch.bfloat16).float()):
                        bad += 1
                        if bad < 4:
                            print("mismatch r", r, "c", c, "got", g.tolist(), "want", want.tolist())
    assert bad == 0, "{} mismatching 16-byte chunks".format(bad)


def _run_tc(direction, geom_t, batch, act, use_mask, use_bias=True):
    """geom_t = (HL,WL,CL),(HS,WS,CS),k,s,p"""
    L, lib = _lib()
    from gccvae_b200._lib import Geom
    (HL, WL, CL), (HS, WS, CS), k, s, p = geom_t
    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(HL * 131 + CL)
    bf = lambda t: t.to(torch.bfloat16)
    W = torch.randn(k, k, CL, CS, generator=g) * (1.0 / (k * (CL if direction == "LS" else CS) ** 0.5))
    geom = Geom(batch, HL, WL, CL, HS, WS, CS, k, k, s, p)
    Wd = W.to(d)
    n_ls, n_sl = lib.gccvae_packed_weight_elems(C.byref(geom), 0), lib.gccvae_packed_weight_elems(C.byref(geom), 1)
    wp_ls = torch.zeros(n_ls, dtype=torch.bfloat16, device=d)
    wp_sl = torch.zeros(n_sl, dtype=torch.bfloat16, device=d)
    sl_ok = (HS == 1 and WS == 1) or (k == 4 and s == 2 and p == 1)
    L.check(lib.gccvae_pack_weights_bf16(C.byref(geom), L.ptr(Wd), L.ptr(wp_ls), L.ptr(wp_sl) if sl_ok else None, _stream()))
    Wr = bf(W).double()
    if direction == "LS":
        X = torch.randn(batch, HL, WL, CL, generator=g)
        bias = torch.randn(CS, generator=g) if use_bias else None
        mask = torch.randn(batch, HS, WS, CS, generator=g) if use_mask else None
        want = O._conv(bf(X).double(), Wr, None if bias is None else bias.double(), s, p)
    else:
        X = torch.randn(batch, HS, WS, CS, generator=g)
        bias = torch.randn(CL, generator=g) if use_bias else None
        mask = torch.randn(batch, HL, WL, CL, generator=g) if use_mask else None
        want = O._convT(bf(X).double(), Wr, None if bias is None else bias.double(), s, p)
    if act == L.ACT_RELU:
        want = torch.relu(want)
    elif act == L.ACT_SIGMOID:
        want = torch.sigmoid(want)
    if mask is not None:
        want = want * (bf(mask).double() > 0)
    Xd = bf(X).to(d).contiguous()
    bd = None if bias is None else bias.to(d)
    md = None if mask is None else bf(mask).to(d).contiguous()
    out = torch.full(want.shape, float("nan"), dtype=torch.bfloat16, device=d)
    fn = lib.gccvae_ls_bf16 if direction == "LS" else lib.gccvae_sl_bf16
    L.check(fn(C.byref(geom), L.ptr(Xd), L.ptr(wp_ls if direction == "LS" else wp_sl), L.ptr(bd), act, L.ptr(md),
               L.ptr(out), 0, _stream()))
    torch.cuda.synchronize()
    got = out.float().cpu().double()
    assert torch.isfinite(got).all(), "output has NaN/unwritten elements"
    err = float((got - want).abs().max() / want.abs().max())
    if direction == "SL" and lib.gccvae_sl_halo_supported(C.byref(geom)):
        # the same layer through the halo kernel ("sl9" packing, one wide MMA per shifted view)
        w9 = torch.zeros(lib.gccvae_packed_weight_elems(C.byref(geom), 2), dtype=torch.bfloat16, device=d)
        job = (L.PackJob * 1)(L.PackJob(6, 16, CL, CS, L.ptr(Wd), L.ptr(w9), 0, 0, 0, 0, 0, 0))
        L.check(lib.gccvae_pack_jobs_bf16(job, 1, _stream()))
        out2 = torch.full(want.shape, float("nan"), dtype=torch.bfloat16, device=d)
        L.check(lib.gccvae_sl_halo_bf16(C.byref(geom), L.ptr(Xd), L.ptr(w9), L.ptr(bd), act, L.ptr(md), L.ptr(out2), 0,
                                        _stream()))
        torch.cuda.synchronize()
        got2 = out2.float().cpu().double()
        assert torch.isfinite(got2).all(), "halo output has NaN/unwritten elements"
        err = max(err, float((got2 - want).abs().max() / want.abs().max()))
    return err


LS_GEOMS = {
    "conv2": ((32, 32, 32), (16, 16, 32), 4, 2, 1),
    "conv3": ((16, 16, 32), (8, 8, 64), 4, 2, 1),
    "conv4": ((8, 8, 64), (4, 4, 128), 4, 2, 1),
    "conv5": ((4, 4, 128), (1, 1, 256), 4, 1, 0),
    "conv2t": ((8, 8, 64), (4, 4, 128), 4, 2, 1),
    "conv3t": ((16, 16, 32), (8, 8, 64), 4, 2, 1),
    "conv4t": ((32, 32, 32), (16, 16, 32), 4, 2, 1),
}


@pytest.mark.parametrize("name", ["conv2", "conv3", "conv4", "conv5"])
@pytest.mark.parametrize("batch", [2, 19, 256])
def test_tc_ls_forward(name, batch):
    L, _ = _lib()
    err = _run_tc("LS", LS_GEOMS[name], batch, L.ACT_RELU, False)
    assert err < TOL, err


@pytest.mark.parametrize("name", ["conv2t", "conv3t", "conv4t"])
@pytest.mark.parametrize("batch", [2, 19, 256])
def test_tc_sl_forward(name, batch):
    L, _ = _lib()
    err = _run_tc("SL", LS_GEOMS[name], batch, L.ACT_RELU, False)
    assert err < TOL, err


@pytest.mark.parametrize("name", ["conv2", "conv3", "conv4", "conv5"])
def test_tc_sl_as_conv_dgrad(name):
    L, _ = _lib()
    err = _run_tc("SL", LS_GEOMS[name], 24, L.ACT_NONE, True, use_bias=False)
    assert err < TOL, err


@pytest.mark.parametrize("name", ["conv2t", "conv3t", "conv4t"])
def test_tc_ls_as_convT_dgrad(name):
    L, _ = _lib()
    err = _run_tc("LS", LS_GEOMS[name], 24, L.ACT_NONE, True, use_bias=False)
    assert err < TOL, err


@pytest.mark.parametrize("name", ["conv2", "conv3", "conv4", "conv5", "conv2t", "conv3t", "conv4t"])
@pytest.mark.parametrize("batch", [3, 64, 300])
def test_tc_wgrad(name, batch):
    L, lib = _lib()
    from gccvae_b200._lib import Geom
    (HL, WL, CL), (HS, WS, CS), k, s, p = LS_GEOMS[name]
    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(7 + HL)
    bf = lambda t: t.to(torch.bfloat16)
    Lt = torch.randn(batch, HL, WL, CL, generator=g)
    St = torch.randn(batch, HS, WS, CS, generator=g)
    geom = Geom(batch, HL, WL, CL, HS, WS, CS, k, k, s, p)
    Ld = bf(Lt).to(d).contiguous()
    Sd = bf(St).to(d).contiguous()
    dW = torch.zeros(k, k, CL, CS, device=d)
    L.check(lib.gccvae_wg_bf16(C.byref(geom), L.ptr(Ld), L.ptr(Sd), L.ptr(dW), _stream()))
    db = torch.zeros(CS, device=d)
    L.check(lib.gccvae_colsum_bf16(L.ptr(Sd), batch * HS * WS, CS, 0, L.ptr(db), _stream()))
    torch.cuda.synchronize()
    Wd = torch.zeros(k, k, CL, CS, dtype=torch.float64, requires_grad=True)
    (O._conv(bf(Lt).double(), Wd, None, s, p) * bf(St).double()).sum().backward()
    err = float((dW.cpu().double() - Wd.grad).abs().max() / Wd.grad.abs().max())
    assert err < 1e-4, err      # fp32 accumulation of exact bf16 products
    errb = float((db.cpu().double() - bf(St).double().sum((0, 1, 2))).abs().max() / bf(St).double().sum((0, 1, 2)).abs().max())
    assert errb < 1e-4, errb
