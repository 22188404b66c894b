"""Host-side executor of the ELBO step: owns the per-batch-size activation buffers and issues the
C-ABI kernel calls (include/gccvae.h) in the order of SURVEY.md §3.2-3.4.  PyTorch is used only
for device memory, streams and (in gated_ccvae.py) torch.distributed.

Layer table (reference: networks.py:11-18 encoder, :43-49 decoder).  Every layer is one L<->S
relation; `dir` says which side is the layer's input."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import ACT_ACCUMULATE, ACT_NONE, ACT_RELU, ACT_SIGMOID, Geom, ptr

#            name        dir   (HL,WL,CL)    (HS,WS,CS)    k  s  p  act
ENC_LAYERS = [
    ("enc.conv1", "LS", (64, 64, 3), (32, 32, 32), 4, 2, 1, ACT_RELU),
    ("enc.conv2", "LS", (32, 32, 32), (16, 16, 32), 4, 2, 1, ACT_RELU),
    ("enc.conv3", "LS", (16, 16, 32), (8, 8, 64), 4, 2, 1, ACT_RELU),
    ("enc.conv4", "LS", (8, 8, 64), (4, 4, 128), 4, 2, 1, ACT_RELU),
    ("enc.conv5", "LS", (4, 4, 128), (1, 1, 256), 4, 1, 0, ACT_RELU),
]
HEAD_LAYERS = [
    ("enc.locs", "LS", (1, 1, 256), (1, 1, 45), 1, 1, 0, ACT_NONE),
    ("enc.std", "LS", (1, 1, 256), (1, 1, 45), 1, 1, 0, ACT_NONE),
]
DEC_LAYERS = [
    ("dec.fc1", "LS", (1, 1, 45), (1, 1, 45), 1, 1, 0, ACT_RELU),
    ("dec.conv1t", "SL", (4, 4, 128), (1, 1, 45), 4, 1, 0, ACT_RELU),
    ("dec.conv2t", "SL", (8, 8, 64), (4, 4, 128), 4, 2, 1, ACT_RELU),
    ("dec.conv3t", "SL", (16, 16, 32), (8, 8, 64), 4, 2, 1, ACT_RELU),
    ("dec.conv4t", "SL", (32, 32, 32), (16, 16, 32), 4, 2, 1, ACT_RELU),
    ("dec.conv5t", "SL", (64, 64, 3), (32, 32, 32), 4, 2, 1, ACT_SIGMOID),
]


def make_geom(layer, batch) -> Geom:
    _, _, (HL, WL, CL), (HS, WS, CS), k, s, p, _ = layer
    return Geom(batch, HL, WL, CL, HS, WS, CS, k, k, s, p)


def in_shape(layer):
    return layer[2] if layer[1] == "LS" else layer[3]


def out_shape(layer):
    return layer[3] if layer[1] == "LS" else layer[2]


def image_u8(xhat):
    """fp32 image in [0,1] -> uint8 min(255, rint(255 x)): fp32 product, round half to even (the rule of
    gccvae_convt_image_bf16)."""
    return torch.clamp(torch.round(xhat * 255.0), max=255.0).to(torch.uint8)


def _stream():
    return torch.cuda.current_stream().cuda_stream


class Engine:
    """fp32 (exact, CUDA-core) executor.  The bf16 tcgen05 executor subclasses this."""

    precision = "fp32"

    def __init__(self, store):
        self.lib = _lib.load()
        self.store = store
        self.device = store.device
        if self.device.type != "cuda":
            raise _lib.GccvaeError("the Gated-CCVAE kernels run on a CUDA device only (got {})".format(self.device))
        _lib.check(self.lib.gccvae_arch_check(self.device.index or 0), "arch_check")
        self._bufs = {}
        self._dec_bufs = {}

    # ---- buffers -----------------------------------------------------------------------------------
    def bufs(self, batch):
        b = self._bufs.get(batch)
        if b is None:
            b = self._alloc(batch)
            self._bufs[batch] = b
        return b

    def _alloc(self, B):
        dev, f32 = self.device, torch.float32
        e = lambda *s: torch.empty(*s, dtype=f32, device=dev)
        b = {}
        for lay in ENC_LAYERS + HEAD_LAYERS + DEC_LAYERS:
            oh, ow, oc = out_shape(lay)
            b[lay[0] + ".out"] = e(B, oh, ow, oc)
            b[lay[0] + ".dout"] = e(B, oh, ow, oc)   # gradient w.r.t. this layer's pre-activation
        b["dz"] = e(B, 45)
        ws_bytes = 0
        for lay in ENC_LAYERS + HEAD_LAYERS + DEC_LAYERS:
            g = make_geom(lay, B)
            ws_bytes = max(ws_bytes, self.lib.gccvae_wg_f32_workspace_bytes(C.byref(g)))
            oh, ow, oc = out_shape(lay)
            ws_bytes = max(ws_bytes, self.lib.gccvae_colsum_f32_workspace_bytes(B * oh * ow, oc))
        b["ws"] = torch.empty(ws_bytes // 4 + 16, dtype=f32, device=dev)
        b["ws_bytes"] = ws_bytes
        return b

    def dec_bufs(self, rows):
        """forward-only decoder buffers for `rows` latent rows (importance-weighted likelihood): the decoder's
        activations and its input z [rows,45], without the encoder's tensors or any gradient."""
        b = self._dec_bufs.get(rows)
        if b is None:
            b = {lay[0] + ".out": torch.empty(rows, *out_shape(lay), dtype=torch.float32, device=self.device)
                 for lay in DEC_LAYERS}
            b["z"] = torch.empty(rows, 45, dtype=torch.float32, device=self.device)
            self._dec_bufs[rows] = b
        return b

    # ---- single layer ops -------------------------------------------------------------------------------
    def layer_fwd(self, lay, B, x, out):
        g = make_geom(lay, B)
        W, bias = self.store.view(lay[0] + ".w"), self.store.view(lay[0] + ".b")
        fn = self.lib.gccvae_ls_f32 if lay[1] == "LS" else self.lib.gccvae_sl_f32
        _lib.check(fn(C.byref(g), ptr(x), ptr(W), ptr(bias), lay[7], None, ptr(out), _stream()), lay[0] + " fwd")

    def layer_bwd(self, lay, B, x, dout, dx, mask, ws, ws_bytes, accumulate=False):
        """dout = grad of this layer's pre-activation.  Writes dW, db into the flat grad buffer and,
        if dx is given, dx = dgrad(dout) * (mask > 0) (mask = the producer layer's ReLU output)."""
        g = make_geom(lay, B)
        W = self.store.view(lay[0] + ".w")
        dW, db = self.store.g(lay[0] + ".w"), self.store.g(lay[0] + ".b")
        st = _stream()
        oh, ow, oc = out_shape(lay)
        L, S = (x, dout) if lay[1] == "LS" else (dout, x)
        _lib.check(self.lib.gccvae_wg_f32(C.byref(g), ptr(L), ptr(S), ptr(dW), ptr(ws), ws_bytes, st), lay[0] + " wgrad")
        _lib.check(self.lib.gccvae_colsum_f32(ptr(dout), B * oh * ow, oc, ptr(db), ptr(ws), ws_bytes, st),
                   lay[0] + " bgrad")
        if dx is not None:
            act = ACT_ACCUMULATE if accumulate else ACT_NONE
            fn = self.lib.gccvae_sl_f32 if lay[1] == "LS" else self.lib.gccvae_ls_f32
            _lib.check(fn(C.byref(g), ptr(dout), ptr(W), None, act, ptr(mask), ptr(dx), st), lay[0] + " dgrad")

    # ---- step hooks shared with the tensor-core engine ------------------------------------------------
    def latent_io(self, b):
        """device pointers / strides through which the fused latent kernels talk to this engine."""
        return dict(loc_pre=ptr(b["enc.locs.out"]), scale_pre=ptr(b["enc.std.out"]), ld_pre=45, z16=None,
                    dz=ptr(b["dz"]), ld_dz=45, dloc_pre=ptr(b["enc.locs.dout"]), dscale_pre=ptr(b["enc.std.dout"]),
                    dpre16=None, db_loc=None, db_scale=None)

    def zero_grads(self):
        """the fp32 kernels overwrite every gradient; nothing to clear."""

    def pack_weights(self, part=None):
        """the fp32 kernels read the fp32 master weights; nothing to pack."""

    def recon(self, x, b, coef, log_pxz, backward):
        """utils.py:101-105 (+ gradient w.r.t. the decoder's pre-sigmoid logits when backward)."""
        B = x.shape[0]
        xhat = b["dec.conv5t.out"]
        dlogit = b["dec.conv5t.dout"] if backward else None
        _lib.check(self.lib.gccvae_recon_f32(ptr(x), ptr(xhat), B, 64 * 64 * 3, ptr(coef) if backward else None,
                                             ptr(log_pxz), ptr(dlogit), _stream()), "recon")
        return xhat

    # ---- encoder / decoder chains ---------------------------------------------------------------------
    def encoder_fwd(self, x, b):
        B = x.shape[0]
        h = x
        for lay in ENC_LAYERS:
            self.layer_fwd(lay, B, h, b[lay[0] + ".out"])
            h = b[lay[0] + ".out"]
        for lay in HEAD_LAYERS:
            self.layer_fwd(lay, B, h, b[lay[0] + ".out"])
        return b["enc.locs.out"].view(B, 45), b["enc.std.out"].view(B, 45)

    def decoder_fwd(self, z, b, z16_ready=False):
        B = z.shape[0]
        h = z
        for lay in DEC_LAYERS:
            self.layer_fwd(lay, B, h, b[lay[0] + ".out"])
            h = b[lay[0] + ".out"]
        return h

    def image_fwd(self, z, b, batch, out_u8, out=None):
        """generation path: the decoder from the latent code z [B,45] -> a fresh [B,64,64,3] image, the fp32 sigmoid
        values or (out_u8) uint8 min(255, rint(255 xhat)) with the product and the rounding in fp32.  `out`: a contiguous
        [batch,64,64,3] tensor of that dtype (e.g. a row slice of a larger image tensor) to write instead; z and the
        buffer set b (`bufs` or `dec_bufs`) may then hold more rows than `batch`, and only the first `batch` are decoded."""
        if out is None:
            xhat = self.decoder_fwd(z, b)
            return image_u8(xhat) if out_u8 else xhat.clone()
        h = z[:batch]
        for lay in DEC_LAYERS:
            dst = out if lay is DEC_LAYERS[-1] and not out_u8 else b[lay[0] + ".out"]
            self.layer_fwd(lay, batch, h, dst)
            h = dst
        if out_u8:
            out.copy_(image_u8(h[:batch]))
        return out

    def complete_begin(self, x, mask):
        """per-call state of image completion: the pixel mask [B,64,64] bool (True = observed) and the composite image
        the encoder reads from the second iteration on."""
        return {"mask": mask.unsqueeze(-1), "img": torch.empty_like(x)}

    def complete_fwd(self, z, b, batch, state, x):
        """one iteration of image completion (the parity path): decode z, then the composite where(mask, x, xhat) of the
        fp32 image x into the image the next encoder pass reads, which is returned."""
        xhat = self.decoder_fwd(z[:batch], b)
        return torch.where(state["mask"], x, xhat, out=state["img"])

    def iw_decoder_ll(self, x, b, batch, kc, dec, log_pxz):
        """importance-weighted likelihood: log_pxz[r] = log p(x_(r / kc) | z_r) for the batch * kc rows of dec["z"]
        (the parity path: the generic decoder, then the reconstruction likelihood against the repeated images)."""
        rows = batch * kc
        xhat = self.decoder_fwd(dec["z"][:rows], dec)
        xr = x.repeat_interleave(kc, 0) if kc > 1 else x
        _lib.check(self.lib.gccvae_recon_f32(ptr(xr), ptr(xhat), rows, 64 * 64 * 3, None, ptr(log_pxz), None,
                                             _stream()), "recon")

    def decoder_bwd(self, z, b, want_dz=True):
        """expects b['dec.conv5t.dout'] = dLoss/d(pre-sigmoid logits); returns dz."""
        B = z.shape[0]
        ws, wsb = b["ws"], b["ws_bytes"]
        for i in range(len(DEC_LAYERS) - 1, -1, -1):
            lay = DEC_LAYERS[i]
            if i > 0:
                prev = DEC_LAYERS[i - 1]
                x, dx, mask = b[prev[0] + ".out"], b[prev[0] + ".dout"], b[prev[0] + ".out"]
            else:
                x, dx, mask = z, (b["dz"] if want_dz else None), None
            self.layer_bwd(lay, B, x, b[lay[0] + ".dout"], dx, mask, ws, wsb)
        return b["dz"]

    def encoder_bwd(self, x, b):
        """expects b['enc.locs.dout'], b['enc.std.dout'] = grads of the heads' pre-activations."""
        B = x.shape[0]
        ws, wsb = b["ws"], b["ws_bytes"]
        h5, dh5 = b["enc.conv5.out"], b["enc.conv5.dout"]
        self.layer_bwd(HEAD_LAYERS[0], B, h5, b["enc.locs.dout"], dh5, None, ws, wsb)
        self.layer_bwd(HEAD_LAYERS[1], B, h5, b["enc.std.dout"], dh5, h5, ws, wsb, accumulate=True)
        for i in range(len(ENC_LAYERS) - 1, -1, -1):
            lay = ENC_LAYERS[i]
            if i > 0:
                prev = ENC_LAYERS[i - 1]
                xin, dx, mask = b[prev[0] + ".out"], b[prev[0] + ".dout"], b[prev[0] + ".out"]
            else:
                xin, dx, mask = x, None, None
            self.layer_bwd(lay, B, xin, b[lay[0] + ".dout"], dx, mask, ws, wsb)
