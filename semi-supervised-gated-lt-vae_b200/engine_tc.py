"""bf16 tensor-core executor of the ELBO step (tcgen05 / TMEM / TMA kernels of csrc/conv_tc.cu).

Activations between the convolutions are bf16; accumulation, biases, the latent stage, the losses and all gradients
of parameters are fp32.  Layer -> kernel map of the default (x2 + s2d) mode, DESIGN.md "Data layout in HBM":

  image            fp32 or uint8 [B,64,64,3] -> x2 blocks [B,33,33,16] (prep_x2; u8/255 through an exact table)
  enc.conv1        c3conv (thread-built im2col tile from x2 blocks, K = 64); wgrad tap4_wg from the same blocks
  enc.conv2-4      tap-GEMM over the s2d form of the input (4 taps x 4 C_L); dgrad = halo kernel (conv2, conv3) or
                   4-phase tap-GEMM; wgrad = wg_s2d (MN-major operands straight from TMA boxes, split-K)
  enc.conv5, heads, dec.fc1, dec.conv1t   dense tcgen05 GEMMs (45-wide operands zero-padded to 64 / 96)
  dec.conv2t-4t    forward = 4-phase tap-GEMM / halo kernel (conv3t, conv4t); dgrad = tap-GEMM over the s2d form of the
                   output gradient; wgrad = wg_s2d
  dec.conv5t       forward fused with sigmoid + Laplace log-likelihood + dLoss/dlogit in x2 block form (convt_recon);
                   dgrad = c3conv over those blocks, wgrad = tap4_wg
  enc.conv5 out .. dec.conv1t out   fused dense chain (csrc/chain.cu): heads, latent stage, fc1, conv1t and their backward,
                   one launch each way
Weight gradients run on two side streams, bias gradients (column sums) on a third, the bulk of Adam (or of the
data-parallel exchange + Adam) on a fourth; packed bf16 weight operands are refreshed from the fp32 master parameters at
the start of every step (one launch).  Scheduling choices are constructor options, not environment switches.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib
from ._lib import ACT_ACCUMULATE, ACT_NONE, ACT_RELU, ACT_SIGMOID, MASK_S2D, OUT_S2D, TAP_HALO, Geom, ptr
from .engine import DEC_LAYERS, ENC_LAYERS, HEAD_LAYERS, Engine, _stream, make_geom, out_shape

BF16 = torch.bfloat16
_ENC = {lay[0]: lay for lay in ENC_LAYERS}
_DEC = {lay[0]: lay for lay in DEC_LAYERS}
TC_ENC = ["enc.conv2", "enc.conv3", "enc.conv4", "enc.conv5"]
TC_DEC = ["dec.conv2t", "dec.conv3t", "dec.conv4t"]
S2D_LAYERS = ["enc.conv2", "enc.conv3", "enc.conv4", "dec.conv2t", "dec.conv3t", "dec.conv4t"]   # k4/s2/p1, C_L >= 32
# tensors stored in s2d block form when the engine runs in s2d mode: the L operands of the layers above
S2D_TENSORS = ["enc.conv1.out", "enc.conv2.out", "enc.conv3.out", "dec.conv4t.dout", "dec.conv3t.dout", "dec.conv2t.dout"]


class EngineTC(Engine):
    precision = "bf16"

    def __init__(self, store, fused_chain=True, wgrad_streams=2, post_chain_stream="side", markers=0,
                 wgrad_plan="201202", dec_wgrad_plan="00000"):
        super().__init__(store)
        # scheduling of the weight-gradient kernels (they feed only the optimiser): the encoder's alternate between
        # `wgrad_streams` side streams so that a layer's weight gradient starts when its operand is ready instead of
        # queueing behind the previous layer's; the small launches that follow the fused chain kernel (fc1 / heads
        # weight gradients, gate backward) go to `post_chain_stream` ("side" = the weight-gradient stream, "side2" =
        # the bias-gradient stream).  Same-box A/B, ms per sup+unsup pair (profiles/r02_ab_log.txt): 1 stream / side
        # 1.344, 2 streams / side 1.336, 2 streams / side2 1.351, 1 stream / side2 1.375
        # which weight-gradient lane (0, 1, 2 = three side streams) takes: the post-chain launches, conv5, conv4, conv3,
        # conv2, conv1 of the encoder backward (decoder weight gradients: lane 0).  After the fused chain kernel the encoder's
        # backward is bound by the weight-gradient streams: with everything on two lanes ("001010") the three small
        # post-chain launches (fc1 / heads weight gradients, gate backward: ~35 us of latency) sat in front of conv5's weight
        # gradient and the chain conv5 -> conv3 -> conv1 ended 70 us after the last dgrad; on their own lane the step is
        # 3 % shorter (profiles/r02_ab_log.txt: 1.304 -> 1.263 ms per pair; "101010" 1.279, "201201" / "201002" 1.264)
        # L -> S layers over s2d blocks (conv2-4 forward, convT dgrads): two column-shifted boxes with one halo row instead
        # of four shifted boxes where the geometry allows it (16x16 outputs: conv2 forward, conv4t dgrad).  Same-box A/B,
        # ms per sup+unsup pair (profiles/r02_ab_log.txt): 1.2569 / 1.2503 against 1.2756 / 1.2752 with four boxes
        self.tap_flag = TAP_HALO
        self.wgrad_plan = [int(c) for c in str(wgrad_plan).zfill(6)]
        self.dec_wgrad_plan = [int(c) for c in str(dec_wgrad_plan).zfill(5)]     # lanes of conv5t, conv4t, conv3t, conv2t, conv1t
        self.wg_lanes = [None, torch.cuda.Stream(device=store.device), torch.cuda.Stream(device=store.device)]
        self._lanes_used = set()
        self.wgrad_streams = int(wgrad_streams)
        self.post_chain_stream = post_chain_stream
        # conv5 -> heads -> latent -> fc1 -> conv1t (and the reverse) as ONE launch each way (csrc/chain.cu); False keeps
        # the layer-by-layer kernels (A/B runs, cross-check in tests/test_gpu_chain.py)
        self.chain = bool(fused_chain)
        dev = self.device
        lib = self.lib
        z16 = lambda *shape: torch.zeros(*shape, dtype=BF16, device=dev)
        self.wp = {}
        for name in TC_ENC + TC_DEC + ["dec.conv5t"]:
            lay = _ENC.get(name) or _DEC[name]
            g = make_geom(lay, 1)
            self.wp[name + ".ls"] = z16(lib.gccvae_packed_weight_elems(C.byref(g), 0))
            self.wp[name + ".sl"] = z16(lib.gccvae_packed_weight_elems(C.byref(g), 1))
        # layers whose S->L direction runs on the halo kernel get the "sl9" packing as well
        self.halo = {}
        for name in TC_ENC + TC_DEC + ["dec.conv5t"]:
            g = make_geom(_ENC.get(name) or _DEC[name], 1)
            if lib.gccvae_sl_halo_supported(C.byref(g)):
                self.halo[name] = True
                self.wp[name + ".sl9"] = z16(lib.gccvae_packed_weight_elems(C.byref(g), 2))
        # x2 (space-to-depth) operands of the 3-channel end layers
        self.wp["enc.conv1.x2"] = z16(32 * 64)       # [cs][(a,b)][(dy,dx,c4)]
        self.wp["dec.conv5t.x2"] = z16(32 * 64)      # same packing: B operand of conv5t's dgrad
        self.wp["dec.conv5t.x2t"] = z16(16 * 128)    # [(dy,dx,c4)][(a,b)][cs]: fused conv5t forward
        self.x2 = True     # 3-channel tensors in x2 block form
        # s2d storage of the L tensors of the six k4/s2/p1 layers in the middle (include/gccvae.h, GCCVAE_OUT_S2D)
        self.s2d = True
        for name in S2D_LAYERS:
            _, _, (HL, WL, CL), (HS, WS, CS), k, s_, p_, _ = (_ENC.get(name) or _DEC[name])
            self.wp[name + ".s2d"] = z16(((CS + 15) // 16 * 16) * 16 * CL)
        # 45-wide dense layers, zero-padded to tensor-core widths (pad regions stay zero forever)
        self.wp["heads.ls"] = z16(96, 256)       # rows 0..44 = W_loc^T, 48..92 = W_std^T
        self.wp["heads.sl"] = z16(256, 96)
        self.wp["heads.bias"] = torch.zeros(96, dtype=torch.float32, device=dev)
        self.wp["fc1.ls"] = z16(64, 64)
        self.wp["fc1.sl"] = z16(64, 64)
        self.wp["conv1t.sl"] = z16(2048, 64)
        self.wp["conv1t.ls"] = z16(64, 2048)
        self._jobs = None
        # bias gradients: a separate bandwidth-bound column-sum pass per layer on its own stream.  Fusing them into the
        # dgrad epilogue (registers -> occupancy) or into the wgrad main loop (the stage release waits for the sums) was
        # measured slower on B200 in both rounds (profiles/r01d_ab_log.txt, r02_ab_log.txt); those options are gone.
        # Weight gradients are off the critical path (only Adam needs them): side streams, parallel graph branches.
        self.side = torch.cuda.Stream(device=dev)
        self.side2 = torch.cuda.Stream(device=dev)
        self._deferred_bias = []
        self.prof = None   # list of (op, start event, end event, algorithmic bytes) while profiling
        # called once per backward pass when every gradient except the first layer's is complete or queued: the
        # Learner hangs the bulk of the Adam update here, so that only the first layer's update follows the last dgrad
        # True while a step is issued whose image blocks b["X2"] were produced by the caller (Learner's graph replay does
        # the x2 transform on the copy stream, one step ahead)
        self.x2_ready = False
        self.tail_hook = None
        self.tail_hook_layer = TC_ENC[0]   # ... called when THIS layer's weight gradient has been issued (its dgrad follows)
        self.side3 = None          # its own stream: the first layer's weight / bias gradients must not queue behind it
        self._side3_used = False
        # debug timeline (markers=1: a globaltimer marker kernel after every op, 2: only at segment ends)
        self.mark_level = int(markers)
        self.mark_buf = torch.zeros(1024, dtype=torch.int64, device=dev) if self.mark_level else None
        self.marks = []

    # ---- packed weights ---------------------------------------------------------------------------------
    def pack_weights(self, part=None):
        """refresh every packed bf16 operand from the fp32 master weights: one kernel launch - or two (`part` 0: the
        first layer's operand, which is all conv1's forward waits for; `part` 1: the rest, under conv1's forward)."""
        if self._jobs is None:
            v = self.store.view
            jobs = []
            J = lambda kind, taps, CL, CS, W, out, sr=0, sk=0, ld=0, ro=0, co=0: jobs.append(
                _lib.PackJob(kind, taps, CL, CS, ptr(W), ptr(out), sr, sk, ld, ro, co, 0))
            J(7, 16, 3, 32, v("enc.conv1.w"), self.wp["enc.conv1.x2"])       # job 0: see `part`
            for name in TC_ENC + TC_DEC:
                lay = _ENC.get(name) or _DEC[name]
                _, _, (HL, WL, CL), (HS, WS, CS), k, s_, p_, _ = lay
                if name not in S2D_LAYERS:     # the s2d layers use the kind-9 operand instead
                    J(0, k * k, CL, CS, v(name + ".w"), self.wp[name + ".ls"])
                J(2 if (HS == 1 and WS == 1) else 1, k * k, CL, CS, v(name + ".w"), self.wp[name + ".sl"])
            J(1, 16, 3, 32, v("dec.conv5t.w"), self.wp["dec.conv5t.sl"])
            for name in self.halo:
                _, _, (HL, WL, CL), (HS, WS, CS), k, s_, p_, _ = (_ENC.get(name) or _DEC[name])
                J(6, 16, CL, CS, v(name + ".w"), self.wp[name + ".sl9"])
            for name in S2D_LAYERS:
                _, _, (HL, WL, CL), (HS, WS, CS), k, s_, p_, _ = (_ENC.get(name) or _DEC[name])
                J(9, 16, CL, CS, v(name + ".w"), self.wp[name + ".s2d"])
            J(7, 16, 3, 32, v("dec.conv5t.w"), self.wp["dec.conv5t.x2"])
            J(8, 16, 3, 32, v("dec.conv5t.w"), self.wp["dec.conv5t.x2t"])
            # kind 4/5: out[(ro + r) * ld + co + k] = W[r * sr + k * sk],  r < taps(R), k < CL(K)
            for off, nm in ((0, "enc.locs"), (48, "enc.std")):
                J(4, 45, 256, 0, v(nm + ".w"), self.wp["heads.ls"], 1, 45, 256, off, 0)
                J(4, 256, 45, 0, v(nm + ".w"), self.wp["heads.sl"], 45, 1, 96, 0, off)
                J(5, 1, 45, 0, v(nm + ".b"), self.wp["heads.bias"], 0, 1, 96, 0, off)
            J(4, 45, 45, 0, v("dec.fc1.w"), self.wp["fc1.ls"], 1, 45, 64)
            J(4, 45, 45, 0, v("dec.fc1.w"), self.wp["fc1.sl"], 45, 1, 64)
            J(4, 2048, 45, 0, v("dec.conv1t.w"), self.wp["conv1t.sl"], 45, 1, 64)
            J(4, 45, 2048, 0, v("dec.conv1t.w"), self.wp["conv1t.ls"], 1, 45, 2048)
            self._jobs = (_lib.PackJob * len(jobs))(*jobs)
            self._jobs_rest = (_lib.PackJob * (len(jobs) - 1))(*jobs[1:])
        if part is None:
            self._run("pack_weights", (), lambda: self.lib.gccvae_pack_jobs_bf16(self._jobs, len(self._jobs), _stream()))
        elif part == 0:
            self._run("pack_weights", (), lambda: self.lib.gccvae_pack_jobs_bf16(self._jobs, 1, _stream()))
        else:
            self._run("pack_weights", (), lambda: self.lib.gccvae_pack_jobs_bf16(self._jobs_rest, len(self._jobs_rest), _stream()))

    # ---- buffers -----------------------------------------------------------------------------------------
    def _alloc(self, B):
        dev = self.device
        e = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)
        b = {}
        # input image in x2 block form [B,33,33,16] bf16, followed (same allocation, so that the graph variants' private
        # copies carry both) by the raw bytes of the blocks [B,33,33,16] uint8 that prep_x2 writes for uint8 images
        b["X2"] = e(B * 33 * 33 * 24, dt=BF16)
        b["D2"] = e(B, 33, 33, 16, dt=BF16)      # dLoss/dlogit of the reconstruction in x2 block form
        b["xhat3"] = None                        # fp32 reconstruction, allocated on demand (tests / API)
        for name in ["enc.conv1", "enc.conv2", "enc.conv3", "enc.conv4", "enc.conv5"]:
            oh, ow, oc = out_shape(_ENC[name])
            b[name + ".out"] = e(B, oh, ow, oc, dt=BF16)
            b[name + ".dout"] = e(B, oh, ow, oc, dt=BF16)
        b["pre96"] = e(B, 96)                    # heads' pre-activations: locs at cols 0..44, std at 48..92
        b["dpre16"] = e(B, 96, dt=BF16)
        b["z16"] = e(B, 64, dt=BF16)
        b["dz64"] = e(B, 64)
        b["dec.fc1.out"] = e(B, 64, dt=BF16)     # 45 real channels
        b["dec.fc1.dout"] = e(B, 64, dt=BF16)
        for name in ["dec.conv1t"] + TC_DEC:
            oh, ow, oc = out_shape(_DEC[name])
            b[name + ".out"] = e(B, oh, ow, oc, dt=BF16)
            b[name + ".dout"] = e(B, oh, ow, oc, dt=BF16)
        b["xhat4"] = None
        for tname in S2D_TENSORS:
            Bq, H, W, Cc = b[tname].shape
            b[tname] = e(B, H // 2 + 1, W // 2 + 1, 4 * Cc, dt=BF16)   # zero borders are never written
        return b

    def dec_bufs(self, rows):
        """forward-only decoder buffers for `rows` latent rows (importance-weighted likelihood): the z16 operand and the
        bf16 activations of fc1 .. conv4t, about 92 KB per row - a fraction of `bufs`, which also holds the encoder's
        tensors and every gradient."""
        b = self._dec_bufs.get(rows)
        if b is None:
            b = {"z16": torch.zeros(rows, 64, dtype=BF16, device=self.device),
                 "dec.fc1.out": torch.zeros(rows, 64, dtype=BF16, device=self.device)}
            for name in ["dec.conv1t"] + TC_DEC:
                b[name + ".out"] = torch.empty(rows, *out_shape(_DEC[name]), dtype=BF16, device=self.device)
            self._dec_bufs[rows] = b
        return b

    def _xhat4(self, b, B):
        if b["xhat4"] is None:     # only the stand-alone Decoder(z) call needs it in x2 mode
            b["xhat4"] = torch.zeros(B, 64, 64, 4, dtype=torch.float32, device=self.device)
        return b["xhat4"]

    def latent_io(self, b):
        pre, g_ = b["pre96"], self.store.g
        return dict(loc_pre=ptr(pre), scale_pre=ptr(pre) + 48 * 4, ld_pre=96, z16=ptr(b["z16"]), dz=ptr(b["dz64"]),
                    ld_dz=64, dloc_pre=None, dscale_pre=None, dpre16=ptr(b["dpre16"]), db_loc=ptr(g_("enc.locs.b")),
                    db_scale=ptr(g_("enc.std.b")))

    def chain_io(self, b):
        """buffers and packed operands the fused chain kernels (gccvae_chain_fwd / _bwd) read and write."""
        v, g_, wp = self.store.view, self.store.g, self.wp
        return dict(h5=b["enc.conv5.out"], pre=b["pre96"], z16=b["z16"], g0=b["dec.fc1.out"], g1=b["dec.conv1t.out"],
                    dg1=b["dec.conv1t.dout"], dg0=b["dec.fc1.dout"], dpre16=b["dpre16"], dh5=b["enc.conv5.dout"],
                    w_heads=wp["heads.ls"], b_heads=wp["heads.bias"], w_fc1=wp["fc1.ls"], b_fc1=v("dec.fc1.b"),
                    w_conv1t=wp["conv1t.sl"], b_conv1t=v("dec.conv1t.b"), w_conv1t_t=wp["conv1t.ls"],
                    w_fc1_t=wp["fc1.sl"], w_heads_t=wp["heads.sl"], db_loc=g_("enc.locs.b"), db_scale=g_("enc.std.b"),
                    db_fc1=g_("dec.fc1.b"), db_conv1t=g_("dec.conv1t.b"), db_conv5=g_("enc.conv5.b"))

    # ---- helpers --------------------------------------------------------------------------------------------
    def _run(self, what, tensors, rc_fn):
        """issue one C-ABI call; with self.prof set, bracket it with CUDA events on the launching stream and
        record (duration, bytes of the tensors it reads/writes = its algorithmic HBM traffic)."""
        if self.prof is None:
            _lib.check(rc_fn(), what)
            if self.mark_level == 1:
                self.mark(what)
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(rc_fn(), what)
        e1.record()
        nbytes = sum(t.numel() * t.element_size() for t in tensors if t is not None)
        self.prof.append((what, e0, e1, nbytes))

    def mark(self, what, coarse=False):
        if self.mark_buf is None or (self.mark_level == 2 and not coarse) or len(self.marks) >= 1024:
            return
        st = torch.cuda.current_stream()
        lane = ("side" if st == self.side else "side2" if st == self.side2 else
                "side3" if (self.side3 is not None and st == self.side3) else
                "wg1" if st == self.wg_lanes[1] else "wg2" if st == self.wg_lanes[2] else "main")
        _lib.check(self.lib.gccvae_debug_mark(ptr(self.mark_buf), len(self.marks), _stream()), "mark")
        self.marks.append((what, lane))

    def _sl(self, name, geom, S, bias, act, mask, L, out_f32, what, mask_s2d=False):
        """S -> L of layer `name` (convT forward / conv dgrad): halo kernel where the geometry allows it."""
        st = _stream()
        if mask_s2d:
            act = act | MASK_S2D
        if name in self.halo:
            W = self.wp[name + ".sl9"]
            self._run(what, (S, mask, L), lambda: self.lib.gccvae_sl_halo_bf16(
                C.byref(geom), ptr(S), ptr(W), ptr(bias), act, ptr(mask), ptr(L), out_f32, st))
        else:
            W = self.wp[name + ".sl"]
            self._run(what, (S, W, mask, L), lambda: self.lib.gccvae_sl_bf16(
                C.byref(geom), ptr(S), ptr(W), ptr(bias), act, ptr(mask), ptr(L), out_f32, st))

    def _gemm(self, rows, K, N, A, Wp, bias, bias_n, bias_mod, act, mask, out, out_f32, what):
        self._run(what, (A, Wp, mask, out), lambda: self.lib.gccvae_gemm_bf16(
            rows, K, N, ptr(A), ptr(Wp), ptr(bias), bias_n, bias_mod, act, ptr(mask), ptr(out), out_f32, _stream()))

    def _gemm_tn(self, rows, M, N, A, Bm, segs, m_valid, what):
        o = _lib.WgOut()
        o.n_seg, o.m_valid = len(segs), m_valid
        for i, (col0, ncols, ld, dst) in enumerate(segs):
            o.seg[i] = _lib.WgSeg(col0, ncols, ld, 0, ptr(dst))
        self._run(what, (A, Bm) + tuple(sg[3] for sg in segs), lambda: self.lib.gccvae_gemm_tn_bf16(
            rows, M, N, ptr(A), ptr(Bm), C.byref(o), _stream()))

    def _bias_grad16(self, dout, name, cols=None, n_valid=0):
        cols = cols or dout.shape[-1]
        rows = dout.numel() // cols
        self._run(name + " bgrad", (dout,), lambda: self.lib.gccvae_colsum_bf16(
            ptr(dout), rows, cols, n_valid, ptr(self.store.g(name + ".b")), _stream()))

    def _flush_deferred_bias(self):
        if not self._deferred_bias:
            return
        def run():
            for dout, name, n in self._deferred_bias:
                cols = dout.shape[-1]
                if cols == 4 * n:        # s2d tensor: four slots of n channels per block (empty slots are zero)
                    cols = n
                self._bias_grad16(dout, name, cols=cols, n_valid=n if n < cols else 0)
        self._on_side2(run)
        self._deferred_bias = []

    def _on_side2(self, fn):
        if self.side2 is None or self.side is None:
            fn()
            return
        self.side2.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.side2):
            fn()

    def _lane(self, k):
        """weight-gradient lane k: 0 = self.side, 1 / 2 = further streams (created on first use, joined by join_side)."""
        if k == 0 or self.wgrad_streams <= 1:
            return self.side
        if self.wg_lanes[k] is None:
            self.wg_lanes[k] = torch.cuda.Stream(device=self.device)
        self._lanes_used.add(k)      # (only lanes that carry work of THIS step may be waited for inside a capture)
        return self.wg_lanes[k]

    def _side(self, fn, lane=0):
        """run fn (weight-gradient launches) on a side stream, after everything issued so far on the main one."""
        if self.side is None:
            fn()
            self._flush_deferred_bias()
            return
        side = self._lane(lane)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        self._flush_deferred_bias()      # column-sum passes requested by fn's _bias

    def join_side(self):
        if self.side is not None:
            torch.cuda.current_stream().wait_stream(self.side)
            if self.side2 is not None:
                torch.cuda.current_stream().wait_stream(self.side2)
            if self._side3_used:
                torch.cuda.current_stream().wait_stream(self.side3)
                self._side3_used = False
            for k in sorted(self._lanes_used):
                torch.cuda.current_stream().wait_stream(self.wg_lanes[k])
            self._lanes_used.clear()

    def _bias(self, name, n, dout):
        """bias gradient of `name` = column sums of its pre-activation gradient `dout`: queued for the bias-gradient
        stream (flushed by _side) unless the fused chain kernel produces it."""
        if name in getattr(self, "_chain_bias", ()):
            return
        self._deferred_bias.append((dout, name, n))

    def zero_grads(self):
        self.store.grad.zero_()   # the tensor-core wgrad / bias-grad kernels accumulate (split-K red.global)

    # ---- forward -----------------------------------------------------------------------------------------------
    def begin_step(self, x, b, log_pxz=None):
        """Work that depends only on the inputs and the parameters - packing the bf16 weight operands, the x2 block
        transform of the image, pre-setting log_pxz - forked onto the two side streams, so that it overlaps the
        gradient memset and the gate kernel on the main stream (parallel branches of the captured graph)."""
        self._begun = False
        if self.side is None:       # (profile_step issues everything serially)
            return
        B = x.shape[0]
        main = torch.cuda.current_stream()
        self.side.wait_stream(main)
        with torch.cuda.stream(self.side):
            self.pack_weights(part=0)
            self._ev_pack0 = torch.cuda.Event()
            self._ev_pack0.record(self.side)
            self.pack_weights(part=1)
        self.side2.wait_stream(main)
        with torch.cuda.stream(self.side2):
            u8 = int(x.dtype == torch.uint8)
            if not self.x2_ready:     # (a replayed step gets its image blocks from the copy stream, ahead of the replay)
                self._run("prep_x2", (x, b["X2"]), lambda: self.prep_x2(x, b["X2"], _stream()))
            if log_pxz is not None:
                _lib.check(self.lib.gccvae_fill_f32(ptr(log_pxz), B, -12288.0 * 0.6931471805599453, _stream()), "fill")
        self._begun = True
        self._log_pxz_ready = log_pxz is not None

    @staticmethod
    def xb_ptr(x2, B):
        """address of the raw-byte blocks behind the B x 1089 bf16 blocks of an X2 buffer"""
        return ptr(x2) + B * 1089 * 32

    def prep_x2(self, x, x2, stream):
        """image [B,64,64,3] (fp32 or uint8) -> x2 blocks (+ raw-byte blocks for uint8 images) in the buffer `x2`"""
        B, u8 = x.shape[0], int(x.dtype == torch.uint8)
        return self.lib.gccvae_prep_x2_bf16(ptr(x), u8, B, ptr(x2), self.xb_ptr(x2, B) if u8 else None, stream)

    def encoder_fwd(self, x, b, heads=True, blocks_ready=False):
        """`blocks_ready`: b["X2"] already holds the image blocks (image completion writes them in place), x only gives
        the batch size: no prep_x2."""
        B = x.shape[0]
        lib, st, v = self.lib, _stream(), self.store.view
        begun, self._begun = getattr(self, "_begun", False), False
        if begun:      # conv1 needs the image blocks and its own operand; the other operands land under its forward
            main = torch.cuda.current_stream()
            main.wait_event(self._ev_pack0)
            main.wait_stream(self.side2)
        else:
            self._log_pxz_ready = False
            self.pack_weights()
            if not (self.x2_ready or blocks_ready):
                self._run("prep_x2", (x, b["X2"]), lambda: self.prep_x2(x, b["X2"], st))
        self._run("enc.conv1 fwd", (b["X2"][:B * 1089 * 16], b["enc.conv1.out"]), lambda: lib.gccvae_c3conv_bf16(
            B, ptr(b["X2"]), ptr(self.wp["enc.conv1.x2"]), 32, ptr(v("enc.conv1.b")), ACT_RELU | OUT_S2D, None,
            ptr(b["enc.conv1.out"]), st))
        if begun:
            self.join_side()
        h = b["enc.conv1.out"]
        for name in TC_ENC:
            if name in S2D_LAYERS:
                # L operand in s2d block form: 2x2 taps of 4 C_L channels; the output is stored in s2d form when the
                # next layer is a stride-2 layer too
                _, _, (HL, WL, CL), (HS, WS, CS), k_, s_, p_, _ = _ENC[name]
                flag = OUT_S2D if (name + ".out") in S2D_TENSORS else 0
                self._run(name + " fwd", (h, self.wp[name + ".s2d"], b[name + ".out"]),
                          lambda h=h, name=name, HS=HS, WS=WS, CL=CL, CS=CS, flag=flag: lib.gccvae_tap4_ls_bf16(
                              B, HS + 1, WS + 1, 4 * CL, ptr(h), ptr(self.wp[name + ".s2d"]), CS, ptr(v(name + ".b")),
                              ACT_RELU | flag | self.tap_flag, None, ptr(b[name + ".out"]), st))
            else:
                g = make_geom(_ENC[name], B)
                self._run(name + " fwd", (h, self.wp[name + ".ls"], b[name + ".out"]),
                          lambda g=g, h=h, name=name: lib.gccvae_ls_bf16(
                              C.byref(g), ptr(h), ptr(self.wp[name + ".ls"]), ptr(v(name + ".b")), ACT_RELU, None,
                              ptr(b[name + ".out"]), 0, st))
            h = b[name + ".out"]
        if heads:      # (inside the ELBO step the fused chain kernel computes them)
            self._gemm(B, 256, 96, h, self.wp["heads.ls"], self.wp["heads.bias"], 96, 0, ACT_NONE, None, b["pre96"], 1,
                       "enc.heads fwd")
        return b["pre96"][:, 0:45], b["pre96"][:, 48:93]

    def decoder_fwd(self, z, b, z16_ready=False, fused_recon=False, batch=None, head=True):
        B = z.shape[0] if batch is None else batch
        lib, st, v = self.lib, _stream(), self.store.view
        if not z16_ready:          # standalone Decoder(z) call; inside the step the latent stage writes z16
            b["z16"][:, :45].copy_(z)
        if head:                   # (inside the ELBO step the fused chain kernel has produced dec.conv1t.out)
            self._gemm(B, 64, 64, b["z16"], self.wp["fc1.ls"], v("dec.fc1.b"), 45, 0, ACT_RELU, None, b["dec.fc1.out"], 0,
                       "dec.fc1 fwd")
            self._gemm(B, 64, 2048, b["dec.fc1.out"], self.wp["conv1t.sl"], v("dec.conv1t.b"), 2048, 128, ACT_RELU, None,
                       b["dec.conv1t.out"], 0, "dec.conv1t fwd")
        h = b["dec.conv1t.out"]
        for name in TC_DEC:
            g = make_geom(_DEC[name], B)
            self._sl(name, g, h, v(name + ".b"), ACT_RELU, None, b[name + ".out"], 0, name + " fwd")
            h = b[name + ".out"]
        if fused_recon:            # conv5t runs fused with the likelihood (decoder_fwd_recon)
            return None
        g = make_geom(_DEC["dec.conv5t"], B)
        xh4 = self._xhat4(b, B)
        self._sl("dec.conv5t", g, h, v("dec.conv5t.b"), ACT_SIGMOID, None, xh4, 2, "dec.conv5t fwd")
        return xh4[..., :3]

    def decoder_fwd_recon(self, x, b, coef, log_pxz, backward, want_recon, head=True):
        """decoder forward with conv5t + sigmoid + Laplace log-likelihood (+ dLoss/dlogit in x2 block form) fused."""
        B = x.shape[0]
        self.decoder_fwd(None, b, z16_ready=True, fused_recon=True, batch=B, head=head)
        xhat = None
        if want_recon:
            if b["xhat3"] is None:
                b["xhat3"] = torch.zeros(B, 64, 64, 3, dtype=torch.float32, device=self.device)
            xhat = b["xhat3"]
        u8 = int(x.dtype == torch.uint8)
        v = self.store.view
        self._run("dec.conv5t fwd+recon", (b["dec.conv4t.out"], x, b["D2"] if backward else None),
                  lambda: self.lib.gccvae_convt_recon_bf16(
                      B, ptr(b["dec.conv4t.out"]), ptr(self.wp["dec.conv5t.x2t"]), ptr(v("dec.conv5t.b")),
                      self.xb_ptr(b["X2"], B) if u8 else ptr(x), 2 * u8,    # uint8 images: the raw-byte blocks prep_x2 wrote
                      ptr(coef) if backward else None, ptr(log_pxz), ptr(b["D2"]) if backward else None, ptr(xhat),
                      ptr(self.store.g("dec.conv5t.b")) if backward else None, int(getattr(self, "_log_pxz_ready", False)),
                      _stream()))
        self._log_pxz_ready = False
        return xhat

    def image_fwd(self, z, b, batch, out_u8, out=None):
        """generation path: the decoder from the z16 operand the latent kernel wrote, conv5t + sigmoid straight into a
        fresh [B,64,64,3] image (gccvae_convt_image_bf16): fp32, or uint8 min(255, rint(255 xhat)).  `out`: a contiguous
        [batch,64,64,3] tensor of that dtype to write instead (a row slice of a larger image tensor: rows are 12 or 48 KB,
        so every slice keeps the kernel's 16-byte alignment); b (`bufs` or `dec_bufs`) may hold more rows than `batch`."""
        self.decoder_fwd(None, b, z16_ready=True, fused_recon=True, batch=batch, head=True)
        if out is None:
            out = torch.empty(batch, 64, 64, 3, dtype=torch.uint8 if out_u8 else torch.float32, device=self.device)
        g4 = b["dec.conv4t.out"]
        self._run("dec.conv5t fwd image", (g4, out), lambda: self.lib.gccvae_convt_image_bf16(
            batch, ptr(g4), ptr(self.wp["dec.conv5t.x2t"]), ptr(self.store.view("dec.conv5t.b")), ptr(out), int(out_u8),
            _stream()))
        return out

    def complete_begin(self, x, mask):
        """per-call state of image completion: the pixel mask [B,64,64] bool (True = observed) in x2 block form,
        [B,33,33] uint8 with bit dy * 2 + dx of block (i, j) set when pixel (2i-1+dy, 2j-1+dx) is observed; pixels outside
        the image count as observed."""
        B = mask.shape[0]
        m = torch.nn.functional.pad(mask.to(torch.uint8), (1, 1, 1, 1), value=1)        # [B,66,66]
        m = m.view(B, 33, 2, 33, 2).permute(0, 1, 3, 2, 4)                               # [B,33,33,dy,dx]
        bit = torch.tensor([[1, 2], [4, 8]], dtype=torch.uint8, device=self.device)
        return {"mask_blocks": (m * bit).sum((-2, -1), dtype=torch.uint8).contiguous()}

    def complete_fwd(self, z, b, batch, state, x):
        """one iteration of image completion: the decoder from the z16 operand the latent kernel wrote, then conv5t +
        sigmoid straight into the unobserved pixels of the encoder's input blocks b["X2"], in place
        (gccvae_convt_complete_bf16).  Returns x: the next encoder pass reads the blocks as they are (blocks_ready)."""
        self.decoder_fwd(None, b, z16_ready=True, fused_recon=True, batch=batch, head=True)
        g4, mb = b["dec.conv4t.out"], state["mask_blocks"]
        self._run("dec.conv5t fwd complete", (g4, mb), lambda: self.lib.gccvae_convt_complete_bf16(
            batch, ptr(g4), ptr(self.wp["dec.conv5t.x2t"]), ptr(self.store.view("dec.conv5t.b")), ptr(mb), ptr(b["X2"]),
            _stream()))
        return x

    def iw_decoder_ll(self, x, b, batch, kc, dec, log_pxz):
        """importance-weighted likelihood: the decoder over the batch * kc rows of dec["z16"], then conv5t + sigmoid +
        Laplace log-likelihood of row r against source image r / kc (gccvae_convt_ll_bf16) into log_pxz.  A uint8 image
        is read from the raw-byte blocks the encoder's prep_x2 wrote into b["X2"]: once per call, not once per sample."""
        rows = batch * kc
        self.decoder_fwd(None, dec, z16_ready=True, fused_recon=True, batch=rows, head=True)
        _lib.check(self.lib.gccvae_fill_f32(ptr(log_pxz), rows, -12288.0 * 0.6931471805599453, _stream()), "fill")
        u8 = int(x.dtype == torch.uint8)
        g4 = dec["dec.conv4t.out"]
        self._run("dec.conv5t fwd ll", (g4[:rows], x), lambda: self.lib.gccvae_convt_ll_bf16(
            rows, kc, ptr(g4), ptr(self.wp["dec.conv5t.x2t"]), ptr(self.store.view("dec.conv5t.b")),
            self.xb_ptr(b["X2"], batch) if u8 else ptr(x), 2 * u8, ptr(log_pxz), _stream()))

    # ---- backward -----------------------------------------------------------------------------------------------
    def decoder_bwd(self, z, b, want_dz=True, tail=True):
        """`tail=False`: stop after conv2t's dgrad (the fused chain kernel continues from dec.conv1t.dout)."""
        B = z.shape[0]
        lib, st, g_ = self.lib, _stream(), self.store.g
        self._chain_bias = set() if tail else {"dec.conv1t", "dec.fc1", "enc.conv5"}
        g4 = b["dec.conv4t.out"]
        # conv5t from the logit gradient in x2 block form (written by the fused forward)
        self._side(lambda: self._run("dec.conv5t wgrad", (b["D2"], g4), lambda: lib.gccvae_tap4_wg_bf16(
            B, ptr(b["D2"]), ptr(g4), 32, ptr(g_("dec.conv5t.w")), None, _stream())), lane=self.dec_wgrad_plan[0])
        self._run("dec.conv5t dgrad", (b["D2"], g4, b["dec.conv4t.dout"]), lambda: lib.gccvae_c3conv_bf16(
            B, ptr(b["D2"]), ptr(self.wp["dec.conv5t.x2"]), 32, None, ACT_NONE | OUT_S2D, ptr(g4),
            ptr(b["dec.conv4t.dout"]), st))
        prev_of = {"dec.conv4t": "dec.conv3t", "dec.conv3t": "dec.conv2t", "dec.conv2t": "dec.conv1t"}
        for name in reversed(TC_DEC):
            dout, pn = b[name + ".dout"], prev_of[name]
            xin, dxin = b[pn + ".out"], b[pn + ".dout"]
            _, _, (HL, WL, CL), (HS, WS, CS), k_, s_, p_, _ = _DEC[name]
            def wg(name=name, dout=dout, xin=xin, HS=HS, WS=WS, CL=CL, CS=CS):
                self._bias(name, CL, dout)
                self._run(name + " wgrad", (dout, xin), lambda: lib.gccvae_wg_s2d_bf16(
                    B, HS, WS, CL, ptr(dout), ptr(xin), CS, ptr(g_(name + ".w")), _stream()))
            self._side(wg, lane=self.dec_wgrad_plan[{"dec.conv4t": 1, "dec.conv3t": 2, "dec.conv2t": 3}[name]])
            flag = OUT_S2D if (pn + ".dout") in S2D_TENSORS else 0
            self._run(name + " dgrad", (dout, self.wp[name + ".s2d"], xin, dxin),
                      lambda name=name, dout=dout, xin=xin, dxin=dxin, HS=HS, WS=WS, CL=CL, CS=CS, flag=flag:
                      lib.gccvae_tap4_ls_bf16(B, HS + 1, WS + 1, 4 * CL, ptr(dout), ptr(self.wp[name + ".s2d"]), CS, None,
                                              ACT_NONE | flag | self.tap_flag, ptr(xin), ptr(dxin), st))
        # conv1t ([B,64(45)] -> [B,2048]) and fc1 as padded dense GEMMs
        dg1, g0, dg0 = b["dec.conv1t.dout"], b["dec.fc1.out"], b["dec.fc1.dout"]
        self._side(lambda: self._gemm_tn(B, 2048, 64, dg1, g0, [(0, 45, 45, g_("dec.conv1t.w"))], 2048,
                                         "dec.conv1t wgrad"), lane=self.dec_wgrad_plan[4])
        if not tail:
            return None
        self._on_side2(lambda: self._bias_grad16(dg1, "dec.conv1t", cols=128))
        self._gemm(B, 2048, 64, dg1, self.wp["conv1t.ls"], None, 0, 0, ACT_NONE, g0, dg0, 0, "dec.conv1t dgrad")
        def wg_fc1():
            self._bias("dec.fc1", 45, dg0)
            self.fc1_wgrad(b, B)
        self._side(wg_fc1)
        if want_dz:
            self._gemm(B, 64, 64, dg0, self.wp["fc1.sl"], None, 0, 0, ACT_NONE, None, b["dz64"], 1, "dec.fc1 dgrad")
        return b["dz64"][:, :45]

    def heads_wgrad(self, b, B):
        """weight gradients of both [256,45] head kernels in one GEMM (bias gradients come from the latent stage)."""
        g_ = self.store.g
        self._gemm_tn(B, 256, 96, b["enc.conv5.out"], b["dpre16"],
                      [(0, 45, 45, g_("enc.locs.w")), (48, 45, 45, g_("enc.std.w"))], 256, "enc.heads wgrad")

    def fc1_wgrad(self, b, B):
        self._gemm_tn(B, 64, 64, b["z16"], b["dec.fc1.dout"], [(0, 45, 45, self.store.g("dec.fc1.w"))], 45, "dec.fc1 wgrad")

    def encoder_bwd(self, x, b, heads=True):
        """`heads=False`: enc.conv5.dout is already there (fused chain kernel), start at conv5's own backward."""
        B = x.shape[0]
        lib, st, g_ = self.lib, _stream(), self.store.g
        h5, dh5, dpre = b["enc.conv5.out"], b["enc.conv5.dout"], b["dpre16"]
        if heads:
            self._side(lambda: self.heads_wgrad(b, B))
            self._gemm(B, 96, 256, dpre, self.wp["heads.sl"], None, 0, 0, ACT_NONE, h5, dh5, 0, "enc.heads dgrad")
        prev_of = {"enc.conv5": "enc.conv4", "enc.conv4": "enc.conv3", "enc.conv3": "enc.conv2",
                   "enc.conv2": "enc.conv1"}
        for name in reversed(TC_ENC):
            geom = make_geom(_ENC[name], B)
            dout, pn = b[name + ".dout"], prev_of[name]
            xin, dxin = b[pn + ".out"], b[pn + ".dout"]
            s2d_l = name in S2D_LAYERS        # xin (L operand, and the ReLU mask of the dgrad) is s2d
            _, _, (HL, WL, CL), (HS, WS, CS), k_, s_, p_, _ = _ENC[name]
            def wg(name=name, geom=geom, dout=dout, xin=xin, s2d_l=s2d_l, HS=HS, WS=WS, CL=CL, CS=CS):
                self._bias(name, dout.shape[-1], dout)
                if s2d_l:
                    self._run(name + " wgrad", (xin, dout), lambda: lib.gccvae_wg_s2d_bf16(
                        B, HS, WS, CL, ptr(xin), ptr(dout), CS, ptr(g_(name + ".w")), _stream()))
                else:
                    self._run(name + " wgrad", (xin, dout), lambda: lib.gccvae_wg_bf16(
                        C.byref(geom), ptr(xin), ptr(dout), ptr(g_(name + ".w")), _stream()))
            self._side(wg, lane=self.wgrad_plan[{"enc.conv5": 1, "enc.conv4": 2, "enc.conv3": 3, "enc.conv2": 4}[name]])
            hook = self.tail_hook if name == self.tail_hook_layer else None
            ev = None
            if hook is not None and self.side is not None:
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream())     # everything the main stream has produced so far
            self._sl(name, geom, dout, None, ACT_NONE, xin, dxin, 0, name + " dgrad", mask_s2d=s2d_l)
            if hook is not None:
                self.tail_hook = None
                if ev is not None:     # under this dgrad: after all earlier weight / bias gradients, not after it
                    if self.side3 is None:
                        self.side3 = torch.cuda.Stream(device=self.device)
                    self.side3.wait_event(ev)
                    self.side3.wait_stream(self.side)
                    self.side3.wait_stream(self.side2)
                    for k in sorted(self._lanes_used):
                        self.side3.wait_stream(self.wg_lanes[k])
                    with torch.cuda.stream(self.side3):
                        hook()
                    self._side3_used = True
                else:
                    hook()
        dh1 = b["enc.conv1.dout"]
        def wg1():     # conv1's bias gradient comes out of the same launch (the ones slot of prep_x2's blocks)
            self._run("enc.conv1 wgrad", (b["X2"][:B * 1089 * 16], dh1), lambda: lib.gccvae_tap4_wg_bf16(
                B, ptr(b["X2"]), ptr(dh1), 32, ptr(g_("enc.conv1.w")), ptr(g_("enc.conv1.b")), _stream()))
        self._side(wg1, lane=self.wgrad_plan[5])
        self.join_side()

    # ---- per-op device timing (bench.py roofline) -------------------------------------------------------------
    def profile_step(self, learner, x, y, steps=3):
        """Run `steps` eager supervised+unsupervised train_steps with every tensor-core / data-movement op
        bracketed by CUDA events; returns {op: (mean ms per launch, launches per step, algorithmic bytes)}."""
        graphs, learner.use_graphs = learner.use_graphs, False
        side, self.side = self.side, None     # serial issue: per-op times are not inflated by stream overlap
        agg = {}
        # The host needs ~25 us per bracketed op (event records + ctypes call + tensor-map encoding), about what the kernels
        # take: without a head start the GPU idles between an op's first event and its launch, and the bracket measures
        # the host.  A spin kernel in front of every train_step lets the host enqueue the whole step first (torch's
        # cuda._sleep, ~5 ms); the events then see device time only.
        spin = int(5e-3 * 1.9e9)
        try:
            for _ in range(steps):
                self.prof = []
                torch.cuda._sleep(spin)
                learner.train_step(x, y, True)
                torch.cuda._sleep(spin)
                learner.train_step(x, None, False)
                torch.cuda.synchronize(self.device)
                for what, e0, e1, nbytes in self.prof:
                    a = agg.setdefault(what, [0.0, 0, nbytes])
                    a[0] += e0.elapsed_time(e1)
                    a[1] += 1
        finally:
            self.prof = None
            self.side = side
            learner.use_graphs = graphs
        return {k: (v[0] / v[1], v[1] / steps, v[2]) for k, v in agg.items()}
