"""Host-side mirror of the reference's CCVAE / Learner (gated_ccvae.py:23-311, 421-455) on top of the
sm_100a kernels.  Same class names, constructor arguments, method names and return conventions:

    learner = Learner(ip_shape, z_dim, z_classify, y_dim, num_samples, supervision, train_config)
    loss, c = learner.sup_loss(x, y)         # gated_ccvae.py:234-300
    loss, c = learner.unsup_loss(x)          # :184-232
    lqx     = learner.classifier_loss(x, y, c, k=100)   # :167-182
    loss, c = learner.train_step(x, y, supervised)      # :302-311  (fwd + bwd + Adam)
    acc     = learner.classifier_accuracy(x, y)         # :421-446
    img     = learner.generate(y) / .reconstruct(x) / .intervene(x, y_new)   # extension, see below
    ll      = learner.log_likelihood(x, y=None, k=100)                        # extension, see below

Extensions the reference lacks (for parity testing, data parallelism, image generation and likelihood evaluation):
  * every stochastic call takes an optional `noise=` dict of explicit draws
    (eps [B,45], eps_k [K,B,45], U_y [B,18], U1/U2 [18,18]); without it noise comes from an
    in-kernel Philox4x32-10 keyed by (seed, step counter);
  * `Learner.last` exposes every per-image term of the last loss call;
  * if torch.distributed is initialised the step is data parallel: the batch given to each rank is
    its shard, gradients are all-reduced (sum) over the flat gradient buffer, the loss is the global
    mean, and the gate sample c is identical on all ranks;
  * a forward-only generation path with no counterpart in the reference: `generate(y)` decodes target labels through
    the conditional prior, `reconstruct(x)` decodes an image's posterior, `intervene(x, y_new)` moves an image's classify
    dims to new labels by a Gaussian counterfactual; each returns a [B,64,64,3] fp32 or uint8 image on the device;
    `walk`, `swap`, `traverse` and `interpolate` decode frames along one label, between images or along one latent dim;
    `complete(x, mask, y_new)` fills in the unobserved pixels of images, optionally steered to target labels;
  * the importance-weighted (IWAE) log-likelihood with K samples: `log_likelihood(x)` bounds log p(x) and
    `log_likelihood(x, y)` bounds log p(x, y) per image (nats, tighter as K grows); `test_log_likelihood(loader)` is its
    `accuracy(loader)` counterpart.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import logging
import math
import os

import numpy as np
import torch

from . import _lib, dp
from ._lib import (GATE_WS_FLOATS, LATENT_PARTIAL_FLOATS, RESULT_SLOT_FLOATS, ChainBwdArgs, ChainFwdArgs, DpArgs,
                   GenLatentArgs, IwLatentArgs, LatentBwdArgs, LatentFwdArgs, ptr)
from .engine import Engine, _stream, image_u8
from .networks import Classifier, Conditional_Prior, Decoder, Encoder, _default_device, as_device_f32
from .params import ParamStore, keras_default_init
from .utils_data import gating_matrix_csv, load_learned_gating_matrix

logger = logging.getLogger(__name__)


class CCVAE:
    """gated_ccvae.py:23-111."""

    def __init__(self, z_dim, z_classify, y_dim, train_config, device=None, precision="fp32", init_seed=0,
                 engine_options=None):
        if (z_dim, z_classify, y_dim) != (45, 18, 18):
            raise ValueError("the sm_100a kernels are specialised for z_dim=45, z_classify=y_dim=18")
        self.z_dim = z_dim
        self.z_classify = z_classify
        self.z_style = z_dim - z_classify
        self.y_dim = y_dim
        self.device = torch.device(device) if device is not None else _default_device()
        self.store = ParamStore(self.device)
        keras_default_init(self.store, init_seed)
        self.engine = make_engine(self.store, precision, **(engine_options or {}))
        self.lib = self.engine.lib
        kw = dict(store=self.store, engine=self.engine)
        self.encoder = Encoder(z_dim, **kw)
        self.decoder = Decoder(hidden_dim=z_dim, **kw)
        self.classifier = Classifier(y_dim, **kw)
        self.cond_prior = Conditional_Prior(z_classify, **kw)
        self.initialise_mu(train_config)

    # gated_ccvae.py:42-60
    def initialise_mu(self, train_config):
        gt, gs = train_config["gate_type"], train_config.get("gate_subtype")
        if gt == "learnable":
            logging.info("Initialising mu with fixed value (learnable)")
            mu_init, self.mu_trainable = np.asarray(train_config["mu_init"]), True
        elif gt == "fixed" and gs == "inferred":
            logging.info("Initialising mu with fixed value")
            mu_init, self.mu_trainable = np.asarray(train_config["mu_init"]), False
        elif gt == "fixed" and gs == "one-one":
            mu_init, self.mu_trainable = np.eye(self.z_classify, self.y_dim), False
        else:
            raise ValueError("Invalid gate type/subtype: {}/{}".format(gt, gs))
        if mu_init.shape != (self.z_classify, self.y_dim):
            raise ValueError("mu_init must be [{}, {}], got {}".format(self.z_classify, self.y_dim, mu_init.shape))
        with torch.no_grad():
            self.store.view("mu").copy_(torch.from_numpy(mu_init.astype(np.float32)))

    @property
    def mu(self):
        return self.store.view("mu")

    @property
    def trainable_variables(self):
        names = [k for k in self.store.names() if k != "mu" or self.mu_trainable]
        return [self.store.view(k) for k in names]

    # gated_ccvae.py:90-93 (explicit noise instead of tf.random)
    def sample_normal(self, mu, std, latent_dim, epsilon=None):
        mu, std = as_device_f32(mu, self.device), as_device_f32(std, self.device)
        if epsilon is None:
            epsilon = torch.randn_like(std)
        return (mu + std * as_device_f32(epsilon, self.device)).reshape(-1, latent_dim)

    # gated_ccvae.py:102-111
    def sample_gating_parameter(self, mu, temperature, EPSILON=1e-20, U1=None, U2=None, seed=0, offset=0):
        if EPSILON != 1e-20:
            raise ValueError("the gate kernel hard-codes EPSILON=1e-20 (gated_ccvae.py:102)")
        mu = as_device_f32(mu, self.device)
        ws = torch.empty(GATE_WS_FLOATS, dtype=torch.float32, device=self.device)
        c = torch.empty(18, 18, dtype=torch.float32, device=self.device)
        U1 = None if U1 is None else as_device_f32(U1, self.device)
        U2 = None if U2 is None else as_device_f32(U2, self.device)
        v = self.store.view
        _lib.check(self.lib.gccvae_gate_fwd(ptr(mu), None, ptr(U1), ptr(U2), seed, offset, None, float(temperature), None,
                                            ptr(v("cls.w")), ptr(v("cls.b")), ptr(v("prior.loc_true")),
                                            ptr(v("prior.loc_false")), ptr(v("prior.scale_true")),
                                            ptr(v("prior.scale_false")), ptr(ws), ptr(c), _stream()), "gate_fwd")
        return c


def make_engine(store, precision, **options):
    if precision == "fp32":
        if options:
            raise ValueError("the fp32 engine has no options (got {})".format(sorted(options)))
        return Engine(store)
    if precision == "bf16":
        from .engine_tc import EngineTC
        return EngineTC(store, **options)
    raise ValueError("precision must be 'fp32' or 'bf16', got {!r}".format(precision))


class KerasAdam:
    """tf.keras.optimizers.Adam(lr) of Keras 2.8 (gated_ccvae.py:144): beta_1=.9, beta_2=.999,
    epsilon=1e-7 outside the sqrt; one fused kernel over the flat parameter buffer."""

    def __init__(self, lr, store, n_params, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        self.lr, self.beta_1, self.beta_2, self.epsilon = float(lr), beta_1, beta_2, epsilon
        self.store, self.n = store, n_params
        self.m = torch.zeros_like(store.flat)
        self.v = torch.zeros_like(store.flat)
        # {t, block ticket}: t lives on the device (the kernels key their Philox streams on it and a captured graph
        # of the step can be replayed); the update kernel itself advances it
        self.step_dev = torch.zeros(2, dtype=torch.int32, device=store.device)
        self.lib = _lib.load()

    @property
    def iterations(self):
        return int(self.step_dev[0].item())

    def apply_gradients(self, lo=0, hi=None, publish=True, result=None):
        """one launch: the Adam update of parameters [lo, hi) of the trainable prefix with t = iterations + 1, the
        gradient buffer cleared behind the read (the next backward pass accumulates into it), and - `publish` - the
        step counter advanced and `result` = (loss, c, ring) copied into ring[(t - 1) % len(ring)].  Returns True if the
        gradient buffer is clean afterwards."""
        n = self.n if hi is None else min(int(hi), self.n)
        zero_hi = self.store.total if hi is None else n
        loss, c, ring = result if (result is not None and publish) else (None, None, None)
        _lib.check(self.lib.gccvae_adam_fused_f32(ptr(self.store.flat), ptr(self.store.grad), ptr(self.m), ptr(self.v),
                                                  int(lo), n, zero_hi, self.lr, self.beta_1, self.beta_2, self.epsilon,
                                                  ptr(self.step_dev), int(bool(publish)), ptr(loss), ptr(c), ptr(ring),
                                                  0 if ring is None else int(ring.shape[0]), _stream()), "adam")
        return bool(publish)


class Learner:
    """gated_ccvae.py:114-311, 421-455."""

    def __init__(self, ip_shape, z_dim, z_classify, y_dim, num_samples, supervision, train_config, device=None,
                 precision="fp32", seed=1234, init_seed=0, graphs=False, adam_tail=True, engine_options=None,
                 dp_exchange="peer"):
        if tuple(ip_shape) != (64, 64, 3):
            raise ValueError("the kernels are specialised for 64x64x3 inputs (gated_ccvae.py:481)")
        self.train_config = train_config
        self.ip_shape = tuple(ip_shape)
        self.z_dim, self.z_classify, self.z_style, self.y_dim = z_dim, z_classify, z_dim - z_classify, y_dim
        self.supervision = supervision
        self.eps = 1e-20
        self.lr = train_config["lr"]
        self.alpha = 0.1 * num_samples
        self.latent_sampler_temp = train_config.get("init_temp", 0.1)
        self._temp_dev = None
        self.gating_sampler_temp = train_config["gating_init_temp"]
        self.model = CCVAE(z_dim, z_classify, y_dim, train_config, device=device, precision=precision,
                           init_seed=init_seed, engine_options=engine_options)
        self.device = self.model.device
        self.p_Y = torch.full((1, y_dim), 0.5, dtype=torch.float32, device=self.device)  # gated_ccvae.py:141
        self.store, self.engine, self.lib = self.model.store, self.model.engine, self.model.lib
        self.n_trainable = self.store.total if self.model.mu_trainable else self.store.n_without_mu
        self.optimiser = KerasAdam(self.lr, self.store, self.n_trainable)
        self.seed = int(seed)
        self.use_graphs = bool(graphs)   # replay the whole train_step as ONE CUDA graph (Philox-noise steps only)
        self._graphs = {}
        self._graph_turn = {}
        self._grads_clean = False        # True right after apply_gradients (it clears the gradient buffer)
        # single GPU, tensor-core engine: Adam runs in two parts - everything but the first layer's parameters as soon
        # as their gradients are complete (on a side stream, under the last dgrad), the first layer at the very end
        self._tail_layer = "enc.conv2"       # the head part starts when this layer's weight gradient has been issued
        self._adam_cut = self.store.offsets[self._tail_layer + ".w"][0]
        self._adam_head_done = False
        self.adam_tail = bool(adam_tail)
        # what train_step returns: the publishing Adam launch copies (loss, c) into slot (t - 1) % RING of this ring, so
        # the tensors handed back stay valid for RING further steps (the replayed graph always writes the same addresses)
        self.RING = 8
        self._ring = torch.zeros(self.RING, RESULT_SLOT_FLOATS, dtype=torch.float32, device=self.device)
        self._t_host = None              # host mirror of optimiser.step_dev[0]; read from the device on first use
        self._copy_stream = None
        self.last = {}
        self._lat = {}
        self._temp_dev = torch.full((1,), self._gating_sampler_temp, dtype=torch.float32, device=self.device)
        # Philox counter offset of the current call: 0 inside train_step (forward and backward regenerate the same noise
        # from the step counter); every forward-only call (sup_loss / unsup_loss / classifier_loss / classifier_accuracy)
        # takes a fresh one, so that e.g. the validation batches of accuracy() see different gate samples and noise,
        # as the reference's tf.random draws do
        self._noise_offset = 0
        self._eval_calls = 0
        self._gate_ws = torch.zeros(GATE_WS_FLOATS, dtype=torch.float32, device=self.device)
        self._c = torch.zeros(18, 18, dtype=torch.float32, device=self.device)
        self._loss = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._acc = torch.zeros(1, dtype=torch.float32, device=self.device)
        # data parallel
        self._dist = dp.dist_or_none()
        self.world, self.rank = dp.world_and_rank(self._dist)
        # gradient exchange: "peer" = two-shot all-reduce over NVLink peer memory fused with Adam (one kernel, inside
        # the step's graph); "nccl" = NCCL all-reduce between the replayed graph and the optimiser.  "peer" falls back
        # to "nccl" where symmetric memory cannot be set up (collectively: every rank takes the same path).
        if dp_exchange not in ("peer", "nccl"):
            raise ValueError("dp_exchange must be 'peer' or 'nccl', got {!r}".format(dp_exchange))
        self._peer = None
        if self.world > 1 and dp_exchange == "peer" and self.device.type == "cuda":
            # the bulk of the exchange (barrier, 4 MB over NVLink, barrier, Adam: ~45 us) needs more room than the last
            # dgrad gives it: it starts one layer earlier and leaves the first TWO layers' gradients to the closing call
            self._tail_layer = "enc.conv3"
            self._adam_cut = self.store.offsets[self._tail_layer + ".w"][0]
            self._peer = self._setup_peer_exchange()
            if self._peer is None:
                self._tail_layer = "enc.conv2"
                self._adam_cut = self.store.offsets[self._tail_layer + ".w"][0]

    def _setup_peer_exchange(self):
        peer, err = None, None
        try:
            peer = dp.PeerExchange(self._dist, self.store.total + 4, self.device, push_floats=self._adam_cut)
        except Exception as e:      # noqa: BLE001 - whatever goes wrong, the NCCL path still works
            err = e
        flag = torch.tensor([0 if peer is not None else 1], device=self.device)
        self._dist.all_reduce(flag)
        if int(flag.item()) != 0:
            if self.rank == 0:
                logger.warning("peer-memory gradient exchange unavailable (%s): using the NCCL all-reduce", err)
            return None
        self.store.adopt_grad_buffer(peer.grad)
        return peer

    def _peer_adam(self, lo, hi, zero_hi, publish, push=False):
        """rank barrier + two-shot all-reduce of grad[lo:hi) + Adam on it, one launch (csrc/dp.cu); `push`: the
        one-barrier variant for the short range that closes the step."""
        a, opt = self._peer.fill_args(DpArgs()), self.optimiser
        a.push = int(bool(push))
        a.param, a.m, a.v = ptr(self.store.flat), ptr(opt.m), ptr(opt.v)
        a.i0, a.n, a.n_zero = int(lo), int(hi), int(zero_hi)
        a.loss_index = self.store.total if publish else -1
        a.lr, a.beta1, a.beta2, a.eps = opt.lr, opt.beta_1, opt.beta_2, opt.epsilon
        a.step_state, a.publish = ptr(opt.step_dev), int(bool(publish))
        a.ring_slots, a.result_loss, a.result_c = self.RING, None, ptr(self._c)
        a.result_ring = ptr(self._ring) if publish else None
        _lib.check(self.lib.gccvae_dp_reduce_adam_f32(C.byref(a), _stream()), "dp_reduce_adam")

    # ---- buffers of the latent stage -------------------------------------------------------------------
    def _latent_bufs(self, B):
        lb = self._lat.get(B)
        if lb is None:
            e = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device=self.device)
            npart = (self.lib.gccvae_chain_partials(B) if getattr(self.engine, "chain", False)
                     else self.lib.gccvae_latent_bwd_partials(B))
            lb = dict(loc=e(B, 45), scale=e(B, 45), z=e(B, 45), terms=e(6, B), logits=e(B, 18),
                      y_i32=e(B, 18, dt=torch.int32), log_pxz=e(B), partials=e(npart + 1, LATENT_PARTIAL_FLOATS),
                      npart=npart)
            self._lat[B] = lb
        return lb

    def _prep_inputs(self, x, y):
        xt = torch.as_tensor(x) if not torch.is_tensor(x) else x
        if xt.dtype == torch.uint8:
            # raw 0..255 pixels (utils_data.py:56 before the /255 of :57-59): normalised on the device, bit-exactly
            # (fp32 division), inside the kernels of the bf16 engine or here for the fp32 engine
            x = xt.to(self.device, non_blocking=True).contiguous()
            if not getattr(self.engine, "x2", False):
                x = x.to(torch.float32) / 255.0
        else:
            x = as_device_f32(x, self.device)
        if x.dim() != 4 or tuple(x.shape[1:]) != self.ip_shape:
            raise ValueError("x must be [B,64,64,3] NHWC, got {}".format(tuple(x.shape)))
        if y is not None:
            y = (torch.as_tensor(y) if not torch.is_tensor(y) else y).to(self.device, torch.int64,
                                                                         non_blocking=True).contiguous()
            if tuple(y.shape) != (x.shape[0], self.y_dim):
                raise ValueError("y must be [B,{}], got {}".format(self.y_dim, tuple(y.shape)))
        return x, y

    def _noise(self, noise, B, supervised, K):
        n = {}
        noise = noise or {}
        for k in ("eps", "eps_k", "U_y", "U1", "U2"):
            v = noise.get(k)
            n[k] = None if v is None else as_device_f32(v, self.device)
        if not supervised:
            n["eps_k"] = None
        if n["eps_k"] is not None:
            ek = n["eps_k"]
            if ek.shape[-1] == self.z_dim:
                ek = ek[..., self.z_style:].clone()   # only the classify dims are consumed (:173)
            if tuple(ek.shape) != (K, B, self.z_classify):
                raise ValueError("eps_k must be [K,B,45] or [K,B,18], got {}".format(tuple(ek.shape)))
            n["eps_k"] = ek
        if (n["U1"] is None) != (n["U2"] is None):
            raise ValueError("U1 and U2 go together")
        return n

    # ---- the ELBO step ----------------------------------------------------------------------------------------
    @property
    def gating_sampler_temp(self):
        """gated_ccvae.py:136: the gate sampler's temperature.  The kernels read it from a device scalar, so assigning it
        (the per-epoch decay, :404-406) reaches captured graphs too - no re-capture, unlike the reference's traced
        graph, which keeps the value it was traced with (SURVEY.md quirk 8)."""
        return self._gating_sampler_temp

    @gating_sampler_temp.setter
    def gating_sampler_temp(self, t):
        t = float(t)
        if not t > 0.0:
            raise ValueError("gating_sampler_temp must be > 0")
        self._gating_sampler_temp = t
        if getattr(self, "_temp_dev", None) is not None:
            self._temp_dev.fill_(t)

    def _gate(self, n, c_in=None):
        v = self.store.view
        _lib.check(self.lib.gccvae_gate_fwd(ptr(self.store.view("mu")), ptr(c_in), ptr(n["U1"]), ptr(n["U2"]),
                                            dp.gate_seed(self.seed), self._noise_offset, ptr(self.optimiser.step_dev),
                                            self._gating_sampler_temp, ptr(self._temp_dev), ptr(v("cls.w")),
                                            ptr(v("cls.b")), ptr(v("prior.loc_true")), ptr(v("prior.loc_false")),
                                            ptr(v("prior.scale_true")), ptr(v("prior.scale_false")),
                                            ptr(self._gate_ws), ptr(self._c), _stream()), "gate_fwd")

    def _latent_fwd(self, B, lb, b, y, n, supervised, K):
        a = LatentFwdArgs()
        a.batch, a.batch_global, a.supervised, a.K = B, dp.batch_global(B, self.world), int(supervised), K
        io = self.engine.latent_io(b)
        a.loc_pre, a.scale_pre, a.ld_pre = io["loc_pre"], io["scale_pre"], io["ld_pre"]
        a.z16 = io["z16"]
        a.y, a.eps, a.eps_k, a.U_y = ptr(y), ptr(n["eps"]), ptr(n["eps_k"]), ptr(n["U_y"])
        a.seed, a.offset = dp.data_seed(self.seed, self.rank), self._noise_offset
        a.step_dev = ptr(self.optimiser.step_dev)
        a.gate_ws = ptr(self._gate_ws)
        a.loc, a.scale, a.z, a.terms, a.logits, a.y_out = (ptr(lb["loc"]), ptr(lb["scale"]), ptr(lb["z"]),
                                                           ptr(lb["terms"]), ptr(lb["logits"]), ptr(lb["y_i32"]))
        _lib.check(self.lib.gccvae_latent_fwd(C.byref(a), _stream()), "latent_fwd")

    def _latent_bwd(self, B, lb, b, n, supervised, K):
        a = LatentBwdArgs()
        a.batch, a.batch_global, a.supervised, a.K = B, dp.batch_global(B, self.world), int(supervised), K
        io = self.engine.latent_io(b)
        a.loc_pre, a.scale_pre, a.ld_pre = io["loc_pre"], io["scale_pre"], io["ld_pre"]
        a.y, a.eps, a.eps_k = ptr(lb["y_i32"]), ptr(n["eps"]), ptr(n["eps_k"])
        a.seed, a.offset = dp.data_seed(self.seed, self.rank), self._noise_offset
        a.step_dev = ptr(self.optimiser.step_dev)
        a.gate_ws, a.terms, a.log_pxz = ptr(self._gate_ws), ptr(lb["terms"]), ptr(lb["log_pxz"])
        a.dz, a.ld_dz = io["dz"], io["ld_dz"]
        a.dloc_pre, a.dscale_pre, a.dpre16 = io["dloc_pre"], io["dscale_pre"], io["dpre16"]
        a.db_loc, a.db_scale = io["db_loc"], io["db_scale"]
        a.partials, a.n_partials, a.loss_out = ptr(lb["partials"]), lb["npart"], None
        _lib.check(self.lib.gccvae_latent_bwd(C.byref(a), _stream()), "latent_bwd")

    def _chain_fwd(self, B, lb, b, y, n, supervised, K):
        """conv5 output -> heads -> latent forward -> fc1 -> conv1t in one launch (bf16 engine, csrc/chain.cu)."""
        a, io = ChainFwdArgs(), self.engine.chain_io(b)
        a.batch, a.batch_global, a.supervised, a.K = B, dp.batch_global(B, self.world), int(supervised), K
        for k_ in ("h5", "w_heads", "b_heads", "w_fc1", "b_fc1", "w_conv1t", "b_conv1t", "pre", "z16", "g0", "g1"):
            setattr(a, k_, ptr(io[k_]))
        a.y, a.eps, a.eps_k, a.U_y = ptr(y), ptr(n["eps"]), ptr(n["eps_k"]), ptr(n["U_y"])
        a.seed, a.offset, a.step_dev = dp.data_seed(self.seed, self.rank), self._noise_offset, ptr(self.optimiser.step_dev)
        a.gate_ws = ptr(self._gate_ws)
        a.loc, a.scale, a.z, a.terms, a.logits, a.y_out = (ptr(lb["loc"]), ptr(lb["scale"]), ptr(lb["z"]),
                                                           ptr(lb["terms"]), ptr(lb["logits"]), ptr(lb["y_i32"]))
        self.engine._run("chain fwd", (io["h5"], io["w_heads"], io["w_conv1t"], io["g1"]),
                         lambda: self.lib.gccvae_chain_fwd(C.byref(a), _stream()))

    def _chain_bwd(self, B, lb, b, n, supervised, K):
        """dec.conv1t.dout -> conv1t / fc1 dgrad -> latent backward -> heads dgrad -> enc.conv5.dout in one launch."""
        a, io = ChainBwdArgs(), self.engine.chain_io(b)
        a.batch, a.batch_global, a.supervised, a.K = B, dp.batch_global(B, self.world), int(supervised), K
        a.n_partials = lb["npart"]
        for k_ in ("dg1", "g0", "h5", "pre", "w_conv1t_t", "w_fc1_t", "w_heads_t", "dg0", "dpre16", "dh5", "db_loc",
                   "db_scale", "db_fc1", "db_conv1t", "db_conv5"):
            setattr(a, k_, ptr(io[k_]))
        a.y, a.eps, a.eps_k = ptr(lb["y_i32"]), ptr(n["eps"]), ptr(n["eps_k"])
        a.seed, a.offset, a.step_dev = dp.data_seed(self.seed, self.rank), self._noise_offset, ptr(self.optimiser.step_dev)
        a.gate_ws, a.terms, a.log_pxz, a.partials = ptr(self._gate_ws), ptr(lb["terms"]), ptr(lb["log_pxz"]), ptr(lb["partials"])
        self.engine._run("chain bwd", (io["dg1"], io["w_conv1t_t"], io["w_heads_t"], io["dh5"]),
                         lambda: self.lib.gccvae_chain_bwd(C.byref(a), _stream()))

    def _elbo(self, x, y, supervised, noise=None, backward=False, k=100):
        x, y = self._prep_inputs(x, y if supervised else None)
        B = x.shape[0]
        n = self._noise(noise, B, supervised, k)
        b, lb = self.engine.bufs(B), self._latent_bufs(B)
        st = _stream()
        learnable = self.model.mu_trainable
        mark = getattr(self.engine, "mark", lambda *a, **k: None)
        mark("step begin", coarse=True)
        if hasattr(self.engine, "begin_step"):
            self.engine.begin_step(x, b, lb["log_pxz"])
        if backward:
            if not self._grads_clean:    # otherwise the previous Adam launch left the buffer zeroed
                self.engine.zero_grads()
            self._grads_clean = False
        chain = getattr(self.engine, "chain", False) and getattr(self.engine, "x2", False)
        self._gate(n)
        mark("zero+gate", coarse=True)
        if chain:
            self.engine.encoder_fwd(x, b, heads=False)
            mark("encoder fwd", coarse=True)
            self._chain_fwd(B, lb, b, y, n, supervised, k)
            mark("chain fwd", coarse=True)
        else:
            self.engine.encoder_fwd(x, b)
            mark("encoder fwd", coarse=True)
            self._latent_fwd(B, lb, b, y, n, supervised, k)
            mark("latent fwd", coarse=True)
        if chain:
            xhat = self.engine.decoder_fwd_recon(x, b, lb["terms"][5], lb["log_pxz"], backward,
                                                 want_recon=not torch.cuda.is_current_stream_capturing(), head=False)
            mark("decoder fwd + recon", coarse=True)
        elif getattr(self.engine, "x2", False):
            xhat = self.engine.decoder_fwd_recon(x, b, lb["terms"][5], lb["log_pxz"], backward,
                                                 want_recon=not torch.cuda.is_current_stream_capturing())
            mark("decoder fwd + recon", coarse=True)
        else:
            self.engine.decoder_fwd(lb["z"], b, z16_ready=True)
            mark("decoder fwd", coarse=True)
            xhat = self.engine.recon(x, b, lb["terms"][5], lb["log_pxz"], backward)
            mark("recon", coarse=True)
        if backward:
            if chain:
                self.engine.decoder_bwd(lb["z"], b, tail=False)
            else:
                self.engine.decoder_bwd(lb["z"], b)
            mark("decoder bwd (main)", coarse=True)
            if chain:
                self._chain_bwd(B, lb, b, n, supervised, k)
                mark("chain bwd", coarse=True)
            else:
                self._latent_bwd(B, lb, b, n, supervised, k)
                mark("latent bwd", coarse=True)
            v, g = self.store.view, self.store.g

            def gate_bwd():
                _lib.check(self.lib.gccvae_gate_bwd(
                    ptr(lb["partials"]), lb["npart"], ptr(v("mu")), ptr(v("cls.w")), ptr(v("prior.loc_true")),
                    ptr(v("prior.loc_false")), ptr(v("prior.scale_true")), ptr(v("prior.scale_false")),
                    ptr(self._gate_ws), float(self.train_config.get("gating_reg", 0.0)), dp.l1_scale(self.world),
                    ptr(g("cls.w")), ptr(g("cls.b")), ptr(g("prior.loc_true")), ptr(g("prior.loc_false")),
                    ptr(g("prior.scale_true")), ptr(g("prior.scale_false")), ptr(g("mu")) if learnable else None,
                    ptr(self.store.loss_slot), _stream()), "gate_bwd")
                mark("gate bwd", coarse=True)

            if chain:
                # the weight gradients that read the chain kernel's outputs, and the reduction of its partial rows into
                # the gate / classifier / prior gradients (they feed only Adam and the returned loss), go to the
                # weight-gradient stream: nothing of them is left on the dgrad chain
                def after_chain():
                    self.engine.fc1_wgrad(b, B)
                    self.engine.heads_wgrad(b, B)
                    gate_bwd()
                if self.engine.post_chain_stream == "side2":
                    self.engine._on_side2(after_chain)
                else:
                    self.engine._side(after_chain, lane=self.engine.wgrad_plan[0])
                self.engine.encoder_bwd(x, b, heads=False)
            else:
                gate_bwd()
                self.engine.encoder_bwd(x, b)
            mark("encoder bwd + join", coarse=True)
        else:
            _lib.check(self.lib.gccvae_elbo_loss_f32(ptr(lb["terms"]), ptr(lb["log_pxz"]), B,
                                                     dp.batch_global(B, self.world), int(supervised),
                                                     ptr(v_mu(self)) if learnable else None,
                                                     float(self.train_config.get("gating_reg", 0.0)) * dp.l1_scale(self.world),
                                                     ptr(self._loss), st), "elbo_loss")
        t = lb["terms"]
        self.last = dict(post_locs=lb["loc"], post_scales=lb["scale"], z=lb["z"], logits=lb["logits"], kl=t[0],
                         log_qy_zc=t[1], log_qy_x=t[2], w=t[3], log_py=t[4], log_pxz=lb["log_pxz"], recon=xhat,
                         y=lb["y_i32"], c=self._c, supervised=supervised)
        return (self.store.loss_slot[0] if backward else self._loss[0]), self._c

    @contextlib.contextmanager
    def _fresh_noise(self):
        """Philox counter offset of a forward-only call: different for every call (see _noise_offset)."""
        self._eval_calls += 1
        self._noise_offset = self._eval_calls << 32
        try:
            yield
        finally:
            self._noise_offset = 0

    # ---- reference API ---------------------------------------------------------------------------------------------
    def sup_loss(self, x, y, noise=None, k=100):
        """gated_ccvae.py:234-300 -> (loss, c).  With autograd enabled on the parameters (`requires_grad_()`), the
        returned loss carries the graph edge the reference's GradientTape records (:302-309): `loss.backward()` leaves
        d loss / d parameters in `self.store.flat.grad` (`gradients()` views it per tensor).  Otherwise forward only."""
        if self._wants_grad():
            return _ElboFunction.apply(self.store.flat, self, x, y, True, noise, k)
        with self._fresh_noise():
            loss, c = self._elbo(x, y, True, noise, backward=False, k=k)
        return self._global_loss(loss).clone(), c.clone()

    def unsup_loss(self, x, noise=None):
        """gated_ccvae.py:184-232 -> (loss, c); differentiable like sup_loss."""
        if self._wants_grad():
            return _ElboFunction.apply(self.store.flat, self, x, None, False, noise, 100)
        with self._fresh_noise():
            loss, c = self._elbo(x, None, False, noise, backward=False)
        return self._global_loss(loss).clone(), c.clone()

    def requires_grad_(self, flag=True):
        """make sup_loss / unsup_loss differentiable w.r.t. the (flat) parameter buffer, torch style."""
        self.store.flat.requires_grad_(bool(flag))
        if not flag:
            self.store.flat.grad = None
        return self

    def _wants_grad(self):
        return torch.is_grad_enabled() and self.store.flat.requires_grad

    def gradients(self):
        """{name: view of d loss / d tensor} after `loss.backward()` (None before)."""
        g = self.store.flat.grad
        return None if g is None else {k: self.store.view(k, g) for k in self.store.names()}

    def classifier_loss(self, x, y, c, k=100, noise=None):
        """gated_ccvae.py:167-182: log q(y|x) ~ logsumexp_k log q(y|z_c^k, c) - log k  -> [B]."""
        x, y = self._prep_inputs(x, y)
        B = x.shape[0]
        n = self._noise(noise, B, True, k)
        b, lb = self.engine.bufs(B), self._latent_bufs(B)
        with self._fresh_noise():
            self._gate(n, c_in=as_device_f32(c, self.device))
            self.engine.encoder_fwd(x, b)
            self._latent_fwd(B, lb, b, y, n, True, k)
        return lb["terms"][2].clone()

    def loss_and_grads(self, x, y, supervised, noise=None, k=100):
        """forward + backward without the optimiser: (loss, c), gradients in self.store.grad."""
        loss, c = self._elbo(x, y, supervised, noise, backward=True, k=k)
        self._allreduce_grads()      # the loss rides in the tail slot of the gradient buffer
        return loss.clone(), c.clone()

    def train_step(self, x, y, supervised, noise=None, k=100, inputs_ready=False):
        """gated_ccvae.py:302-311: loss, gradients of all trainable variables, Adam update -> (loss, c), both fresh
        for the next RING steps (rows of the result ring the publishing Adam launch fills).
        `inputs_ready` (graph replay only): the caller promises that DEVICE tensors x / y are complete - nothing that
        writes them is pending on any stream - so their staging (copy into the graph's input buffers, x2 transform) may
        run under the step in flight instead of behind it.  Host tensors are always staged that way."""
        if self._t_host is None:
            self._t_host = self.optimiser.iterations
        slot = self._ring[self._t_host % self.RING]
        if self.use_graphs and noise is None:
            self._train_step_graphed(x, y, supervised, k, inputs_ready)
        else:
            self._step_body(x, y, supervised, noise, k)
        self._t_host += 1
        return slot[0], slot[1:1 + 324].view(18, 18)

    def _adam_head(self):
        if self._peer is not None:
            self._peer_adam(self._adam_cut, self.n_trainable, self.store.total, publish=False)
        else:
            self.optimiser.apply_gradients(lo=self._adam_cut, hi=None, publish=False)
        getattr(self.engine, "mark", lambda *a, **k: None)("adam head", coarse=True)
        self._adam_head_done = True

    def _result(self):
        return (self.store.loss_slot, self._c, self._ring)

    def _step_body(self, x, y, supervised, noise, k):
        """forward + backward + (all-reduce) + Adam, as issued eagerly or captured into the step's graph."""
        split = (self.world == 1 or self._peer is not None) and hasattr(self.engine, "tail_hook") and self.adam_tail
        self._adam_head_done = False
        if split:
            self.engine.tail_hook, self.engine.tail_hook_layer = self._adam_head, self._tail_layer
        loss, c = self._elbo(x, y, supervised, noise, backward=True, k=k)
        if split:
            self.engine.tail_hook = None
        if self._peer is not None:
            if self._adam_head_done:
                self._peer_adam(0, self._adam_cut, self._adam_cut, publish=True, push=True)
            else:
                self._peer_adam(0, self.n_trainable, self.store.total, publish=True)
            self._grads_clean = True
        elif self._adam_head_done:
            self._grads_clean = self.optimiser.apply_gradients(lo=0, hi=self._adam_cut, publish=True,
                                                               result=self._result())
        else:
            self._allreduce_grads()
            self._grads_clean = self.optimiser.apply_gradients(result=self._result())
        return loss, c

    # ---- CUDA-graph replay of the step (the reference's @tf.function, gated_ccvae.py:302) -------------------------
    def _train_step_graphed(self, x, y, supervised, k, inputs_ready=False):
        B = int(x.shape[0])
        x = torch.as_tensor(x)
        u8 = x.dtype == torch.uint8 and getattr(self.engine, "x2", False)
        key = (B, bool(supervised), int(k), bool(u8))      # (the gate temperature is a device scalar: not part of the key)
        # two captured variants per key with their own static input buffers, used alternately: the host->device copy
        # of a batch goes STRAIGHT into the static input of the variant that is not executing (no staging copy) and
        # overlaps the step in flight
        variants = self._graphs.setdefault(key, [None, None])
        turn = self._graph_turn.get(key, 0)
        self._graph_turn[key] = turn ^ 1
        g = variants[turn]
        if g is None:
            g = variants[turn] = self._capture(key)
        if x.dtype == torch.uint8 and not u8:
            x = x.to(self.device, non_blocking=True).to(torch.float32) / 255.0
        main = torch.cuda.current_stream()
        if x.device.type == "cpu" or g["x2"] is not None:
            # inputs travel on the copy stream: the copy of a host batch - or of a resident one - into this variant's static
            # buffers and (bf16 engine) the x2 block transform of the image run AHEAD of the replay, under the step in flight
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=self.device)
            cs = self._copy_stream
            if g.get("done") is not None:
                cs.wait_event(g["done"])          # the previous replay of this variant no longer reads its inputs
            else:
                cs.wait_stream(main)
            if x.device.type != "cpu" and not inputs_ready:
                cs.wait_stream(main)              # a resident batch may still be in production on the caller's stream
            with torch.cuda.stream(cs):
                g["x"].copy_(x, non_blocking=True)
                if supervised:
                    g["y"].copy_(torch.as_tensor(y), non_blocking=True)
                if g["x2"] is not None:
                    _lib.check(self.engine.prep_x2(g["x"], g["x2"], cs.cuda_stream), "prep_x2")
                ready = torch.cuda.Event()
                ready.record(cs)
            main.wait_event(ready)
        else:
            g["x"].copy_(x, non_blocking=True)
            if supervised:
                g["y"].copy_(torch.as_tensor(y), non_blocking=True)
        if g["clean"] and not self._grads_clean:
            self.engine.zero_grads()   # the graph was captured without a memset: it relies on the previous Adam launch
        g["graph"].replay()
        self.lib.gccvae_add_launch_count(g["launches"])
        if self.world > 1 and self._peer is None:   # NCCL stays outside the graph: replay(fwd+bwd) -> all-reduce -> Adam
            self._allreduce_grads()
            self._grads_clean = self.optimiser.apply_gradients(result=self._result())
        else:
            self._grads_clean = g["clean"]
        # the next host->device copy into this variant's inputs may start once this event fires.  Recorded AFTER the
        # all-reduce: measured on 2 B200s, an all-reduce that runs while a host->device copy to the same GPU is in
        # flight does not complete before the copy does (1.82 instead of 1.47 ms per step pair, proportional to the
        # bytes copied) - so the copy is released behind it and overlaps the next replay instead.
        g["done"] = torch.cuda.Event()
        g["done"].record(main)
        return g["loss"], self._c

    def _capture(self, key):
        B, supervised, k, u8 = key
        xs = torch.zeros(B, *self.ip_shape, dtype=torch.uint8 if u8 else torch.float32, device=self.device)
        ys = torch.zeros(B, self.y_dim, dtype=torch.int64, device=self.device) if supervised else None
        # bf16 engine: this variant's own image blocks, filled ahead of each replay on the copy stream (_train_step_graphed)
        x2 = bufs = None
        if getattr(self.engine, "x2", False):
            bufs = self.engine.bufs(B)
            x2 = torch.zeros_like(bufs["X2"])

        def body():
            if getattr(self.engine, "marks", None) is not None:
                self.engine.marks = []
            if self.world == 1 or self._peer is not None:   # the whole step, exchange + optimiser included, is one graph
                loss, _ = self._step_body(xs, ys, supervised, None, k)
                getattr(self.engine, "mark", lambda *a, **k: None)("adam", coarse=True)
            else:       # NCCL stays outside the graph: the all-reduce and Adam follow the replay
                loss, _ = self._elbo(xs, ys, supervised, None, backward=True, k=k)
            return loss

        # warm-up on a side stream (first-use attribute calls, buffer allocation), state restored afterwards
        saved = (self.store.flat.clone(), self.optimiser.m.clone(), self.optimiser.v.clone(),
                 self.optimiser.step_dev.clone())
        if x2 is not None:
            saved_x2, bufs["X2"], self.engine.x2_ready = bufs["X2"], x2, True
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        n0 = self.lib.gccvae_launch_count()
        # the captured step carries no gradient memset: every replay starts from the buffer the (fused) Adam launch of
        # the previous step cleared - inside the graph on one GPU, after the all-reduce in data-parallel runs
        fused = True
        if not self._grads_clean:
            self.engine.zero_grads()
        self._grads_clean = True
        with torch.cuda.graph(graph):
            loss = body()
        launches = self.lib.gccvae_launch_count() - n0
        torch.cuda.synchronize(self.device)
        for dst, src in zip((self.store.flat, self.optimiser.m, self.optimiser.v, self.optimiser.step_dev), saved):
            dst.copy_(src)
        self._grads_clean = True         # nothing ran during the capture: the buffer is as clean as before it
        if x2 is not None:
            bufs["X2"], self.engine.x2_ready = saved_x2, False
        return dict(graph=graph, x=xs, y=ys, x2=x2, loss=loss, launches=launches, done=None, clean=fused)

    def classifier_accuracy(self, x, y, noise=None):
        """gated_ccvae.py:421-446."""
        x, y = self._prep_inputs(x, y)
        B = x.shape[0]
        n = self._noise(noise, B, False, 0)
        b, lb = self.engine.bufs(B), self._latent_bufs(B)
        with self._fresh_noise():
            self._gate(n)
            self.engine.encoder_fwd(x, b)
            self._latent_fwd(B, lb, b, None, n, False, 0)
        _lib.check(self.lib.gccvae_accuracy_f32(ptr(lb["logits"]), ptr(y), B * self.y_dim, ptr(self._acc),
                                                _stream()), "accuracy")
        return self._acc[0].clone()

    def accuracy(self, data_loader):
        """gated_ccvae.py:448-455 (data_loader.step() yields (xs, ys); .n_s = number of samples)."""
        acc = 0.0
        iterator = iter(data_loader.step())
        num_batches = math.ceil(data_loader.n_s / self.train_config["batch_size"])
        for _ in range(int(num_batches)):
            xs, ys = next(iterator)
            acc += float(self.classifier_accuracy(xs, ys))
        return acc / num_batches

    # ---- generation path (an extension: the reference has no call that turns labels into images) --------------------
    def generate(self, y, sample=True, c=None, noise=None, dtype=torch.float32):
        """Images for target labels y [B,18] (nonzero = 1): z_s = eps_s, z_c = loc_p(y,c) + scale_p(y,c) eps_c with the
        conditional prior p(z_c|y,c) (networks.py:118-127); `sample=False`: z_s = 0, z_c = loc_p(y,c).
        Returns a fresh [B,64,64,3] NHWC device tensor: fp32 sigmoid values (`dtype=torch.float32`) or uint8
        min(255, rint(255 x)) (`dtype=torch.uint8`).  See `intervene` for c, noise and `last`."""
        return self._image_call(_lib.GEN_GENERATE, None, y, None, sample, c, noise, dtype)

    def reconstruct(self, x, sample=False, noise=None, dtype=torch.float32):
        """Decoded posterior of images x [B,64,64,3] (fp32 in [0,1] or uint8 0..255): z = the posterior mean (heads after
        relu / clipped softplus, networks.py:17-18,33-34); `sample=True`: z = loc + scale eps.  Returns the image as
        `generate` does."""
        return self._image_call(_lib.GEN_RECONSTRUCT, x, None, None, sample, None, noise, dtype)

    def intervene(self, x, y_new, y=None, sample=False, c=None, noise=None, dtype=torch.float32):
        """Counterfactual of images x: z as in `reconstruct`, then the classify dims move from the labels y to y_new
        ([B,18] each, nonzero = 1) by abduction - action - prediction under the conditional prior:
            e = (z_c - loc_p(y,c)) / scale_p(y,c),  z_c' = z_c + (loc_p(y_new,c) - loc_p(y,c)) + (scale_p(y_new,c) - scale_p(y,c)) e.
        y_new == y leaves z bit-identical (the result equals `reconstruct(x)`); the style dims are never touched.
        y=None: the classifier's decision sigmoid(logit) > 0.5 on the z_c being moved.  Returns the image as `generate`.

        Common to the three calls: c [18,18] is a fresh gate sample at the current `gating_sampler_temp` unless given
        (pass the same c to a series of edits); `noise={"eps": [B,45], "U1": [18,18], "U2": [18,18]}` makes the draws
        explicit (eps layout: style dims 0..26, classify dims 27..44); without it every call draws new noise.
        `self.last` = {"z": [B,45], "c": [18,18], "y_src": [B,18] int32 labels moved from (intervene) or None}.
        In data-parallel runs every rank works on its own batch; there is no collective."""
        return self._image_call(_lib.GEN_INTERVENE, x, y_new, y, sample, c, noise, dtype)

    def _gen_labels(self, y, B, what):
        t = torch.as_tensor(y) if not torch.is_tensor(y) else y
        if t.dim() != 2 or t.shape[1] != self.y_dim or t.shape[0] == 0 or (B is not None and t.shape[0] != B):
            raise ValueError("{} must be [B,{}]{}, got {}".format(what, self.y_dim, "" if B is None else " with B={}".format(B),
                                                                tuple(t.shape)))
        return (t.to(self.device, non_blocking=True) != 0).to(torch.int64).contiguous()

    @staticmethod
    def _check_dtype(dtype):
        if dtype not in (torch.float32, torch.uint8):
            raise ValueError("dtype must be torch.float32 or torch.uint8, got {}".format(dtype))

    def _gen_images(self, x):
        """images of the forward-only calls -> (device tensor, B)."""
        x, _ = self._prep_inputs(x, None)
        if x.shape[0] == 0:
            raise ValueError("x holds no image")
        return x, x.shape[0]

    def _gen_noise_c(self, noise, c, shapes):
        """explicit draws and gate of the forward-only calls, checked: shapes = {noise key: required shape}."""
        n = self._noise(noise, None, False, 0)
        for k, shape in list(shapes.items()) + [("U1", (18, 18)), ("U2", (18, 18))]:
            if n[k] is not None and tuple(n[k].shape) != shape:
                raise ValueError("noise[{!r}] must be {}, got {}".format(k, list(shape), tuple(n[k].shape)))
        if c is not None:
            c = as_device_f32(c, self.device)
            if tuple(c.shape) != (18, 18):
                raise ValueError("c must be [18,18], got {}".format(tuple(c.shape)))
        return n, c

    @staticmethod
    def _check_max_rows(max_rows):
        if isinstance(max_rows, bool) or not isinstance(max_rows, (int, np.integer)) or max_rows < 1:
            raise ValueError("max_rows must be an integer >= 1, got {!r}".format(max_rows))
        return int(max_rows)

    def _image_call(self, mode, x, y_tgt, y_src, sample, c, noise, dtype, frames=None, complete=None):
        """generate / reconstruct / intervene (one frame per image, decoded in `bufs(B)`) and, with frames = (kind, items,
        values, max_rows), the calls with several frames per image (decoded in chunks through `dec_bufs`): "walk" (items:
        labels), "traverse" (items: latent dims) and "pair" (items: the mixed range (lo, hi); x = (x_a, x_b)).  Checks,
        gate, encoder or weight packing, then per chunk gccvae_gen_latent and the decoder into the chunk's rows of the
        output.  complete = (mask, iters): that body `iters` times, each time on the composite of x's observed pixels and
        the previous decode (`complete`), with the gate of the first."""
        self._check_dtype(dtype)
        kind, shape = None, ()
        if frames is not None:
            kind, items, values, max_rows = frames
            max_rows = self._check_max_rows(max_rows)
            values = self._walk_alphas(values, "alphas" if kind == "walk" else "values" if kind == "traverse" else "ts")
            if kind == "walk":
                items = self._walk_labels(items)
            elif kind == "traverse":
                items = self._traverse_dims(items)
            shape = (values.numel(),) if kind == "pair" else (len(items), values.numel())
        B = None
        if kind == "pair":
            xa, B = self._gen_images(x[0])
            xb, Bb = self._gen_images(x[1])
            if Bb != B:
                raise ValueError("the two image sets must hold as many images, got {} and {}".format(B, Bb))
            if xa.dtype != xb.dtype:     # one of each: both as fp32 in [0,1], the division the kernels do on uint8 images
                xa, xb = (t.to(torch.float32) / 255.0 if t.dtype == torch.uint8 else t for t in (xa, xb))
            x = torch.cat([xa, xb])
        elif x is not None:
            x, B = self._gen_images(x)
        elif frames is not None and y_tgt is None:
            raise ValueError("{} needs images x or labels y".format(kind))
        if y_tgt is not None:
            y_tgt = self._gen_labels(y_tgt, B, "y" if x is None else "y_new")
            B = y_tgt.shape[0]
        if y_src is not None:
            y_src = self._gen_labels(y_src, B, "y")
        iters = 1
        if complete is not None:
            mask, iters = self._complete_mask(complete[0], B), complete[1]
        n, c = self._gen_noise_c(noise, c, {"eps": (B, self.z_dim) if complete is None else (iters, B, self.z_dim)})
        rows = B * math.prod(shape)
        if rows >= 1 << 31:
            raise ValueError("{} of {} frames: at most 2^31 - 1".format(kind, rows))
        out = torch.empty(B, *shape, 64, 64, 3, dtype=dtype, device=self.device)
        z = torch.empty(B, *shape, self.z_dim, dtype=torch.float32, device=self.device)
        y_used = torch.empty(B, self.y_dim, dtype=torch.int32, device=self.device) if mode == _lib.GEN_INTERVENE else None
        a = GenLatentArgs()
        a.batch, a.mode, a.sample = B, mode, int(bool(sample))
        if frames is None:
            dec, chunks = self.engine.bufs(B), [(0, B, z, out)]
        else:
            chunk = min(max_rows, rows)
            dec = self.engine.dec_bufs(chunk)
            z_rows, out_rows = z.view(rows, self.z_dim), out.view(rows, 64, 64, 3)
            chunks = [(r0, min(chunk, rows - r0), z_rows[r0:r0 + chunk], out_rows[r0:r0 + chunk])
                      for r0 in range(0, rows, chunk)]
            if kind == "walk":
                a.n_labels = len(items)
                a.labels[:len(items)] = items
            elif kind == "traverse":
                a.n_dims = len(items)
                a.dims[:len(items)] = items
            else:
                a.pair, (a.mix_lo, a.mix_hi) = 1, items
            a.n_alpha = values.numel()
            values = values.to(self.device)
            a.alphas = ptr(values)
        # (one iteration decodes straight into the output: no composite, no mask blocks)
        state = self.engine.complete_begin(x, mask) if iters > 1 else None
        x_in = x
        for t in range(iters):
            # a pair reads no gate, prior or noise: it leaves c and the noise stream of the other calls as they were
            with contextlib.nullcontext() if kind == "pair" else self._fresh_noise():
                if kind != "pair" and t == 0:
                    self._gate(n, c_in=c)
                if x is None:
                    self.engine.pack_weights()
                else:
                    b = self.engine.bufs(x.shape[0])
                    if t > 0 and getattr(self.engine, "x2", False):   # the composite is already in b["X2"]
                        self.engine.encoder_fwd(x_in, b, blocks_ready=True)
                    else:
                        self.engine.encoder_fwd(x_in, b)
                    io = self.engine.latent_io(b)
                    a.loc_pre, a.scale_pre, a.ld_pre = io["loc_pre"], io["scale_pre"], io["ld_pre"]
                eps = n["eps"] if complete is None or n["eps"] is None else n["eps"][t]
                a.y_tgt, a.y_src, a.eps = ptr(y_tgt), ptr(y_src), ptr(eps)
                a.seed, a.offset, a.step_dev = dp.data_seed(self.seed, self.rank), self._noise_offset, ptr(self.optimiser.step_dev)
                a.gate_ws, a.z16, a.y_src_out = ptr(self._gate_ws), ptr(dec.get("z16")), ptr(y_used)
                for r0, nr, z_chunk, out_chunk in chunks:
                    a.row0, a.rows, a.z = r0, nr, ptr(z_chunk)
                    _lib.check(self.lib.gccvae_gen_latent(C.byref(a), _stream()), "gen_latent")
                    if t + 1 < iters:
                        x_in = self.engine.complete_fwd(z_chunk, dec, nr, state, x)
                    else:
                        self.engine.image_fwd(z_chunk, dec, nr, dtype == torch.uint8, out=out_chunk)
        if complete is not None:    # the observed pixels are x's, converted to dtype as the image calls convert
            if dtype == torch.uint8 and x.dtype != torch.uint8:
                x = image_u8(x)
            elif dtype == torch.float32 and x.dtype == torch.uint8:
                x = torch.div(x, 255.0)     # fp32 u / 255, as x.to(torch.float32) / 255.0 in one pass
            out = torch.where(mask.unsqueeze(-1), x, out)
        if kind == "pair":
            self.last = dict(z=z)
        elif kind == "traverse":
            self.last = dict(z=z, c=self._c.clone())
        else:
            self.last = dict(z=z, c=self._c.clone(), y_src=y_used)
        return out

    def walk(self, x=None, y=None, labels=None, alphas=None, sample=False, c=None, noise=None, dtype=torch.float32,
             max_rows=8192):
        """Frames along single labels: for every image, every label l of `labels` and every value a of `alphas`, the
        image decoded with y_l replaced by the real number a and the other labels kept.  The conditional prior is affine
        in y before its softplus (networks.py:118-127), so it is defined at any finite a: a = 0 and a = 1 are the prior's
        own boolean terms, bit for bit, values beyond [0, 1] extrapolate.
          From images (x [B,64,64,3] given), the counterpart of `intervene`: z as in `reconstruct`, then the classify dims
            move from the labels y (default: the classifier's decision on z_c) to y with y_l = a, by the counterfactual of
            `intervene`.  The frame at a = y_l is `reconstruct(x)`; a = 1 - y_l is `intervene` with label l flipped.
          From labels (x=None, y [B,18] required), the counterpart of `generate`: z_s = eps_s, z_c = loc_p + scale_p eps_c
            at the walked labels (`sample=False`: z_s = 0, z_c = loc_p).
        labels: distinct label indices in [0, 18), in output order (default: all 18); alphas: a non-empty 1-D sequence of
        finite floats, taken as fp32 (default: 8 points from 0 to 1, both ends exact).  The noise of an image is drawn
        once and shared by all its frames; c, `noise={"eps": [B,45], "U1", "U2"}` and `dtype` are as in `generate`.
        Returns a fresh [B, L, T, 64, 64, 3] device tensor (L labels, T alphas), decoded in chunks of at most `max_rows`
        frames, which bounds the memory and changes no value.
        `self.last` = {"z": [B,L,T,45] fp32, "c": [18,18], "y_src": [B,18] int32 labels walked from (images) or None}.
        In data-parallel runs every rank works on its own batch; there is no collective."""
        frames = ("walk", labels, alphas, max_rows)
        if x is None:
            return self._image_call(_lib.GEN_GENERATE, None, y, None, sample, c, noise, dtype, frames)
        return self._image_call(_lib.GEN_INTERVENE, x, None, y, sample, c, noise, dtype, frames)

    def _walk_labels(self, labels):
        if labels is None:
            return list(range(self.y_dim))
        v = np.asarray(labels.cpu() if torch.is_tensor(labels) else labels)
        if v.ndim != 1 or v.size == 0 or v.dtype.kind not in "iu":
            raise ValueError("labels must be a non-empty 1-D sequence of integers, got {!r}".format(labels))
        out = [int(t) for t in v]
        if min(out) < 0 or max(out) >= self.y_dim or len(set(out)) != len(out):
            raise ValueError("labels must be distinct indices in [0, {}), got {}".format(self.y_dim, out))
        return out

    @staticmethod
    def _walk_alphas(alphas, name="alphas"):
        """alphas of `walk`, values of `traverse`, ts of `interpolate`; None: 8 points from 0 to 1, both ends exact."""
        if alphas is None:
            return torch.arange(8, dtype=torch.float64).div(7).float()     # 0/7 .. 7/7: both ends exact
        try:
            v = torch.as_tensor(alphas.detach().cpu() if torch.is_tensor(alphas) else alphas, dtype=torch.float32)
        except (TypeError, ValueError, RuntimeError) as e:
            raise ValueError("{} must be a 1-D sequence of floats, got {!r}".format(name, alphas)) from e
        if v.dim() != 1 or v.numel() == 0 or not bool(torch.isfinite(v).all()):
            raise ValueError("{} must be a non-empty 1-D sequence of finite floats, got {!r}".format(name, alphas))
        return v.contiguous()

    def traverse(self, x=None, y=None, dims=None, values=None, sample=False, c=None, noise=None, dtype=torch.float32,
                 max_rows=8192):
        """Frames along single latent dims: for every image, every dim d of `dims` and every value v of `values`, the
        image decoded from the base code with z_d set to v; every other dim keeps the base code's bits.  This shows what
        one latent encodes, also a style dim (0..26) that no label reaches or a classify dim (27..44) that a learned gate
        wires to several labels or to none.
          From images (x [B,64,64,3] given): the base code is `reconstruct(x, sample)`'s z.
          From labels (x=None, y [B,18] required): the base code is `generate(y, sample)`'s z.
        dims: distinct latent indices in [0, 45), in output order (default: all 45); values: a non-empty 1-D sequence of
        finite floats, taken as fp32, the absolute value given to z_d (default: the integers -3 .. 3).  The frame whose
        value is the base's own z_d is the base image, bit for bit.  The noise of an image is drawn once and shared by
        all its frames; c, `noise={"eps": [B,45], "U1", "U2"}` and `dtype` are as in `generate`.
        Returns a fresh [B, D, T, 64, 64, 3] device tensor (D dims, T values), decoded in chunks of at most `max_rows`
        frames, which bounds the memory and changes no value.  `self.last` = {"z": [B,D,T,45] fp32, "c": [18,18]}.
        In data-parallel runs every rank works on its own batch; there is no collective."""
        if values is None:
            values = torch.arange(-3, 4, dtype=torch.float32)
        frames = ("traverse", dims, values, max_rows)
        if x is None:
            if y is None:
                raise ValueError("traverse needs images x or labels y")
            return self._image_call(_lib.GEN_GENERATE, None, y, None, sample, c, noise, dtype, frames)
        if y is not None:
            raise ValueError("traverse takes images x or labels y, not both")
        return self._image_call(_lib.GEN_RECONSTRUCT, x, None, None, sample, c, noise, dtype, frames)

    def _traverse_dims(self, dims):
        if dims is None:
            return list(range(self.z_dim))
        v = np.asarray(dims.cpu() if torch.is_tensor(dims) else dims)
        if v.ndim != 1 or v.size == 0 or v.dtype.kind not in "iu":
            raise ValueError("dims must be a non-empty 1-D sequence of integers, got {!r}".format(dims))
        out = [int(t) for t in v]
        if min(out) < 0 or max(out) >= self.z_dim or len(set(out)) != len(out):
            raise ValueError("dims must be distinct indices in [0, {}), got {}".format(self.z_dim, out))
        return out

    def interpolate(self, x_a, x_b, ts=None, part="all", dtype=torch.float32, max_rows=8192):
        """Frames on the straight line between the posterior means z_a of x_a and z_b of x_b: for every pair and every t
        of `ts`, the image decoded from z with z = z_a outside the mixed dims and, inside them, z_a + t (z_b - z_a) -
        exactly z_a at t = 0 and exactly z_b at t = 1; values beyond [0, 1] extrapolate.  part: the mixed dims, "all"
        (0..44), "style" (0..26) or "classify" (27..44).  So part "classify" at t = 1 is `swap(x_a, x_b)` and part "all"
        at t = 1 is `reconstruct(x_b)`, bit for bit.  No gate, prior or noise is involved.
        x_a, x_b: [B,64,64,3] each (fp32 in [0,1] or uint8), one encoder pass over the 2B images; ts: a non-empty 1-D
        sequence of finite floats, taken as fp32 (default: 8 points from 0 to 1, both ends exact).  Returns a fresh
        [B, T, 64, 64, 3] device tensor, decoded in chunks of at most `max_rows` frames (this changes no value), as
        `generate` does for `dtype`.  `self.last` = {"z": [B,T,45] fp32}.
        In data-parallel runs every rank works on its own batch; there is no collective."""
        ranges = {"all": (0, self.z_dim), "style": (0, self.z_style), "classify": (self.z_style, self.z_dim)}
        if not isinstance(part, str) or part not in ranges:
            raise ValueError("part must be one of 'all', 'style', 'classify', got {!r}".format(part))
        return self._image_call(_lib.GEN_RECONSTRUCT, (x_a, x_b), None, None, False, None, None, dtype,
                                ("pair", ranges[part], ts, max_rows))

    def swap(self, x_style, x_char, dtype=torch.float32):
        """Characteristic swap: images decoded from z = [z_s of x_style, z_c of x_char], both posterior means (the style
        of one image with the label-linked latents of another).  x_style and x_char are [B,64,64,3] each (fp32 in [0,1]
        or uint8) and go through one encoder pass over 2B images; no gate and no prior are involved, so swap(x, x) is
        reconstruct(x).  It is `interpolate(x_style, x_char, ts=[1.0], part="classify")`.  Returns a fresh [B,64,64,3]
        image as `generate` does; `self.last` = {"z": [B,45]}."""
        out = self.interpolate(x_style, x_char, ts=[1.0], part="classify", dtype=dtype)
        self.last = dict(z=self.last["z"][:, 0])
        return out[:, 0]

    def complete(self, x, mask, y_new=None, y=None, iters=10, sample=False, c=None, noise=None, dtype=torch.float32):
        """Completion of partially observed images x [B,64,64,3] (fp32 in [0,1] or uint8): mask [B,64,64] or [64,64]
        (broadcast over the batch), bool or integer, nonzero = the pixel (all three channels) is observed.  The pixels
        that are not observed start from whatever x holds there (the caller's initial fill, e.g. grey or noise).  Each of
        the `iters` iterations (pseudo-Gibbs / iterative reconstruction) encodes the current composite, takes z as
        `reconstruct` does (`sample=False`: the posterior mean, `sample=True`: loc + scale eps) and - with target labels
        y_new [B,18] - moves the classify dims from y (default: the classifier's decision on that iteration's z_c) to
        y_new as `intervene` does; the decoder's mean (the sigmoid every image call returns) then replaces the unobserved
        pixels of the composite.  Observed pixels never change.  So one iteration is `reconstruct` / `intervene` of the
        composite, bit for bit, followed by torch.where(mask, x, image) in fp32.
        c [18,18]: one gate sample per call unless given, shared by every iteration; iteration t draws its noise as the
        t-th of `iters` consecutive calls would; `noise={"eps": [iters,B,45], "U1": [18,18], "U2": [18,18]}` makes the
        draws explicit.  Returns a fresh [B,64,64,3] device tensor of `dtype`: the observed pixels are x (uint8 -> fp32
        as u / 255, fp32 -> uint8 as min(255, rint(255 x))), the others the last iteration's decode, as `generate`
        returns it.  `self.last` = {"z": [B,45] of the last iteration, "c": [18,18], "y_src": [B,18] int32 labels the last
        iteration moved from (with y_new) or None}.
        On the bf16 engine the decode of every iteration but the last goes straight into the unobserved pixels of the
        encoder's input blocks (gccvae_convt_complete_bf16): no image, mask pass or block transform in between.
        In data-parallel runs every rank works on its own batch; there is no collective."""
        if y is not None and y_new is None:
            raise ValueError("complete: source labels y need target labels y_new")
        if isinstance(iters, bool) or not isinstance(iters, (int, np.integer)) or iters < 1:
            raise ValueError("iters must be an integer >= 1, got {!r}".format(iters))
        mode = _lib.GEN_RECONSTRUCT if y_new is None else _lib.GEN_INTERVENE
        return self._image_call(mode, x, y_new, y, sample, c, noise, dtype, complete=(mask, int(iters)))

    def _complete_mask(self, mask, B):
        """mask of `complete` -> [B,64,64] bool device tensor (True = observed)."""
        m = torch.as_tensor(mask) if not torch.is_tensor(mask) else mask
        if (m.dtype.is_floating_point or m.dtype.is_complex or m.dim() not in (2, 3) or tuple(m.shape[-2:]) != (64, 64)
                or (m.dim() == 3 and m.shape[0] != B)):
            raise ValueError("mask must be [B,64,64] or [64,64] bool or integer with B={}, got {} {}".format(
                B, tuple(m.shape), m.dtype))
        return (m.to(self.device, non_blocking=True) != 0).expand(B, 64, 64).contiguous()

    # ---- importance-weighted log-likelihood (an extension: the reference scores a model by accuracy only) ------------
    def log_likelihood(self, x, y=None, k=100, c=None, noise=None, max_rows=8192, keep_log_w=False):
        """Importance-weighted (IWAE) estimate of log p(x) - or of log p(x, y) when labels y [B,18] (nonzero = 1) are
        given - per image, in nats: log p_hat = logsumexp_k log w_k - ln k over k samples z_k = loc + scale eps_k of the
        posterior, with
            log w_k = log p(x|z_k) + log p(z_s) + log p(z_c|y_k, c) + log p(y_k) - log q(z_k|x) [- log q(y_k|z_c, c)]
        where y_k = y, or (y=None) y_k ~ Bernoulli(sigmoid(classifier(z_c))) as unsup_loss draws it and the bracketed
        term is included.  A lower bound that tightens as k grows; conditional on the call's gate sample c (in one-one
        mode c = I exactly).  x: [B,64,64,3] fp32 in [0,1] or uint8.  Returns a fresh fp32 [B] device tensor.
          c [18,18]: a fresh gate sample per call unless given (as `generate`);
          noise={"eps": [k,B,45], "U_y": [k,B,18], "U1": [18,18], "U2": [18,18]}: explicit draws (eps layout: style
            dims 0..26, classify dims 27..44); without it every call draws new noise;
          max_rows: decoder rows per chunk - the k samples are decoded in chunks of max(1, max_rows // B) samples per
            image; this bounds memory and changes only the order of float sums (no draw depends on it);
          keep_log_w: also keep every log w_k.
        `self.last` = {"ess": [B] effective sample size (sum w)^2 / sum w^2, "c": [18,18], "log_w": [k,B] or None}.
        In data-parallel runs every rank works on its own batch; there is no collective."""
        if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or k < 1:
            raise ValueError("k must be an integer >= 1, got {!r}".format(k))
        max_rows = self._check_max_rows(max_rows)
        K = int(k)
        x, B = self._gen_images(x)
        x = x.contiguous()
        if y is not None:
            y = self._gen_labels(y, B, "y")
        n, c = self._gen_noise_c(noise, c, {"eps": (K, B, self.z_dim), "U_y": (K, B, self.y_dim)})
        kc = max(1, min(K, max_rows // B))
        b, dec = self.engine.bufs(B), self.engine.dec_bufs(B * kc)
        e = lambda *s: torch.empty(*s, dtype=torch.float32, device=self.device)
        lw_part, log_pxz, state, est, ess = e(B * kc), e(B * kc), e(B, 3), e(B), e(B)
        log_w = e(K, B) if keep_log_w else None
        with self._fresh_noise():
            self._gate(n, c_in=c)
            self.engine.encoder_fwd(x, b)
            io = self.engine.latent_io(b)
            a = IwLatentArgs()
            a.batch, a.K, a.labelled = B, K, int(y is not None)
            a.loc_pre, a.scale_pre, a.ld_pre = io["loc_pre"], io["scale_pre"], io["ld_pre"]
            a.y, a.eps, a.U_y = ptr(y), ptr(n["eps"]), ptr(n["U_y"])
            a.seed, a.offset, a.step_dev = dp.data_seed(self.seed, self.rank), self._noise_offset, ptr(self.optimiser.step_dev)
            a.gate_ws, a.lw_part, a.z, a.z16 = ptr(self._gate_ws), ptr(lw_part), ptr(dec.get("z")), ptr(dec.get("z16"))
            for k0 in range(0, K, kc):
                kcc = min(kc, K - k0)
                a.k0, a.kc = k0, kcc
                _lib.check(self.lib.gccvae_iw_latent(C.byref(a), _stream()), "iw_latent")
                self.engine.iw_decoder_ll(x, b, B, kcc, dec, log_pxz)
                _lib.check(self.lib.gccvae_iw_accumulate(B, kcc, k0, K, ptr(lw_part), ptr(log_pxz), ptr(state), ptr(log_w),
                                                         int(k0 == 0), int(k0 + kcc == K), ptr(est), ptr(ess), _stream()),
                           "iw_accumulate")
        self.last = dict(ess=ess, c=self._c.clone(), log_w=log_w)
        return est

    def test_log_likelihood(self, data_loader, k=100, labelled=False):
        """The `accuracy(data_loader)` counterpart of `log_likelihood`: one gate sample c is drawn and used for every
        batch; returns (mean nats per image, mean nats per pixel value (64 x 64 x 3 = 12288 per image), c).  The means
        weight every image equally (a short last batch counts by its images).  `labelled=True` scores log p(x, y) with
        the loader's labels, otherwise log p(x)."""
        with self._fresh_noise():
            self._gate(self._noise(None, 1, False, 0))
        c = self._c.clone()
        iterator = iter(data_loader.step())
        num_batches = math.ceil(data_loader.n_s / self.train_config["batch_size"])
        total = torch.zeros((), dtype=torch.float64, device=self.device)
        images = 0
        for _ in range(int(num_batches)):
            xs, ys = next(iterator)
            est = self.log_likelihood(xs, ys if labelled else None, k=k, c=c)
            total += est.double().sum()
            images += est.shape[0]
        mean = float(total) / images
        return mean, mean / (64 * 64 * 3), c

    # ---- checkpoints (gated_ccvae.py:146-165, 391-419) ---------------------------------------------------------------
    # file stem -> parameter prefix; inside a file the tensors follow Keras' own order (layer_names x weight_names),
    # which is the order of params.param_specs()
    _H5_FILES = (("encoder_model", "enc."), ("decoder_model", "dec."), ("classifier", "cls."), ("cond_prior", "prior."))

    def load_model(self, param_dir, model_id):
        """gated_ccvae.py:146-165: the four Keras `save_weights` files `{encoder_model,decoder_model,classifier,
        cond_prior}_{model_id}.h5` (read by the pure-Python HDF5 subset reader `h5lite`; Keras layouts = ours: HWIO
        conv kernels, [Cin... ] conv-transpose kernels [kh,kw,Cout,Cin], [in,out] dense kernels) and, in learnable
        mode, `learned_gating_matrix_{model_id}.npy` into mu."""
        from .h5lite import keras_weights
        logger.info("Loading model from {} of model_id {}".format(param_dir, model_id))
        loaded = {}
        for stem, prefix in self._H5_FILES:
            path = os.path.join(param_dir, "{}_{}.h5".format(stem, model_id))
            names = [n for n in self.store.names() if n.startswith(prefix)]
            weights = keras_weights(path)
            if len(weights) != len(names):
                raise ValueError("{}: {} weight tensors, expected {}".format(path, len(weights), len(names)))
            for name, (wname, arr) in zip(names, weights):
                shape = self.store.offsets[name][2]
                if tuple(arr.shape) != tuple(shape):
                    raise ValueError("{}: {} has shape {}, expected {} for {}".format(path, wname, arr.shape, shape, name))
                loaded[name] = arr
        self.store.load_dict(loaded)
        if self.train_config["gate_type"] == "learnable":
            mu_init = load_learned_gating_matrix(param_dir, model_id)
            with torch.no_grad():
                self.store.view("mu").copy_(torch.from_numpy(np.asarray(mu_init, dtype=np.float32)))
            logging.info("Loaded learned mu")

    # Keras layer names of a fresh build of the four models (first instances; `load_weights` matches by order and
    # shape, not by name): (file stem, model name, [(layer name, number of weight tensors)])
    _H5_LAYOUT = (
        ("encoder_model", "encoder", [("conv2d", 2), ("conv2d_1", 2), ("conv2d_2", 2), ("conv2d_3", 2), ("conv2d_4", 2),
                                      ("flatten", 0), ("dense", 2), ("dense_1", 2)]),
        ("decoder_model", "decoder", [("dense_2", 2), ("reshape", 0), ("conv2d_transpose", 2), ("conv2d_transpose_1", 2),
                                      ("conv2d_transpose_2", 2), ("conv2d_transpose_3", 2), ("conv2d_transpose_4", 2)]),
        ("classifier", "classifier", [("my_inference_layer", 2)]),
        ("cond_prior", "conditional__prior", [("my_cond_generation_layer", 1), ("my_cond_generation_layer_1", 1),
                                              ("my_cond_generation_layer_2", 1), ("my_cond_generation_layer_3", 1)]),
    )

    def save_model(self, param_dir, model_id):
        """gated_ccvae.py:391-419: the four `save_weights` files `{encoder_model,decoder_model,classifier,cond_prior}_
        {model_id}.h5` in Keras' HDF5 layout (`h5lite.write_keras_weights`: layer_names / weight_names attributes,
        `<model>/<layer>/kernel:0|bias:0` datasets - readable by `load_model` here; written to the format of the
        reference's own files but not verified against libhdf5, which is not available), and in learnable mode the
        gating matrix exactly as the reference writes it: `.npy` and `.csv` (z1..z18 x label names)."""
        from .h5lite import write_keras_weights
        os.makedirs(param_dir, exist_ok=True)
        d = {k: v.cpu().numpy() for k, v in self.store.to_dict().items()}
        for (stem, model, layout), (_, prefix) in zip(self._H5_LAYOUT, self._H5_FILES):
            tensors = [d[n] for n in self.store.names() if n.startswith(prefix)]
            layers, i = [], 0
            for lname, n in layout:
                kinds = ("kernel:0", "bias:0")[:n]
                layers.append((lname, [("{}/{}/{}".format(model, lname, kind), tensors[i + j])
                                       for j, kind in enumerate(kinds)]))
                i += n
            assert i == len(tensors), (stem, i, len(tensors))
            write_keras_weights(os.path.join(param_dir, "{}_{}.h5".format(stem, model_id)), layers)
        if self.train_config["gate_type"] == "learnable":
            mu = d["mu"]
            np.save(os.path.join(param_dir, "learned_gating_matrix_{}.npy".format(model_id)), mu)
            with open(os.path.join(param_dir, "learned_gating_matrix_{}.csv".format(model_id)), "w") as fh:
                fh.write(gating_matrix_csv(mu))

    # ---- training loop (gated_ccvae.py:313-419) ------------------------------------------------------------------------
    @staticmethod
    def epoch_schedule(perc_supervision, n_sup, n_unsup, batch_size):
        """-> list of booleans, one per batch of an epoch: is this batch supervised?  (gated_ccvae.py:319-357:
        `is_supervised = (i % period_sup_batches == 0) and ctr_sup < sup_batches`.)"""
        if perc_supervision == 1.0:
            sup_batches = batches = math.ceil(n_sup / batch_size)
            period = 1
        elif perc_supervision > 0.0:
            sup_batches = math.ceil(n_sup / batch_size)
            batches = sup_batches + math.ceil(n_unsup / batch_size)
            period = int(batches / sup_batches)
        elif perc_supervision == 0.0:
            sup_batches, batches, period = 0, math.ceil(n_unsup / batch_size), None
        else:
            assert False, "Data frac not correct"
        out, ctr = [], 0
        for i in range(int(batches)):
            sup = period is not None and (i % period == 0) and ctr < sup_batches
            ctr += int(sup)
            out.append(bool(sup))
        return out

    @staticmethod
    def next_gating_temperature(t):
        """gated_ccvae.py:404-406: the per-epoch decay of the gate sampler's temperature (host float, as there)."""
        t *= 0.99
        return t

    def train(self, data_loaders, param_dir, fig_path=None, on_batch=None):
        """gated_ccvae.py:313-419: per epoch the supervised / unsupervised batches are interleaved by
        `epoch_schedule`, every batch is one `train_step`, the epoch ends with the validation accuracy, a
        best-model checkpoint, and (learnable gates) `gating_sampler_temp *= 0.99`; the last model is saved at the
        end.  `data_loaders` = {'sup','unsup','valid'} objects with `.n_s` and `.step()` (utils_data.py).  A NaN in the
        gate sample raises (the reference calls sys.exit(-1), :373-375).  Returns the per-epoch log."""
        cfg = self.train_config
        perc = cfg["perc_supervision"]
        best_val_acc, history = -np.inf, []
        for epoch in range(cfg["n_epochs"]):
            n_sup = data_loaders["sup"].n_s if perc != 0.0 else 0
            n_unsup = data_loaders["unsup"].n_s if perc != 1.0 else 0
            schedule = self.epoch_schedule(perc, n_sup, n_unsup, cfg["batch_size"])
            sup_iter = iter(data_loaders["sup"].step()) if perc != 0.0 else None
            unsup_iter = iter(data_loaders["unsup"].step()) if perc != 1.0 else None
            sup_loss = unsup_loss = None
            c = None
            last = torch.zeros(2, dtype=torch.float32, device=self.device)   # last sup / unsup loss of the epoch
            for i, is_sup in enumerate(schedule):
                xs, ys = next(sup_iter if is_sup else unsup_iter)
                loss, c = self.train_step(xs, ys if is_sup else None, supervised=is_sup)
                # train_step's results live in a ring of RING steps: keep the epoch's last losses in their own buffer
                last[0 if is_sup else 1].copy_(loss)
                if is_sup:
                    sup_loss = last[0]
                else:
                    unsup_loss = last[1]
                if on_batch is not None:
                    on_batch(epoch, i, is_sup, loss, c)
            # one device->host read per epoch instead of per batch (the reference reads loss and c every batch for its
            # progress bar): the NaN check on the gate sample keeps its meaning, it just fires at the epoch end
            if c is not None and bool(torch.isnan(c).any()):
                raise FloatingPointError("gate sample c contains NaN (gated_ccvae.py:373-375)")
            val_acc = self.accuracy(data_loaders["valid"]) if perc else -np.inf
            logger.info("[Epoch %03d] Val Acc %.3f" % (epoch, val_acc))
            if val_acc > best_val_acc:
                logger.info("Saving best model...")
                best_val_acc = val_acc
                self.save_model(param_dir, "best")
            if cfg["gate_type"] == "learnable":
                self.gating_sampler_temp = self.next_gating_temperature(self.gating_sampler_temp)   # (device scalar)
                logger.info("gating_sampler_temp decayed to: %.4f" % self.gating_sampler_temp)
            history.append(dict(epoch=epoch, sup_loss=None if sup_loss is None else float(sup_loss),
                                unsup_loss=None if unsup_loss is None else float(unsup_loss), val_acc=float(val_acc),
                                n_sup=sum(schedule), n_unsup=len(schedule) - sum(schedule),
                                gating_sampler_temp=float(self.gating_sampler_temp)))
        logger.info("Saving last model...")
        self.save_model(param_dir, "last")
        return history

    # ---- data parallel ---------------------------------------------------------------------------------------------------
    def _allreduce_grads(self):
        dp.allreduce_sum_(self._dist, self.store.grad_full, self.store.total + 1)

    def _global_loss(self, loss):
        return dp.global_scalar(self._dist, loss)


def v_mu(learner):
    return learner.store.view("mu")


class _ElboFunction(torch.autograd.Function):
    """sup_loss / unsup_loss as a differentiable function of the flat parameter buffer.  The kernels compute forward and
    backward in one pass, so `forward` already produces d loss / d parameters (all-reduced in data-parallel runs) and
    `backward` only scales it by the incoming gradient - what tape.gradient(loss, trainable_variables) returns in
    gated_ccvae.py:309.  Frozen mu (fixed gate types) gets a zero gradient."""

    @staticmethod
    def forward(ctx, flat, learner, x, y, supervised, noise, k):
        with learner._fresh_noise():
            loss, c = learner._elbo(x, y, supervised, noise, backward=True, k=k)
            learner._allreduce_grads()
        grad = learner.store.grad.clone()
        if not learner.model.mu_trainable:
            learner.store.view("mu", grad).zero_()
        ctx.save_for_backward(grad)
        loss, c = loss.clone(), c.clone()
        ctx.mark_non_differentiable(c)
        return loss, c

    @staticmethod
    def backward(ctx, g_loss, _g_c):
        (grad,) = ctx.saved_tensors
        return g_loss * grad, None, None, None, None, None, None
