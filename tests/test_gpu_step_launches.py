"""GPU: every launch the bf16 step makes, at the batch it ships with, against fp64 recomputed from that launch's own inputs.

The step runs through the public Learner API as it always does, with two changes that do not change what any kernel
computes: everything is issued serially on the current stream (engine.side = None, as EngineTC.profile_step does), and
the engine's `_run` - the one place every kernel call of the engine and of the fused chain goes through - is replaced on
the instance by a recorder.  For each launch it prints the op's name (so that a launch that faults is named in the log),
synchronises, copies the engine buffers the op reads (and the gradient buffer, which the weight / bias gradient kernels
add into), runs the launch, synchronises and copies what it wrote.  tests/launch_reference.py recomputes each launch in
fp64 from those copies and the master weights and bounds every element (see there); a table of the worst
|got - want| / bound per (workload, op) is printed, and every entry must be <= 1.

The set of ops each workload issues is pinned by a literal list: a launch added to the engine later fails here until it
has a reference."""
import pytest
import torch

import gccvae_oracle as O
import launch_reference as R
from helpers import cfg_for

pytestmark = pytest.mark.gpu

ENC_FWD = ["prep_x2", "enc.conv1 fwd", "enc.conv2 fwd", "enc.conv3 fwd", "enc.conv4 fwd", "enc.conv5 fwd"]
DEC_FWD = ["dec.conv2t fwd", "dec.conv3t fwd", "dec.conv4t fwd"]
CONV_BWD = ["dec.conv5t wgrad", "dec.conv5t dgrad",
            "dec.conv4t wgrad", "dec.conv4t bgrad", "dec.conv4t dgrad",
            "dec.conv3t wgrad", "dec.conv3t bgrad", "dec.conv3t dgrad",
            "dec.conv2t wgrad", "dec.conv2t bgrad", "dec.conv2t dgrad",
            "dec.conv1t wgrad", "dec.fc1 wgrad", "enc.heads wgrad",
            "enc.conv5 wgrad", "enc.conv5 dgrad",
            "enc.conv4 wgrad", "enc.conv4 bgrad", "enc.conv4 dgrad",
            "enc.conv3 wgrad", "enc.conv3 bgrad", "enc.conv3 dgrad",
            "enc.conv2 wgrad", "enc.conv2 bgrad", "enc.conv2 dgrad",
            "enc.conv1 wgrad"]
FUSED_OPS = ["pack_weights"] + ENC_FWD + ["chain fwd"] + DEC_FWD + ["dec.conv5t fwd+recon"] + CONV_BWD + ["chain bwd"]
LAYERED_OPS = (["pack_weights"] + ENC_FWD + ["enc.heads fwd", "dec.fc1 fwd", "dec.conv1t fwd"] + DEC_FWD
               + ["dec.conv5t fwd+recon"] + CONV_BWD
               + ["dec.conv1t bgrad", "dec.conv1t dgrad", "dec.fc1 bgrad", "dec.fc1 dgrad", "enc.heads dgrad", "enc.conv5 bgrad"])
LL_OPS = (["pack_weights"] + ENC_FWD + ["enc.heads fwd", "dec.fc1 fwd", "dec.conv1t fwd"] + DEC_FWD
          + ["dec.conv5t fwd ll"])


class LaunchRecorder:
    """serial issue + a snapshot of each launch's own buffers; restores the engine on exit."""

    def __init__(self, lrn):
        self.lrn, self.eng = lrn, lrn.engine
        self.launches = []            # (op, rows, pre, post)
        self.ll_rows, self.ll_out = None, None

    def __enter__(self):
        eng = self.eng
        self._side, self._orig_run, self._orig_iw = eng.side, eng._run, eng.iw_decoder_ll
        eng.side = None
        eng._run = self._run
        eng.iw_decoder_ll = self._iw_decoder_ll
        return self

    def __exit__(self, *exc):
        eng = self.eng
        eng.side = self._side
        del eng._run, eng.iw_decoder_ll       # the instance attributes: back to the class's methods
        return False

    def _iw_decoder_ll(self, x, b, batch, kc, dec, log_pxz):
        """the likelihood's decoder works on batch * kc rows of buffers sized for the largest chunk"""
        self.ll_rows, self.ll_out = batch * kc, log_pxz
        return self._orig_iw(x, b, batch, kc, dec, log_pxz)

    def _buffers(self, tensors):
        ptrs = {t.data_ptr() for t in tensors if t is not None}
        for B, b in self.eng._bufs.items():
            if any(torch.is_tensor(v) and v.data_ptr() in ptrs for v in b.values()):
                return b, B
        for _, d in self.eng._dec_bufs.items():
            if any(v.data_ptr() in ptrs for v in d.values()):
                return d, self.ll_rows
        return None, None

    def _get(self, key, b, rows):
        if key == "grad":
            return self.lrn.store.grad
        if key.startswith("lb:"):
            return self.lrn._latent_bufs(rows)[key[3:]]
        if key == "ll:log_pxz":
            return self.ll_out[:rows]
        if key == "X2":
            return b[key]
        return b[key][:rows]

    def _run(self, what, tensors, rc_fn):
        print("launch:", what, flush=True)
        torch.cuda.synchronize()
        reads, writes, _ = R.OPS.get(what, ((), (), None))
        b, rows = self._buffers(tensors)
        pre = {k: self._get(k, b, rows).clone() for k in reads}
        self._orig_run(what, tensors, rc_fn)
        torch.cuda.synchronize()
        post = {k: self._get(k, b, rows).clone() for k in writes}
        self.launches.append((what, rows, pre, post))


def _learner(mode, frac, fused=True):
    import gccvae_b200 as G
    lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 1.0, cfg_for(mode, frac), precision="bf16",
                    engine_options=dict(fused_chain=fused))
    lrn.store.load_dict(O.init_params(0, trained_like=True))
    return lrn


def _images(B, u8, seed=7):
    """(what the Learner is given, the same images as fp32 in [0, 1]) on the device"""
    g = torch.Generator().manual_seed(seed)
    if u8:
        xi = torch.randint(0, 256, (B, 64, 64, 3), generator=g, dtype=torch.uint8)
        return xi.cuda(), (xi.float() / 255.0).cuda()
    x = torch.rand(B, 64, 64, 3, generator=g).cuda()
    return x, x


def _ctx(lrn, x_raw, x01, **kw):
    store = lrn.store
    names = store.names()
    P = {k: store.view(k).double() for k in names}
    W = {k: store.view(k).to(torch.bfloat16).double() for k in names if k.endswith(".w")}
    grads = lambda flat: {k: store.view(k, flat) for k in names}
    return R.Ctx(W, P, grads, x=x01, x_raw=x_raw, c=lrn._c.clone(), **kw)


def _check(workload, rec, ctx, expected):
    """per-op worst ratio over the recorded launches; prints the table, returns the failures."""
    ops = [op for op, _, _, _ in rec.launches]
    assert sorted(set(ops)) == sorted(set(expected)), (workload, sorted(set(ops) ^ set(expected)))
    unknown = [op for op in set(ops) if op not in R.OPS and op not in R.UNCHECKED]
    assert not unknown, ("launches without a reference", unknown)
    worst = {}
    for op, rows, pre, post in rec.launches:
        if op in R.UNCHECKED:
            continue
        for label, r in R.check_launch(op, pre, post, ctx, rows):
            if r > worst.get(op, ("", -1.0))[1]:
                worst[op] = (label, r)
    rec.launches.clear()
    bad = []
    for op in expected:
        if op in worst:
            label, r = worst[op]
            print("{:<34s} {:<24s} {:8.3f}  {}".format(workload, op, r, label))
            if not r <= 1.0:
                bad.append((op, label, r))
    return bad


def _step(workload, mode, frac, B, K, supervised, u8, fused, plain_too=False):
    lrn = _learner(mode, frac, fused)
    _, y, noise = O.make_inputs(B, k=K)
    x_raw, x01 = _images(B, u8)
    with LaunchRecorder(lrn) as rec:
        loss, _ = lrn.loss_and_grads(x_raw, y, supervised, noise=noise, k=K)
    torch.cuda.synchronize()
    dev = x01.device
    ctx = _ctx(lrn, x_raw, x01, supervised=supervised, K=K, y=y.to(dev), eps=noise["eps"].to(dev),
               eps_k=noise["eps_k"].to(dev), U_y=noise["U_y"].to(dev))
    bad = _check(workload, rec, ctx, FUSED_OPS if fused else LAYERED_OPS)
    extra = None
    if plain_too:
        recorded = (float(loss), lrn.store.grad.clone())
        loss2, _ = lrn.loss_and_grads(x_raw, y, supervised, noise=noise, k=K)
        torch.cuda.synchronize()
        extra = (recorded, (float(loss2), lrn.store.grad.clone()), lrn)
    return bad, extra


@pytest.mark.parametrize("supervised", [True, False])
def test_step_launches_batch1024_u8(supervised):
    """BASELINE.json configs[1] as bench.py runs it: fixed-inferred gate 0.2, B = 1024, K = 100, uint8 images, fused chain;
    the recorded run and a plain run (side streams, no recorder) give the same loss and gradients."""
    name = "B1024 u8 {}".format("sup" if supervised else "unsup")
    bad, (rec, plain, lrn) = _step(name, "inferred", "0.2", 1024, 100, supervised, True, True, plain_too=True)
    assert not bad, bad
    assert abs(rec[0] - plain[0]) <= 1e-6 * abs(plain[0]), (rec[0], plain[0])
    for k in lrn.store.names():
        a, b = lrn.store.view(k, rec[1]), lrn.store.view(k, plain[1])
        den = float(b.abs().max())
        assert float((a - b).abs().max()) <= 1e-5 * den, (k, float((a - b).abs().max()), den)


def test_step_launches_ragged_batch1001():
    """learnable gate 0.5, B = 1001, fp32 images: the last group of images is ragged in every tile shape that packs
    several images, and the chain kernel's last group is partial."""
    bad, _ = _step("B1001 f32 sup learnable", "learnable", "0.5", 1001, 100, True, False, True)
    assert not bad, bad


def test_step_launches_layer_by_layer():
    """fused_chain=False: heads, latent stage, fc1 and conv1t as separate dense GEMMs (gemm_bf16 / gemm_tn)."""
    bad, _ = _step("B1024 f32 sup layered", "inferred", "0.2", 1024, 100, True, False, False)
    assert not bad, bad


@pytest.mark.parametrize("max_rows,chunks", [(8192, [8100, 1900]), (16384, [10000])])
def test_log_likelihood_launches(max_rows, chunks):
    """B = 100, k = 100: chunks of 8100 and 1900 decoder rows (64 M-tiles of 128 and a ragged last one) or one chunk of
    10000 rows (79 M-tiles: conv1t's GEMM takes its 256-column slabs)."""
    lrn = _learner("inferred", "0.2")
    x_raw, x01 = _images(100, False, seed=11)
    with LaunchRecorder(lrn) as rec:
        lrn.log_likelihood(x_raw, k=100, max_rows=max_rows)
        torch.cuda.synchronize()
    assert [r for op, r, _, _ in rec.launches if op == "dec.conv5t fwd ll"] == chunks
    bad = _check("loglik max_rows={}".format(max_rows), rec, _ctx(lrn, x_raw, x01), LL_OPS)
    assert not bad, bad
