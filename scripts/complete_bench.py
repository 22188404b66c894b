"""Image completion on the bf16 engine with the shipped checkpoint: Learner.complete against the same completion built
from public calls (`reconstruct` + torch.where, the composite in fp32), in the same process.  Inputs: B = 1024 uint8
images the checkpoint generates from random labels (sample=False), each with a centred 24 x 24 hole filled with grey
(128); `iters` in {1, 10}, uint8 and fp32 output.  Per call: event time, host issue time and device time, and the peak
device memory of a call.  Also conv5t alone - gccvae_convt_complete_bf16 (into the x2 blocks, in place) against
gccvae_convt_image_bf16 (fp32 image) - at the same batch, and, for information, how fast the iteration settles: the mean
|change| of the hole pixels between consecutive iterations t - 1 and t, t = 1 .. 20 (t = 0 is the grey fill).

    python scripts/complete_bench.py [--out result.json]

Times as in scripts/latent_edit_bench.py: CUDA events around back-to-back calls after warm-up; host issue time: the host
clock around the same loop before its synchronise; device time: the same calls enqueued behind a spin kernel long enough
to cover their issue, so that the events see device work only."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gccvae_b200 as G  # noqa: E402
import gccvae_b200._lib as L  # noqa: E402
from latent_edit_bench import device_time  # noqa: E402
from likelihood_bench import CKPT, gpu_info, spin, time_calls  # noqa: E402


def public_calls(lrn, x, m4, xf, iters, dtype):
    """the completion from public calls: `iters` reconstruct calls, each followed by the fp32 composite."""
    comp = x
    for t in range(iters):
        img = lrn.reconstruct(comp, dtype=dtype if t == iters - 1 else torch.float32)
        comp = torch.where(m4, xf, img)
    return torch.where(m4, x if dtype == torch.uint8 else xf, img)


def timed(fn, calls, B):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    t_ev, t_host = time_calls(fn, calls, warmup=2)
    t_dev = device_time(fn, calls, t_host)
    return dict(calls=calls, ms_per_call=round(t_ev * 1e3, 3), host_issue_ms_per_call=round(t_host * 1e3, 3),
                device_ms_per_call=round(t_dev * 1e3, 3), img_s_device=round(B / t_dev),
                peak_allocated_mb=round(peak / 2 ** 20, 1), allocated_before_call_mb=round(base / 2 ** 20, 1))


def kernel_times(lrn, B, m, launches):
    """conv5t alone at batch B: the completion kind into the x2 blocks against the fp32 image kind."""
    eng = lrn.engine
    eng.pack_weights()
    g = torch.Generator(device="cuda").manual_seed(2)
    g4 = torch.relu(torch.randn(B, 32, 32, 32, device="cuda", generator=g)).to(torch.bfloat16)
    X2 = torch.zeros(B * 1089 * 24, dtype=torch.bfloat16, device="cuda")
    img = torch.empty(B, 64, 64, 3, dtype=torch.float32, device="cuda")
    mb = eng.complete_begin(None, m)["mask_blocks"]
    wp, bias = L.ptr(eng.wp["dec.conv5t.x2t"]), L.ptr(lrn.store.view("dec.conv5t.b"))
    st = torch.cuda.current_stream().cuda_stream
    kinds = {"convt_complete_bf16": lambda: L.check(lrn.lib.gccvae_convt_complete_bf16(
                 B, L.ptr(g4), wp, bias, L.ptr(mb), L.ptr(X2), st), "convt_complete"),
             "convt_image_bf16_fp32": lambda: L.check(lrn.lib.gccvae_convt_image_bf16(
                 B, L.ptr(g4), wp, bias, L.ptr(img), 0, st), "convt_image")}
    out = {}
    for _ in range(2):      # alternate the two kinds twice; the second round is reported
        for name, launch in kinds.items():
            for _ in range(8):
                launch()
            torch.cuda.synchronize()
            spin()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                launch()
            e1.record()
            torch.cuda.synchronize()
            out[name] = dict(batch=B, launches=launches, us_per_launch=round(e0.elapsed_time(e1) * 1e3 / launches, 2))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--hole", type=int, default=24, help="side of the centred square hole")
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--settle", type=int, default=20, help="iterations of the settling curve")
    ap.add_argument("--kernel-launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if min(a.batch, a.hole, a.calls, a.settle, a.kernel_launches) < 1 or a.hole > 64:
        ap.error("every count must be >= 1 and the hole at most 64")
    if not torch.cuda.is_available():
        raise SystemExit("complete_bench needs a CUDA device: the numbers it reports are GPU times")
    torch.cuda.set_device(0)
    cfg = dict(gate_type="learnable", gate_subtype=None, mu_init=[[0.0] * 18] * 18, gating_reg=0.2, lr=1e-4,
               gating_init_temp=1.0, batch_size=a.batch)
    lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 0.2, cfg, precision="bf16")
    lrn.load_model(CKPT, "best")
    B = a.batch
    g = torch.Generator().manual_seed(0)
    y = (torch.rand(B, 18, generator=g) < 0.5).cuda()
    full = lrn.generate(y, sample=False, dtype=torch.uint8)         # the images the holes are cut into
    lo = (64 - a.hole) // 2
    m = torch.ones(B, 64, 64, dtype=torch.bool, device="cuda")
    m[:, lo:lo + a.hole, lo:lo + a.hole] = False
    m4 = m.unsqueeze(-1)
    x = torch.where(m4, full, torch.full_like(full, 128))
    xf = x.to(torch.float32) / 255.0
    res = dict(gpu=gpu_info(), batch=B, input="uint8", hole="centred {0} x {0}, grey fill".format(a.hole), calls={})
    for iters in (1, 10):
        for dtype in (torch.uint8, torch.float32):
            key = "iters{}_{}".format(iters, str(dtype).replace("torch.", ""))
            fused = timed(lambda: lrn.complete(x, m, iters=iters, dtype=dtype), a.calls, B)
            public = timed(lambda: public_calls(lrn, x, m4, xf, iters, dtype), a.calls, B)
            same = torch.equal(lrn.complete(x, m, iters=iters, dtype=dtype), public_calls(lrn, x, m4, xf, iters, dtype))
            res["calls"][key] = dict(complete=fused, reconstruct_plus_where=public, bitwise_equal=bool(same),
                                     device_saving_ms=round(public["device_ms_per_call"] - fused["device_ms_per_call"], 3),
                                     device_saving_frac=round(1 - fused["device_ms_per_call"] / public["device_ms_per_call"], 4))
    res["conv5t_kernel"] = kernel_times(lrn, B, m, a.kernel_launches)
    # settling of the iteration on the trained model (sample=False): the completion after t iterations is the composite
    # of iteration t, so consecutive calls with iters = t - 1 and t give the change of iteration t
    hole = ~m4.expand(B, 64, 64, 3)
    prev, curve = xf, []
    for t in range(1, a.settle + 1):
        cur = lrn.complete(x, m, iters=t)
        curve.append(round(float((cur - prev)[hole].abs().mean()), 6))
        prev = cur
    res["settling_mean_abs_change_of_hole_pixels"] = dict(iterations=list(range(1, a.settle + 1)), values=curve)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
