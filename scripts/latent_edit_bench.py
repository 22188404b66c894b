"""Throughput of the latent traversal and the pair interpolation on the bf16 engine (the shipped checkpoint, uint8 input
images): Learner.traverse from B = 64 images over all 45 dims x 8 values (23 040 decoded rows per call, three chunks at
the default max_rows = 8192) and Learner.interpolate of 512 pairs x 16 values of t (8 192 rows, one chunk), for both
output dtypes; event, host issue and device time per call, decoded rows/s, the peak device memory of a call, and the
latent kernel (gccvae_gen_latent) alone per 8 192-row chunk for a one-frame call, a label walk, a traversal and a pair.

    python scripts/latent_edit_bench.py [--out result.json]

Times as in scripts/walk_bench.py: CUDA events around back-to-back calls after warm-up; host issue time: the host clock
around the same loop before its synchronise; device time: the same calls enqueued behind a spin kernel long enough to
cover their issue, so that the events see device work only.  Kernel time: CUDA events around `--kernel-launches`
launches behind a spin kernel, on fixed random head pre-activations (the kernel reads nothing else of the encoder)."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gccvae_b200 as G  # noqa: E402
import gccvae_b200._lib as L  # noqa: E402
from likelihood_bench import CKPT, gpu_info, spin, time_calls  # noqa: E402


def device_time(fn, calls, host_s):
    """CUDA events around `calls` calls enqueued behind a spin kernel that outlasts their issue (host_s per call)."""
    torch.cuda.synchronize()
    torch.cuda._sleep(int(max(20e-3, 1.5 * calls * host_s) * 1.9e9))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / calls


def peak_memory(fn, rows, chunk, lrn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return dict(dtype="uint8", peak_allocated_mb=round(torch.cuda.max_memory_allocated() / 2 ** 20, 1),
                allocated_before_call_mb=round(base / 2 ** 20, 1), output_mb=round(rows * 12288 / 2 ** 20, 1),
                decoder_buffers_mb=round(sum(t.numel() * t.element_size() for t in
                                             lrn.engine.dec_bufs(chunk).values()) / 2 ** 20, 1))


def time_call(make, rows, B, calls):
    out = {}
    for dtype in (torch.uint8, torch.float32):
        fn = make(dtype)
        t_ev, t_host = time_calls(fn, calls, warmup=3)
        t_dev = device_time(fn, calls, t_host)
        out[str(dtype).replace("torch.", "")] = dict(
            calls=calls, ms_per_call=round(t_ev * 1e3, 3), host_issue_ms_per_call=round(t_host * 1e3, 3),
            device_ms_per_call=round(t_dev * 1e3, 3), decoded_rows_s=round(rows / t_ev),
            decoded_rows_s_device=round(rows / t_dev), img_s_device=round(B / t_dev))
    return out


def kernel_times(lrn, launches):
    """gen_latent_kernel alone per 8 192-row chunk, one per frame kind."""
    rows = 8192
    g = torch.Generator(device="cuda").manual_seed(1)
    pre = torch.randn(2 * rows, 2, 45, device="cuda", generator=g)      # [row, loc | scale, 45]
    y = torch.randint(0, 2, (rows, 18), device="cuda", generator=g, dtype=torch.int64)
    al = torch.arange(16, dtype=torch.float32, device="cuda") / 15
    dec = lrn.engine.dec_bufs(rows)

    def args(mode, B):
        a = L.GenLatentArgs()
        a.batch, a.mode, a.row0, a.rows = B, mode, 0, rows
        a.loc_pre, a.scale_pre, a.ld_pre = L.ptr(pre), L.ptr(pre) + 45 * 4, 90
        a.gate_ws, a.z16, a.alphas = L.ptr(lrn._gate_ws), L.ptr(dec["z16"]), L.ptr(al)
        return a

    one = args(L.GEN_INTERVENE, rows)                 # intervene(x, y_new): the one-frame call with the most work
    one.y_tgt = L.ptr(y)
    walk = args(L.GEN_INTERVENE, 64)                  # walk of 64 images, 18 labels x 8 values: its first chunk
    walk.n_labels, walk.n_alpha = 18, 8
    walk.labels[:18] = list(range(18))
    trav = args(L.GEN_RECONSTRUCT, 64)                # traversal of 64 images, 45 dims x 8 values: its first chunk
    trav.n_dims, trav.n_alpha = 45, 8
    trav.dims[:45] = list(range(45))
    pair = args(L.GEN_RECONSTRUCT, 512)               # interpolation of 512 pairs x 16 values, all dims
    pair.pair, pair.n_alpha, pair.mix_lo, pair.mix_hi = 1, 16, 0, 45
    st = torch.cuda.current_stream().cuda_stream
    out = {}
    for name, a in (("one_frame_intervene", one), ("walk", walk), ("traverse", trav), ("pair", pair)):
        launch = lambda a=a: L.check(lrn.lib.gccvae_gen_latent(C.byref(a), st), "gen_latent")
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
        t = e0.elapsed_time(e1) / 1e3 / launches
        out[name] = dict(rows=rows, us_per_launch=round(t * 1e6, 2), rows_per_s=round(rows / t))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64, help="images of the traversal")
    ap.add_argument("--values", type=int, default=8, help="values per traversed dim")
    ap.add_argument("--pairs", type=int, default=512)
    ap.add_argument("--ts", type=int, default=16, help="values of t per pair")
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--kernel-launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if min(a.batch, a.values, a.pairs, a.ts, a.calls, a.kernel_launches) < 1:
        ap.error("every count must be >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("latent_edit_bench needs a CUDA device: the numbers it reports are GPU times")
    torch.cuda.set_device(0)
    cfg = dict(gate_type="learnable", gate_subtype=None, mu_init=[[0.0] * 18] * 18, gating_reg=0.2, lr=1e-4,
               gating_init_temp=1.0, batch_size=a.batch)
    lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 0.2, cfg, precision="bf16")
    lrn.load_model(CKPT, "best")
    g = torch.Generator().manual_seed(0)
    x = torch.randint(0, 256, (a.batch, 64, 64, 3), generator=g, dtype=torch.uint8).cuda()
    xa = torch.randint(0, 256, (a.pairs, 64, 64, 3), generator=g, dtype=torch.uint8).cuda()
    xb = torch.randint(0, 256, (a.pairs, 64, 64, 3), generator=g, dtype=torch.uint8).cuda()
    values = torch.linspace(-3.0, 3.0, a.values).tolist()
    ts = [t / (a.ts - 1) if a.ts > 1 else 0.0 for t in range(a.ts)]
    res = dict(gpu=gpu_info(), input="uint8", max_rows=8192)
    # traversal
    rows = a.batch * 45 * a.values
    trav = lambda dtype=torch.uint8: (lambda: lrn.traverse(x, values=values, dtype=dtype))
    mem = peak_memory(trav(), rows, min(8192, rows), lrn)
    res["traverse"] = dict(batch=a.batch, dims=45, values=a.values, decoded_rows=rows, peak_memory=mem,
                           calls=time_call(trav, rows, a.batch, a.calls))
    # interpolation
    rows = a.pairs * a.ts
    interp = lambda dtype=torch.uint8: (lambda: lrn.interpolate(xa, xb, ts=ts, dtype=dtype))
    mem = peak_memory(interp(), rows, min(8192, rows), lrn)
    res["interpolate"] = dict(pairs=a.pairs, ts=a.ts, part="all", decoded_rows=rows, peak_memory=mem,
                              calls=time_call(interp, rows, a.pairs, a.calls))
    res["gen_latent_kernel"] = kernel_times(lrn, a.kernel_launches)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
