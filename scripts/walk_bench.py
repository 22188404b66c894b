"""Throughput of the label walk on the bf16 engine: Learner.walk from images at B = 64 (uint8 images, the shipped
checkpoint), all 18 labels, 8 values each (9216 decoded rows per call, two chunks at the default max_rows = 8192), for
both output dtypes; event, host issue and device time per call, decoded rows/s, the peak device memory of a call, and
the latent kernel of the walk (gccvae_gen_latent) alone.

    python scripts/walk_bench.py [--batch 64] [--out result.json]

Times as in scripts/likelihood_bench.py: CUDA events around back-to-back calls after warm-up; host issue time: the host
clock around the same loop before its synchronise; device time: the same calls enqueued behind a spin kernel, so that the
events see device work only.  Kernel time: CUDA events around `--kernel-launches` launches of the first chunk (8192 rows)
behind a spin kernel."""
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
from likelihood_bench import CKPT, device_time, gpu_info, spin, time_calls  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--alphas", type=int, default=8)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--kernel-launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.batch < 1 or a.alphas < 1 or a.calls < 1:
        ap.error("--batch, --alphas and --calls must be >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("walk_bench needs a CUDA device: the numbers it reports are GPU times")
    torch.cuda.set_device(0)
    B, T = a.batch, a.alphas
    cfg = dict(gate_type="learnable", gate_subtype=None, mu_init=[[0.0] * 18] * 18, gating_reg=0.2, lr=1e-4,
               gating_init_temp=1.0, batch_size=B)
    lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 0.2, cfg, precision="bf16")
    lrn.load_model(CKPT, "best")
    g = torch.Generator().manual_seed(0)
    x = torch.randint(0, 256, (B, 64, 64, 3), generator=g, dtype=torch.uint8).cuda()
    alphas = [t / (T - 1) if T > 1 else 0.0 for t in range(T)]
    rows = B * 18 * T
    res = dict(gpu=gpu_info(), batch=B, labels=18, alphas=T, decoded_rows=rows, input="uint8", max_rows=8192,
               calls={})
    # peak memory of one call from a clean allocator state (the Learner's own tensors included), uint8 output
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    lrn.walk(x, alphas=alphas, dtype=torch.uint8)
    torch.cuda.synchronize()
    res["peak_memory"] = dict(dtype="uint8", peak_allocated_mb=round(torch.cuda.max_memory_allocated() / 2 ** 20, 1),
                              allocated_before_first_call_mb=round(base / 2 ** 20, 1),
                              output_mb=round(rows * 12288 / 2 ** 20, 1),
                              decoder_buffers_mb=round(sum(t.numel() * t.element_size() for t in
                                                           lrn.engine.dec_bufs(min(8192, rows)).values()) / 2 ** 20, 1))
    for dtype in (torch.uint8, torch.float32):
        fn = lambda dtype=dtype: lrn.walk(x, alphas=alphas, dtype=dtype)
        t_ev, t_host = time_calls(fn, a.calls, warmup=3)
        t_dev = device_time(fn, a.calls)
        res["calls"][str(dtype).replace("torch.", "")] = dict(
            calls=a.calls, ms_per_call=round(t_ev * 1e3, 3), host_issue_ms_per_call=round(t_host * 1e3, 3),
            device_ms_per_call=round(t_dev * 1e3, 3), decoded_rows_s=round(rows / t_ev),
            decoded_rows_s_device=round(rows / t_dev), img_s_device=round(B / t_dev))
    # the latent kernel alone: the first chunk of a walk from images, on the encoder output the last call left
    eng = lrn.engine
    chunk = min(8192, rows)
    io, dec = eng.latent_io(eng.bufs(B)), eng.dec_bufs(chunk)
    al = torch.tensor(alphas, dtype=torch.float32, device="cuda")
    w = L.GenLatentArgs()
    w.batch, w.mode, w.sample, w.n_labels, w.n_alpha = B, L.GEN_INTERVENE, 0, 18, T
    w.labels[:18] = list(range(18))
    w.alphas, w.row0, w.rows = L.ptr(al), 0, chunk
    w.loc_pre, w.scale_pre, w.ld_pre = io["loc_pre"], io["scale_pre"], io["ld_pre"]
    w.gate_ws, w.z16 = L.ptr(lrn._gate_ws), L.ptr(dec["z16"])
    st = torch.cuda.current_stream().cuda_stream
    launch = lambda: L.check(eng.lib.gccvae_gen_latent(C.byref(w), st), "gen_latent")
    for _ in range(8):
        launch()
    torch.cuda.synchronize()
    spin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.kernel_launches):
        launch()
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3 / a.kernel_launches
    res["gen_latent_kernel"] = dict(rows=chunk, us_per_launch=round(t * 1e3 * 1e3, 2),
                                    rows_per_s=round(chunk / t))
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
