"""Throughput of the importance-weighted log-likelihood on the bf16 engine: img/s and decoded rows/s of
Learner.log_likelihood at B = 1024 for K = 1, 10, 100, 1000 (uint8 images, the shipped checkpoint), device and host
time per call, the per-launch time and algorithmic bandwidth of the likelihood kernel (gccvae_convt_ll_bf16), and the
peak device memory of a call at the default max_rows.

    python scripts/likelihood_bench.py [--batch 1024] [--out result.json]

Call times: CUDA events around back-to-back calls after warm-up (the device time of the window, launch gaps included);
host issue time: the host clock around the same loop before its synchronise; device time: the same calls enqueued behind
a spin kernel, so that the events see device work only.  Kernel time: CUDA events around `--kernel-launches` launches
behind a spin kernel at rows = 8192 (kc = 8 decoded rows per source image), rotating over 4 copies of the conv4t
operand (4 x 512 MB > the 126 MB L2, so the reads come from HBM).  Algorithmic bytes: the g4 operand (32x32x32 bf16 =
64 KB per decoded row) + the raw-byte blocks of the source images (33x33x16 = 17 KB per image); the 4 KB weight
operand and the 4-byte likelihood per row are left out."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gccvae_b200 as G  # noqa: E402
import gccvae_b200._lib as L  # noqa: E402

CKPT = os.path.join(ROOT, "tests", "golden", "models", "params_0.2_learnable")
DATASHEET_HBM_GBS = 7700.0


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "nvidia-smi failed"
    except (OSError, subprocess.SubprocessError) as e:
        return "nvidia-smi unavailable ({})".format(e)


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    return DATASHEET_HBM_GBS, "data sheet (MEASURED_PEAKS.json absent)"


def spin():
    torch.cuda._sleep(int(20e-3 * 1.9e9))


def time_calls(fn, calls, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    t_host = time.perf_counter() - t0
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / calls, t_host / calls


def device_time(fn, calls):
    torch.cuda.synchronize()
    spin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--ks", default="1,10,100,1000")
    ap.add_argument("--kernel-launches", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ks = [int(v) for v in a.ks.split(",")]
    if a.batch < 1 or min(ks) < 1:
        ap.error("--batch and every K must be >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("likelihood_bench needs a CUDA device: the numbers it reports are GPU times")
    torch.cuda.set_device(0)
    B = a.batch
    cfg = dict(gate_type="learnable", gate_subtype=None, mu_init=[[0.0] * 18] * 18, gating_reg=0.2, lr=1e-4,
               gating_init_temp=1.0, batch_size=B)
    lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 0.2, cfg, precision="bf16")
    lrn.load_model(CKPT, "best")
    g = torch.Generator().manual_seed(0)
    x = torch.randint(0, 256, (B, 64, 64, 3), generator=g, dtype=torch.uint8).cuda()
    res = dict(gpu=gpu_info(), batch=B, input="uint8", max_rows=8192, calls={})
    # peak memory of one call at the default max_rows, from a clean allocator state (the Learner's own tensors included)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    lrn.log_likelihood(x, k=100)
    torch.cuda.synchronize()
    res["peak_memory"] = dict(k=100, peak_allocated_mb=round(torch.cuda.max_memory_allocated() / 2 ** 20, 1),
                              allocated_before_first_call_mb=round(base / 2 ** 20, 1),
                              decoder_buffers_mb=round(sum(t.numel() * t.element_size() for t in
                                                           lrn.engine.dec_bufs(8192).values()) / 2 ** 20, 1))
    for K in ks:
        calls = max(3, min(50, 2000 // K))
        fn = lambda K=K: lrn.log_likelihood(x, k=K)
        t_ev, t_host = time_calls(fn, calls, warmup=2)
        t_dev = device_time(fn, calls) if K <= 100 else t_ev    # (the host issue of K=1000 hides under its device work)
        res["calls"]["K={}".format(K)] = dict(
            calls=calls, ms_per_call=round(t_ev * 1e3, 3), host_issue_ms_per_call=round(t_host * 1e3, 3),
            device_ms_per_call=round(t_dev * 1e3, 3), img_s=round(B / t_ev), decoded_rows_s=round(B * K / t_ev),
            img_s_device=round(B / t_dev), decoded_rows_s_device=round(B * K / t_dev))
    # the likelihood kernel alone at rows = 8192 (kc = 8)
    eng = lrn.engine
    kc = 8
    rows = B * kc if B * kc <= 8192 else 8192 - 8192 % kc
    src = rows // kc
    lrn.log_likelihood(x, k=kc)
    torch.cuda.synchronize()
    g4s = [torch.rand(rows, 32, 32, 32, device="cuda").mul_(0.5).to(torch.bfloat16) for _ in range(4)]
    out = torch.empty(rows, dtype=torch.float32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    w, bias = L.ptr(eng.wp["dec.conv5t.x2t"]), L.ptr(lrn.store.view("dec.conv5t.b"))
    xb = eng.xb_ptr(eng.bufs(B)["X2"], B)
    launch = lambda i: L.check(eng.lib.gccvae_convt_ll_bf16(rows, kc, L.ptr(g4s[i % 4]), w, bias, xb, 2, L.ptr(out), st),
                               "convt_ll")
    for i in range(8):
        launch(i)
    torch.cuda.synchronize()
    spin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(a.kernel_launches):
        launch(i)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3 / a.kernel_launches
    nbytes = rows * 32 * 32 * 32 * 2 + src * 33 * 33 * 16
    peak, peak_src = hbm_peak()
    res["ll_kernel"] = dict(rows=rows, kc=kc, source_images=src, rotation="4 operand buffers of {:.0f} MB".format(
        rows * 65536 / 1e6), us_per_launch=round(t * 1e6, 2), algorithmic_mb=round(nbytes / 1e6, 2),
        achieved_gbs=round(nbytes / t / 1e9, 1), hbm_peak_gbs=peak, hbm_peak_source=peak_src,
        share_of_hbm_peak=round(nbytes / t / 1e9 / peak, 3))
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
