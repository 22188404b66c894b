"""Throughput of the generation path on the bf16 engine: img/s of Learner.generate / reconstruct / intervene at
B = 1024 for fp32 and uint8 output, whether the eager calls are bound by the host's issue, and the per-launch time and
achieved bandwidth of the image kernel (gccvae_convt_image_bf16) from its algorithmic bytes.

    python scripts/generate_bench.py [--batch 1024] [--calls 100] [--warmup 10] [--out result.json]

Model: the shipped trained checkpoint (tests/golden/models/params_0.2_learnable).  Inputs: seeded random uint8 images
and labels.  Call times: CUDA events around `--calls` back-to-back calls (the device time of the window, launch gaps
included); host issue time: the host clock around the same loop before its synchronise; device time: the same calls
enqueued behind a spin kernel, so that the events see device work only.  The calls are host-bound when the issue time
is close to the event time and the device time is clearly shorter.  Kernel time: CUDA events around 200 launches
enqueued behind a spin kernel, rotating over 4 copies of the conv4t output and 4 output buffers (256 MB of operands +
outputs > the 126 MB L2, so the reads come from HBM).  Bytes: the g4
operand (32x32x32 bf16 = 64 KB per image) + the image (12 KB uint8 / 48 KB fp32 per image); the 4 KB weight operand is
left out."""
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


def device_time(fn, calls, chunk=20):
    """device time per call without the host's issue gaps: a spin kernel in front of every `chunk` calls lets the host
    enqueue them first (chunks keep the launch queue short), the events then bracket device work only."""
    tot = 0.0
    for _ in range(calls // chunk):
        torch.cuda.synchronize()
        torch.cuda._sleep(int(20e-3 * 1.9e9))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(chunk):
            fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1) / 1e3
    return tot / (calls // chunk * chunk)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--calls", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--kernel-launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.calls < 100 or a.batch < 1:
        ap.error("--calls must be >= 100 and --batch >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("generate_bench needs a CUDA device: the numbers it reports are GPU times")
    torch.cuda.set_device(0)
    B = a.batch
    cfg = dict(gate_type="learnable", gate_subtype=None, mu_init=[[0.0] * 18] * 18, gating_reg=0.2, lr=1e-4,
               gating_init_temp=1.0, batch_size=B)
    lrn = G.Learner((64, 64, 3), 45, 18, 18, 1000, 0.2, cfg, precision="bf16")
    lrn.load_model(CKPT, "best")
    g = torch.Generator().manual_seed(0)
    x = torch.randint(0, 256, (B, 64, 64, 3), generator=g, dtype=torch.uint8).cuda()
    y = (torch.rand(B, 18, generator=g) < 0.5).long().cuda()
    y_new = 1 - y
    res = dict(gpu=gpu_info(), batch=B, calls=a.calls, warmup=a.warmup, calls_img_s={})
    for dt_name, dt in (("fp32", torch.float32), ("uint8", torch.uint8)):
        for mode, fn in (("generate", lambda: lrn.generate(y, dtype=dt)),
                         ("reconstruct", lambda: lrn.reconstruct(x, dtype=dt)),
                         ("intervene", lambda: lrn.intervene(x, y_new, dtype=dt))):
            t_dev, t_host = time_calls(fn, a.calls, a.warmup)
            t_gpu = device_time(fn, a.calls)
            res["calls_img_s"]["{}/{}".format(mode, dt_name)] = dict(
                img_s=round(B / t_dev), ms_per_call=round(t_dev * 1e3, 4), host_issue_ms_per_call=round(t_host * 1e3, 4),
                device_ms_per_call=round(t_gpu * 1e3, 4), img_s_device_bound=round(B / t_gpu),
                host_bound=bool(t_host >= 0.9 * t_dev and t_gpu < 0.9 * t_dev))
    # the image kernel alone
    eng = lrn.engine
    lrn.reconstruct(x)
    torch.cuda.synchronize()
    g4s = [eng.bufs(B)["dec.conv4t.out"].clone() for _ in range(4)]
    peak, peak_src = hbm_peak()
    res["image_kernel"] = dict(hbm_peak_gbs=peak, hbm_peak_source=peak_src, rotation="4 operand + 4 output buffers")
    st = torch.cuda.current_stream().cuda_stream
    w, bias = L.ptr(eng.wp["dec.conv5t.x2t"]), L.ptr(lrn.store.view("dec.conv5t.b"))
    for dt_name, dt, u8 in (("fp32", torch.float32, 0), ("uint8", torch.uint8, 1)):
        outs = [torch.empty(B, 64, 64, 3, dtype=dt, device="cuda") for _ in range(4)]
        launch = lambda i: L.check(eng.lib.gccvae_convt_image_bf16(B, L.ptr(g4s[i % 4]), w, bias, L.ptr(outs[i % 4]), u8,
                                                                  st), "convt_image")
        for i in range(8):
            launch(i)
        torch.cuda.synchronize()
        torch.cuda._sleep(int(20e-3 * 1.9e9))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.kernel_launches):
            launch(i)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / 1e3 / a.kernel_launches
        nbytes = B * (32 * 32 * 32 * 2 + 64 * 64 * 3 * (1 if u8 else 4))
        res["image_kernel"][dt_name] = dict(us_per_launch=round(t * 1e6, 2), algorithmic_mb=round(nbytes / 1e6, 2),
                                            achieved_gbs=round(nbytes / t / 1e9, 1),
                                            share_of_hbm_peak=round(nbytes / t / 1e9 / peak, 3))
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
