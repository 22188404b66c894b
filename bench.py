#!/usr/bin/env python
"""Benchmark of the Gated-CCVAE ELBO training step (BASELINE.json metric: training images/sec of the
supervised + unsupervised ELBO step).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|fp32]
                    [--dump-outputs DIR]

One "step" = one supervised train_step + one unsupervised train_step (forward, backward, gradient
all-reduce, Adam), each on `--batch` images per GPU (default: BASELINE.json configs[1], fixed-inferred
gating from gating_matrix_0.2, batch 1024 per GPU).  Data parallel, weak scaling: every rank processes
its own shard; value = images all ranks processed / max-over-ranks device time.

Prints ONE JSON line (rank 0).  Keys beyond the base contract: roofline, cpu_baseline, e2e, clocks,
gpu_launches.  `--impl reference` times the CPU oracle (the reference cannot run here: it needs
TensorFlow, SURVEY.md F2) on the host cores on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np
import torch

METRIC = "training images/sec (sup+unsup ELBO step)"
UNIT = "images/s"
WORKLOAD = "Gated CCVAE {gate} gating (gating_matrix_{frac}), 64x64x3, 18 attrs, K=100, batch {b} per GPU"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("GCCVAE_PRECISION", "auto"))
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--ref-batch", type=int, default=None,
                    help="batch of the CPU arm (default: --batch, i.e. the same configuration as the GPU arm)")
    ap.add_argument("--cpu-baseline-steps", type=int, default=15,
                    help="timed oracle steps of the cpu_baseline leg (15 x ~0.7 s at batch 1024 = ~10 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    # the other BASELINE.json configs (parity / study cases, not the headline line)
    ap.add_argument("--gate", default="inferred", choices=["one-one", "inferred", "learnable"])
    ap.add_argument("--frac", default="0.2", help="which data/gating_matrix_<frac>.npy initialises mu")
    ap.add_argument("--unsup-per-sup", type=int, default=1, help="unsupervised train_steps per supervised one")
    ap.add_argument("--dp-exchange", default="peer", choices=["peer", "nccl"],
                    help="gradient exchange of the data-parallel step: fused two-shot all-reduce + Adam over NVLink peer "
                         "memory (csrc/dp.cu) or NCCL all-reduce")
    ap.add_argument("--engine-options", default="", help="A/B runs: comma-separated key=value options of the bf16 engine "
                                                          "(fused_chain, wgrad_streams, post_chain_stream)")
    ap.add_argument("--e2e-input", default="uint8", choices=["uint8", "fp32"],
                    help="host image dtype of the headline e2e run (the other one is reported as e2e_alt)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (sup/unsup loss and c) and the parameters after it "
                         "as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.ref_batch is None:
        args.ref_batch = args.batch
    return args


def train_cfg(gate="inferred", frac="0.2"):
    mu = np.load(os.path.join(ROOT, "data", "gating_matrix_{}.npy".format(frac)))
    base = dict(mu_init=mu, gating_reg=0.2, lr=1e-4, batch_size=1024, init_temp=0.1)
    if gate == "learnable":
        return dict(base, gate_type="learnable", gate_subtype=None, gating_init_temp=1.0)
    return dict(base, gate_type="fixed", gate_subtype=gate, gating_init_temp=0.3)


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle in the reference's literal structure (two encoder passes, python K loop)
# ---------------------------------------------------------------------------------------------------
def cpu_oracle_rate(batch, steps, warmup, gate="inferred", frac="0.2"):
    import gccvae_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = train_cfg(gate, frac)
    p = O.init_params(0)
    mu, _ = O.initialise_mu(cfg)
    opt = O.KerasAdam(cfg["lr"])
    x, y, noise = O.make_inputs(batch, k=100)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for sup in (True, False):
            _, g = O.loss_and_grads(p, mu, x, y, noise, cfg, cfg["gating_init_temp"], sup)
            opt.apply(p, g)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    return 2 * batch / (ms / 1e3), ms


def run_reference(args, rank):
    if rank != 0:
        return
    # bounded: one oracle step pair at batch 1024 takes ~0.7 s on 16 cores; at most ~3 minutes of it are timed
    steps = max(1, min(args.steps, int(180 * 1500 / max(1, args.ref_batch)) or 1))
    warmup = max(1, min(args.warmup, 5))
    rate, ms = cpu_oracle_rate(args.ref_batch, steps, warmup, args.gate, args.frac)
    cores = os.cpu_count() or 1
    sample = ("oracle (PyTorch-CPU restatement of the TF reference), sup+unsup step on batch {} per step, {} timed "
              "steps after {} warm-up".format(args.ref_batch, steps, warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(gate=args.gate, frac=args.frac, b=args.batch),
                   "reference_sample_batch": args.ref_batch, "same_config": args.ref_batch == args.batch},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# data-parallel self-check (world > 1): sharded step == whole-batch step, with this repo's fp32 engine on both sides
# ---------------------------------------------------------------------------------------------------
def dp_equivalence_check(G, cfg, dev, rank, world, exchange, b_local=8, K=10):
    """One supervised + one unsupervised fp32 train_step with explicit noise: `world` ranks on their shards of a batch of
    b_local x world images (gradient exchange + Adam through the product's data-parallel path) against ONE device on the
    whole batch.  Returns the relative loss differences and the fraction of parameters that differ by more than 2e-5
    after the two updates (lr 1e-3: a wrong exchange moves every parameter by ~1e-3)."""
    import torch.distributed as dist
    g = torch.Generator().manual_seed(99)
    n = b_local * world
    x = torch.rand(n, 64, 64, 3, generator=g)
    y = (torch.rand(n, 18, generator=g) < 0.5).to(torch.int64)
    noise = dict(eps=torch.randn(n, 45, generator=g), eps_k=torch.randn(K, n, 45, generator=g),
                 U_y=torch.rand(n, 18, generator=g), U1=torch.rand(18, 18, generator=g), U2=torch.rand(18, 18, generator=g))
    sl = slice(rank * b_local, (rank + 1) * b_local)
    shard = dict(eps=noise["eps"][sl], eps_k=noise["eps_k"][:, sl], U_y=noise["U_y"][sl], U1=noise["U1"], U2=noise["U2"])
    c = dict(cfg, lr=1e-3, batch_size=n)
    mk = lambda ex: G.Learner((64, 64, 3), 45, 18, 18, 1000, 1.0, c, device=dev, precision="fp32", seed=1, dp_exchange=ex)
    dpl, ref = mk(exchange), mk("nccl")
    ref._dist, ref.world, ref.rank = None, 1, 0
    out = {"ranks": world, "exchange": "peer" if dpl._peer is not None else "nccl", "batch_per_rank": b_local}
    for sup in (True, False):
        l1, _ = dpl.train_step(x[sl], y[sl] if sup else None, sup, noise=shard, k=K)
        l0, _ = ref.train_step(x, y if sup else None, sup, noise=noise, k=K)
        out["loss_rel_diff_sup" if sup else "loss_rel_diff_unsup"] = abs(float(l1) - float(l0)) / abs(float(l0))
    t = torch.stack([((dpl.store.flat - ref.store.flat).abs() > 2e-5).float().mean(),
                     (dpl.store.flat - ref.store.flat).abs().max()])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out["params_differing_frac"], out["params_max_abs_diff"] = float(t[0]), float(t[1])
    out["ok"] = bool(out["params_differing_frac"] < 0.01 and max(out["loss_rel_diff_sup"], out["loss_rel_diff_unsup"]) < 1e-5)
    return out


def dump_outputs(path, lrn, last):
    """The last timed step's results as float32 .npy files: what its train_steps returned (loss_sup, c_sup, loss_unsup,
    c_unsup) and the parameters it left (params, the flat store of the model, ~4 MB)."""
    os.makedirs(path, exist_ok=True)
    arrays = {"params": lrn.store.flat}
    for kind, (loss, c) in last.items():
        arrays["loss_" + kind], arrays["c_" + kind] = loss, c
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().to(torch.float32).cpu().numpy())


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    import gccvae_b200 as G

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    precision = args.precision
    if precision == "auto":
        precision = "bf16" if os.path.exists(os.path.join(ROOT, "semi-supervised-gated-lt-vae_b200",
                                                           "engine_tc.py")) else "fp32"
    B = args.batch
    cfg = train_cfg(args.gate, args.frac)
    U = max(0, args.unsup_per_sup)
    imgs_per_step = (1 + U) * B
    eopts = {}
    for kv in filter(None, (args.engine_options or os.environ.get("GCCVAE_BENCH_ENGINE_OPTIONS", "")).replace(":", ",").split(",")):
        k_, v_ = kv.split("=")
        eopts[k_] = int(v_) if v_.lstrip("-").isdigit() else v_
    lrn = G.Learner((64, 64, 3), 45, 18, 18, 162770, 0.2, cfg, device=dev, precision=precision, seed=1234,
                    graphs=not args.no_graph, dp_exchange=args.dp_exchange, engine_options=eopts or None)
    dp_check = dp_equivalence_check(G, cfg, dev, rank, world, args.dp_exchange) if world > 1 else None

    # synthetic data: a ring of NBUF different batches (> L2 in total) resident in HBM for `value`,
    # and the same ring in pinned host memory for `e2e`
    # Images are synthetic 8-bit pixels, as CelebA JPEGs decode to (utils_data.py:53-56); the fp32 form is the
    # reference loader's np.float32(img) / 255.0 (utils_data.py:57-59) of the SAME pixels, so both host formats
    # describe identical inputs.
    gen = torch.Generator().manual_seed(1234 + rank)
    NBUF = 4
    host_u8 = [torch.randint(0, 256, (B, 64, 64, 3), generator=gen, dtype=torch.uint8).pin_memory() for _ in range(NBUF)]
    host_x = [(t.to(torch.float32) / 255.0).pin_memory() for t in host_u8]
    host_y = [(torch.rand(B, 18, generator=gen) < 0.5).to(torch.int64).pin_memory() for _ in range(NBUF)]
    # `value`: the batches are resident in HBM in the dataset's native form (uint8 pixels) for the bf16 engine, which
    # normalises inside its first kernel; fp32 (u8/255) for the fp32 engine
    dev_x = [(t if precision == "bf16" else f).to(dev) for t, f in zip(host_u8, host_x)]
    dev_y = [t.to(dev) for t in host_y]

    last = {}   # (loss, c) of the latest supervised / unsupervised train_step, for --dump-outputs

    def step_resident(i):
        j = i % NBUF
        # (the resident ring was written once, before the warm-up: nothing that produces these tensors is pending)
        out = last["sup"] = lrn.train_step(dev_x[j], dev_y[j], True, inputs_ready=True)
        for u in range(U):
            out = last["unsup"] = lrn.train_step(dev_x[(j + 1 + u) % NBUF], None, False, inputs_ready=True)
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lrn.lib.gccvae_reset_launch_count()
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = lrn.lib.gccvae_launch_count()
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, launches = timed(step_resident, args.steps, max(3, args.warmup))
    if args.dump_outputs and rank == 0:
        # now: the returned tensors are ring slots that later steps overwrite, and the e2e runs below train on
        dump_outputs(args.dump_outputs, lrn, last)
    ms_step = ms_total / args.steps
    value = imgs_per_step * world / (ms_step / 1e3)

    # ---- e2e: host buffers in, loss out, every step --------------------------------------------------------
    loss_host = torch.zeros(args.steps + 8).pin_memory()

    def make_e2e(host_imgs):
        def step_e2e(i):
            # the public API call with HOST (pinned) buffers: H2D of x (sup + unsup batch) and y every step, and a
            # D2H read of the step's loss into pinned memory (asynchronous; completed inside the timed region by the
            # closing synchronize, so the host never stalls the pipeline)
            j = i % NBUF
            loss, _ = lrn.train_step(host_imgs[j], host_y[j], True)
            for u in range(U):
                loss, _ = lrn.train_step(host_imgs[(j + 1 + u) % NBUF], None, False)
            loss_host[i % loss_host.numel()].copy_(loss, non_blocking=True)
        return step_e2e

    e2e = {}
    u8_ok = precision == "bf16"     # the fp32 engine converts uint8 on the device too, but is not the bench path
    for kind, imgs, bpp in (("uint8", host_u8, 1), ("fp32", host_x, 4)):
        if kind == "uint8" and not u8_ok:
            continue
        ms_k, _ = timed(make_e2e(imgs), args.steps, 3)
        ms_k /= args.steps
        e2e[kind] = {"value": imgs_per_step * world / (ms_k / 1e3), "unit": UNIT,
                     "h2d_bytes_per_step": (1 + U) * B * 64 * 64 * 3 * bpp + B * 18 * 8, "d2h_bytes_per_step": 4,
                     "ms_per_step": ms_k, "host_image_dtype": kind}
    # the clock sampler runs from the start of the timed `value` region to the end of the (equally loaded) e2e regions:
    # with the driver's 20 steps the value region alone is 24 ms, one or two 20 ms samples
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "timed value region + e2e regions"
    head = args.e2e_input if args.e2e_input in e2e else "fp32"
    alt = [k for k in e2e if k != head]

    # ---- per-kernel timing for the roofline of the dominant kernel ---------------------------------------------
    roof, top = None, None
    if hasattr(lrn.engine, "profile_step"):
        # same process, right after the timed region: every op of 3 eager steps bracketed by CUDA events on the
        # launching stream; the dominant op = largest total device time per step
        prof = lrn.engine.profile_step(lrn, dev_x[0], dev_y[0], steps=3)
        tot = sum(ms * n for ms, n, _ in prof.values())
        order = sorted(prof.items(), key=lambda kv: -kv[1][0] * kv[1][1])
        name, (ms, n, nbytes) = order[0]
        roof = {"bound": "hbm", "kernel": name, "achieved": nbytes / (ms * 1e-3) / 1e9, "unit": "GB/s",
                "bytes_per_launch": nbytes, "ms_per_launch": ms, "launches_per_step": n,
                "share_of_profiled_step": ms * n / tot, "traffic": None}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            roof["traffic"] = traffic.get(name)
        except Exception:
            pass
        top = [{"op": k, "ms": round(v[0], 4), "per_step": v[1], "GB/s": round(v[2] / (v[0] * 1e-3) / 1e9, 1)}
               for k, v in order[:8]]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(gate=args.gate, frac=args.frac, b=B),
                   "step": "1 supervised + {} unsupervised train_step(s) (fwd+bwd+allreduce+Adam)".format(U),
                   "precision": precision, "noise": "in-kernel Philox4x32-10",
                   "images": "synthetic 8-bit pixels (what a CelebA JPEG decodes to); `value`: uint8 batches resident in HBM; "
                             "`e2e`: HOST uint8 batches; both are normalised u8/255 on the device, bit-exactly as the "
                             "reference loader does on the host (utils_data.py:57-59); `e2e_alt`: HOST fp32 batches "
                             "(the reference API's dtype, 4x the PCIe bytes)",
                   "l2": "ring of 4 input batches (201 MB) + ~1 GB of activations per step exceed the 126 MB L2",
                   "parallelism": "dp{}".format(world),
                   "dp_exchange": (None if world == 1 else
                                   ("two-shot all-reduce + Adam in one kernel over NVLink peer memory, inside the step's graph"
                                    if lrn._peer is not None else "NCCL all-reduce between graph replay and Adam"))},
        "e2e": e2e[head],
        "e2e_alt": e2e[alt[0]] if alt else None,
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if dp_check is not None:
        line["dp_check"] = dp_check
    if roof is not None:
        pk = peaks.get("hbm_gbs") if roof["bound"] == "hbm" else peaks.get("bf16_tflops_sustained")
        src = "measured"
        if pk is None:
            pk, src = (6650.0 if roof["bound"] == "hbm" else 1590.0), "fallback"
        roof["peak"], roof["peak_source"] = pk, src
        roof["frac"] = roof["achieved"] / pk
        # the step as a whole against both bounds of the layer-by-layer model (SURVEY.md 8d: 1.21 MB of activation
        # traffic and 120.24 MFLOP per image and training step; one GPU's share of `value`)
        per_gpu = value / world
        hbm_pk = peaks.get("hbm_gbs", 6650.0)
        tc_pk = peaks.get("bf16_tflops_sustained", 1590.0)
        roof["step"] = {
            "images_per_s_per_gpu": per_gpu,
            "hbm": {"bytes_per_image": 1.21e6, "achieved_GBps": per_gpu * 1.21e6 / 1e9, "peak_GBps": hbm_pk,
                    "frac": per_gpu * 1.21e6 / 1e9 / hbm_pk},
            "tensor": {"flop_per_image": 120.24e6, "achieved_TFLOPs": per_gpu * 120.24e6 / 1e12, "peak_TFLOPs": tc_pk,
                       "frac": per_gpu * 120.24e6 / 1e12 / tc_pk},
        }
        line["roofline"] = roof
        line["top_ops"] = top
    if not args.no_cpu_baseline:
        rate, ms = cpu_oracle_rate(args.ref_batch, args.cpu_baseline_steps, 1, args.gate, args.frac)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                                "sample": "oracle sup+unsup step, batch {}, {} timed steps ({:.0f} ms each)".format(
                                    args.ref_batch, args.cpu_baseline_steps, ms)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
