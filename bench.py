#!/usr/bin/env python
"""bench.py — SDXL UNet conditioned-forward passes/sec (rank-4 LoRA, 1024 px) on 1..8 B200s.

Workload (BASELINE.json metric; SURVEY.md §8d): SDXL-base UNet, synthetic seeded weights (no checkpoint is reachable
offline), rank-4 alpha-1 LoRA on the `noxattn` + `c3lier` leaf set (346 adaptors, lora_up != 0, multiplier 1), latents
[B,4,128,128] (1024 px), text embeddings [B,77,2048], pooled [B,1280], time ids [1024,1024,0,0,1024,1024], timestep 500.
One *step* = one UNet forward over B conditioned passes per GPU (B = 8: the reference's per-iteration fan-out of
4 predictions x CFG pair, train_lora_xl.py:236-322).

  value     passes/s over all ranks, inputs resident in HBM, CUDA-graph replay of the whole forward, timed with CUDA
            events on the launching stream, max over ranks.
  e2e       the same metric through the public call (`sliders_b200.train_util.predict_noise_xl`, the reference's
            `unet(...)` call site + CFG combine) with HOST (pinned) input buffers: H2D of latents and embeddings and D2H
            of the guided eps are inside the timed region, every step.
  roofline  tensor-bound.  The launches of one forward are recorded while the forward's CUDA graph is captured and
            re-captured per kernel class (gemm_kernel = every Linear / conv; attention; norms; the rest) as graphs of
            their own on the same buffers; each class graph is replayed and timed with CUDA events like the forward.
            achieved = algorithmic FLOPs of the gemm_kernel launches / their time; peak = MEASURED_PEAKS.json
            bf16_tflops_sustained.  (Round 1 bracketed eager launches with events, which counted host launch jitter.)
  configs   the other BASELINE.json configurations (extra keys, the headline is unchanged): SD-1.5 bf16 at
            B in {1, 2, 8} (config 2), the sharded text-slider iteration (config 3, `train`), the rank-8 image-slider
            step (config 4), a bounded sample of the 50-step x 11-scale x batch-16 inference sweep (config 5) and, on the
            host cores, one SD-1.5 text-slider iteration in fp32 (config 1).
  cpu_baseline  the reference's CPU path for the headline workload on the host cores (rank 0, N = 1), bounded sample.
`--impl reference`: times that CPU path alone — the reference's unmodified `train_util.predict_noise_xl` + `lora.py`
hook on the fp32 oracle UNet where /root/reference exists (kind "reference"), else the port of the same code in
oracle/port.py (kind "port"; the GPU box has no /root/reference and diffusers is not installable anywhere here).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_PASS = {"sdxl": 6.761e12, "sd15": 0.803e12}      # SURVEY.md §8d / BASELINE.md §2
FLOPS_LORA = {("sdxl", 4): 0.0189e12, ("sdxl", 8): 0.0378e12, ("sd15", 4): 0.0038e12}
METRIC = "SDXL UNet conditioned-fwd passes/sec (rank-4 LoRA, 1024px)"
UNIT = "passes/s"
LATENT = {"sdxl": 128, "sd15": 64}
CTX_DIM = {"sdxl": 2048, "sd15": 768}
KERNEL_CLASS = {"gemm": "gemm", "conv3x3": "gemm", "attention": "attention", "groupnorm": "norm", "layernorm": "norm"}
DUMP_LIMIT_BYTES = 64 << 20


def host_threads() -> int:
    """CPU threads this process can really use: min(affinity mask, cgroup CPU quota).  os.cpu_count() alone
    reports the host's cores (128 on the GPU boxes) even when the container is throttled to a fraction of them, and
    oversubscribing a quota makes the fp32 oracle several times slower."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts and parts[0] != "max":
                    n = min(n, max(1, int(float(parts[0]) / float(parts[1]) + 0.5)))
            else:
                quota = int(parts[0])
                with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                    period = int(f2.read().split()[0])
                if quota > 0:
                    n = min(n, max(1, int(quota / period + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    env = os.environ.get("SLIDERS_CPU_THREADS")
    if env:
        n = int(env)
    return max(1, min(n, 64))  # MKL/oneDNN fp32 convs stop scaling (and start thrashing) well before 64 threads


def dump_outputs(directory, arrays):
    """--dump-outputs: each output of the last timed step as `<directory>/<name>.npy` in float32, so that two builds run
    with the same arguments (hence the same seeded inputs) can be compared output for output.  When the outputs exceed
    64 MiB in all, each array above an equal share of that is replaced by a fixed, seeded sample of its elements
    (flattened, in index order; the indices depend only on the array's size)."""
    import numpy as np

    total = sum(4 * t.numel() for t in arrays.values())
    cap = DUMP_LIMIT_BYTES // (4 * len(arrays)) if total > DUMP_LIMIT_BYTES else None
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().to("cpu", torch.float32)
        if cap is not None and t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            t = t.reshape(-1)[idx]
        np.save(os.path.join(directory, name + ".npy"), t.numpy())


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"sustained": float(p["bf16_tflops_sustained"]), "burst": float(p["bf16_tflops"]),
                "hbm": float(p["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
    return {"sustained": 1400.0, "burst": 1590.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampler running during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx = float(p[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
def build_product(dev, arch="sdxl", rank=4, seed=0, share=None):
    """UNet (seeded synthetic weights, or the parameters of `share`) + LoRANetwork(noxattn, c3lier) with lora_up != 0."""
    from sliders_b200 import lora as plora
    from sliders_b200 import synthetic
    from sliders_b200.unet import UNet2DConditionModel, UNetConfig

    cfg = UNetConfig.sdxl() if arch == "sdxl" else UNetConfig.sd15()
    if share is not None:
        with torch.device("meta"):
            unet = UNet2DConditionModel(cfg).to(torch.bfloat16)
        unet.load_state_dict(share.state_dict(), assign=True)   # same storage: 5 GB are not duplicated
    else:
        with torch.device(dev):
            unet = UNet2DConditionModel(cfg).to(torch.bfloat16)
        synthetic.init_synthetic_(unet, seed=seed + 1)
    unet.requires_grad_(False)
    unet.eval()
    torch.manual_seed(seed)  # lora_down keeps its kaiming init, drawn from the global generator: same adaptors every run
    saved = list(plora.DEFAULT_TARGET_REPLACE)
    plora.DEFAULT_TARGET_REPLACE += plora.UNET_TARGET_REPLACE_MODULE_CONV  # c3lier (train_lora_xl.py:50-52)
    try:
        net = plora.LoRANetwork(unet, rank=rank, multiplier=1.0, alpha=1.0, train_method="noxattn").to(dev, torch.bfloat16)
    finally:
        del plora.DEFAULT_TARGET_REPLACE[len(saved):]
    synthetic.init_lora_nonzero_(net, seed=seed + 2, up_std=0.02)
    return unet, net


def make_host_inputs(batch, arch="sdxl", seed=0, pin=True):
    g = torch.Generator().manual_seed(seed)
    n = LATENT[arch]
    lat = torch.randn(batch, 4, n, n, generator=g)
    ehs = torch.randn(batch, 77, CTX_DIM[arch], generator=g).to(torch.bfloat16)
    pooled = torch.randn(batch, 1280, generator=g).to(torch.bfloat16)
    tids = torch.tensor([[8.0 * n, 8.0 * n, 0., 0., 8.0 * n, 8.0 * n]] * batch)
    ts = [lat, ehs, pooled, tids]
    if pin and torch.cuda.is_available():
        ts = [t.pin_memory() for t in ts]
    return ts


def timed(fn, steps, warmup, dist_mod=None, sampler=None):
    """ms per call of `fn`, CUDA events on the current stream, barrier + synchronize on both sides, max over ranks."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_mod is not None:
        dist_mod.barrier()
    if sampler is not None:
        sampler.start()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if dist_mod is not None:
        dist_mod.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if dist_mod is not None:
        dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
    return t.item() / steps


def class_timings(unet, call, steps, warmup):
    """Records the C-ABI calls of one forward while its CUDA graph is captured, re-captures them per kernel class and
    times each class graph.  Returns ({class: {"ms", "launches", "flops"}}, kernels per forward)."""
    from sliders_b200 import ops

    ops.record_calls = []
    ops.launch_count = 0
    unet.use_cuda_graph = True
    call()                                   # first graphed call of this shape: warm-up passes + capture
    torch.cuda.synchronize()
    calls, ops.record_calls = ops.record_calls, None
    n_capture_passes = 3                     # _CapturedForward: two eager warm-ups + the captured pass
    launches = ops.launch_count // n_capture_passes
    groups = {}
    for c in calls:
        groups.setdefault(KERNEL_CLASS.get(c[2], "other"), []).append(c)
    out = {}
    for cls, cl in groups.items():
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            ops.replay_calls(cl)
        ms = timed(g.replay, steps, warmup)
        out[cls] = {"ms": ms, "launches": len(cl), "flops": sum(c[3] for c in cl)}
    return out, launches


# ---------------------------------------------------------------------------------------------------- CPU legs
def cpu_pair_call(arch="sdxl", rank=4, seed=0, lora_state=None, unet_state=None):
    """The reference's CPU path for one CFG-pair call of the headline workload: `predict_noise_xl` with the LoRA hook
    live on the fp32 oracle UNet.  Returns (callable -> eps, kind, description)."""
    from oracle import reference_bridge as rb
    from oracle import unet as ounet
    from sliders_b200 import synthetic

    xl = arch == "sdxl"
    cfg = ounet.UNetConfig.sdxl() if xl else ounet.UNetConfig.sd15()
    with torch.device("meta"):
        om = ounet.UNet2DConditionModel(cfg)
    om = om.to_empty(device="cpu")
    if unet_state is not None:   # the kernel path's own (bf16) weights: the device generator draws a different stream
        om.load_state_dict({k: unet_state[k].detach().to("cpu", torch.float32).contiguous() for k, _ in om.named_parameters()},
                           assign=True)
    else:
        om.load_state_dict({k: synthetic.synthetic_tensor(k, p.shape, seed + 1, "cpu")
                            for k, p in om.named_parameters()}, assign=True)
    om.requires_grad_(False)
    om.eval()
    torch.manual_seed(seed)  # the adaptors' kaiming init of lora_down: same weights every run
    if rb.available():
        lora, tu, mu = rb.load("lora"), rb.load("train_util"), rb.load("model_util")
        saved = list(lora.DEFAULT_TARGET_REPLACE)
        lora.DEFAULT_TARGET_REPLACE += lora.UNET_TARGET_REPLACE_MODULE_CONV
        try:
            net = lora.LoRANetwork(om, rank=rank, multiplier=1.0, alpha=1.0, train_method="noxattn")
        finally:
            del lora.DEFAULT_TARGET_REPLACE[len(saved):]
        sched = mu.create_noise_scheduler("ddim")
        predict_xl, predict, kind = tu.predict_noise_xl, tu.predict_noise, "reference"
        what = ("the reference's unmodified trainscripts/textsliders/train_util.py + lora.py (LoRA hook live) on the fp32 "
                "oracle UNet (oracle/unet.py = diffusers 0.20.2 restated; diffusers itself is not installable)")
    else:
        from oracle import ddim as oddim
        from oracle import port

        net = port.LoRAHooks(om, rank=rank, alpha=1.0, c3lier=True)
        sched = oddim.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                    num_train_timesteps=1000, clip_sample=False)
        predict_xl, predict, kind = port.predict_noise_xl, port.predict_noise, "port"
        what = ("oracle/port.py (port of the reference's train_util.py + lora.py hook, pinned against them in "
                "tests/test_oracle.py) on the fp32 oracle UNet; /root/reference is absent on this box")
    synthetic.init_lora_nonzero_(net, seed=seed + 2, up_std=0.02)
    if lora_state is not None:   # the kernel path's adaptor weights, so that the two runs compute the same function
        own = net.state_dict()
        net.load_state_dict({k: lora_state[k].detach().float().cpu().reshape(own[k].shape) for k in own if k in lora_state},
                            strict=False)
    sched.set_timesteps(1000)
    lat, ehs, pooled, tids = make_host_inputs(2, arch, seed=seed, pin=False)
    lat1 = lat[:1].to(torch.bfloat16).float()

    def call():
        with torch.no_grad(), net:
            if xl:
                return predict_xl(om, sched, 500, lat1, ehs.float(), pooled.float(), tids, guidance_scale=3.0)
            return predict(om, sched, 500, lat1, ehs.float(), guidance_scale=3.0)

    return call, kind, what, (lat1, ehs, pooled, tids)


def run_cpu_arm(steps, warmup, threads):
    call, kind, what, _ = cpu_pair_call("sdxl")
    torch.set_num_threads(threads)
    times, eps = [], None
    for i in range(warmup + steps):
        t0 = time.time()
        eps = call()
        if i >= warmup:
            times.append(time.time() - t0)
    return times, kind, what, eps


def cpu_config1(threads):
    """BASELINE config 1: one SD-1.5 text-slider iteration on the host cores, fp32 (timesteps_to fixed to 1: one denoise
    step + 4 CFG-pair predictions = 10 passes forward, one backward, one AdamW step)."""
    from oracle import ddim as oddim
    from oracle import port
    from oracle import unet as ounet
    from sliders_b200 import synthetic

    torch.set_num_threads(threads)
    with torch.device("meta"):
        om = ounet.UNet2DConditionModel(ounet.UNetConfig.sd15())
    om = om.to_empty(device="cpu")
    om.load_state_dict({k: synthetic.synthetic_tensor(k, p.shape, 1, "cpu") for k, p in om.named_parameters()}, assign=True)
    om.requires_grad_(False)
    om.eval()
    net = port.LoRAHooks(om, rank=4, alpha=1.0, c3lier=True)
    net.__exit__()
    sched = oddim.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                num_train_timesteps=1000, clip_sample=False)
    opt = torch.optim.AdamW(net.prepare_optimizer_params(), lr=2e-4)
    g = torch.Generator().manual_seed(3)
    emb = {k: torch.randn(1, 77, 768, generator=g) for k in ("target", "positive", "unconditional", "neutral")}
    lat = torch.randn(1, 4, 64, 64, generator=g)
    t0 = time.time()
    loss = port.text_slider_iteration(om, net, sched, opt, emb, lat, timesteps_to=1, guidance_scale=4.0, action="enhance")
    dt = time.time() - t0
    return {"what": "SD-1.5 text-slider iteration (train_lora.py:155-309) on the host cores, fp32, rank-4 LoRA (150 adaptors), "
                    "512 px, timesteps_to = 1: 10 forward passes + backward-to-LoRA + AdamW; oracle/port.py loop",
            "s_per_iteration": dt, "passes_per_s": 10 / dt, "cores": threads, "loss": float(loss), "kind": "port"}


# ---------------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline forward, e2e call, per-class graphs, SD-1.5 forwards (config 2) and "
                         "the --impl reference arm; configs 3 and 4 time 3 iterations, config 5 one sweep")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8, help="conditioned passes per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=30.0)
    ap.add_argument("--no-train", action="store_true", help="skip the training-iteration timings (configs 3 and 4)")
    ap.add_argument("--no-extra", action="store_true", help="skip BASELINE configs 1, 2 and 5")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each timed path returned to DIR/<name>.npy (float32, rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(min(args.warmup, 1), 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    peaks = load_peaks()
    config = {"workload": f"sdxl_unet_fwd_{args.batch}passes_per_gpu_1024px_lora_r4_noxattn_c3lier",
              "latent": [args.batch, 4, 128, 128], "timestep": 500, "lora": "rank4 alpha1 noxattn+c3lier (346)",
              "parallelism": f"dp{world} (independent passes, weights replicated, no data-path collective)",
              "l2": "working set (5.1 GB bf16 weights + activations) >> 126 MB L2; no flush needed"}

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return
        threads = host_threads()
        times, kind, what, eps = run_cpu_arm(args.steps, args.warmup, threads=threads)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"cpu_guided_eps": eps})
        ms = 1e3 * statistics.mean(times)
        v = 2.0 * 1e3 / ms                       # a CFG-pair call is two conditioned passes
        sample = (f"{len(times)} timed CFG-pair calls (predict_noise_xl, batch 1 = 2 passes each, guidance 3, rank-4 LoRA "
                  f"hook live) of the same SDXL@128x128 workload, fp32, {threads} threads; {what}")
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
                          "steps": len(times), "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
                          "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ our arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the sliders_b200 path has no CPU fallback "
                         "(use --impl reference for the CPU timing)")
    import torch.distributed as dist
    from sliders_b200 import generate, ops, parallel, train_util, trainer
    from sliders_b200.scheduler import create_noise_scheduler

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dm = dist if world > 1 else None
    B = args.batch
    unet, net = build_product(dev, "sdxl", 4)
    lat_h, ehs_h, pooled_h, tids_h = make_host_inputs(B, "sdxl", seed=rank)
    lat, ehs = lat_h.to(dev), ehs_h.to(dev)
    added = {"text_embeds": pooled_h.to(dev), "time_ids": tids_h.to(dev)}
    fwd = lambda: unet(lat, 500, ehs, added_cond_kwargs=added).sample
    dump, last = {}, {}   # --dump-outputs: what the last timed call of each path returned

    def keep(name, fn):
        if not args.dump_outputs:
            return fn

        def step():
            last[name] = fn()
        return step

    def record(name, make):
        if args.dump_outputs:
            dump[name] = make()

    # ---- per-kernel-class graphs (also captures the whole-forward graph used below)
    net.__enter__()  # multiplier = 1 (lora.py:252-254)
    with torch.no_grad():
        classes, launches_per_fwd = class_timings(unet, fwd, args.steps, args.warmup)

        # ---- value: graph replay of the whole forward, inputs resident
        sampler = ClockSampler(local_rank)
        ms_step = timed(keep("sample", fwd), args.steps, args.warmup, dm, sampler)
        clocks = sampler.stop()
        record("sdxl_fwd_sample", lambda: last["sample"].float().cpu())   # graph output buffer: copy before the next replay
    value = world * B / (ms_step * 1e-3)
    gm = classes.get("gemm", {"ms": 0.0, "launches": 0, "flops": 0.0})
    achieved = gm["flops"] / (gm["ms"] * 1e-3) / 1e12 if gm["ms"] > 0 else 0.0
    traffic, traffic_note = None, None
    try:  # per-launch DRAM bytes of the dominant kernel from the committed ncu capture of this workload
        with open(os.path.join(ROOT, "profiles", "r02_dram_b8.json")) as f:
            dj = json.load(f)["per_kernel"]["gemm_kernel"]
        if B == 8:
            traffic = dj["dram_read_bytes_per_launch"] + dj["dram_write_bytes_per_launch"]
            traffic_note = dj.get("note")
    except (OSError, KeyError, ValueError):
        pass
    sum_ms = sum(c["ms"] for c in classes.values())
    roofline = {"bound": "tensor", "kernel": "gemm_kernel (tcgen05 GEMM / implicit-GEMM conv)",
                "achieved": achieved, "peak": peaks["sustained"], "unit": "TFLOP/s",
                "frac": achieved / peaks["sustained"], "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": peaks["source"], "launches": gm["launches"],
                "avg_launch_us": 1e3 * gm["ms"] / max(gm["launches"], 1),
                "share_of_step": gm["ms"] / ms_step,
                "breakdown_ms": {k: round(v["ms"], 3) for k, v in sorted(classes.items())},
                "breakdown_sum_ms": round(sum_ms, 3),
                "how": "per-class CUDA graphs re-captured from the forward's recorded launches, CUDA-event timed "
                       f"({args.steps} replays each)",
                "whole_forward_frac": (value / world) * (FLOPS_PER_PASS["sdxl"] + FLOPS_LORA[("sdxl", 4)]) / 1e12 / peaks["sustained"]}

    # ---- e2e: public API, host buffers, H2D + D2H inside the timed region
    sched = create_noise_scheduler("ddim")
    sched.set_timesteps(1000)
    half = max(B // 2, 1)
    eps_host = torch.empty(half, 4, 128, 128, dtype=torch.float32).pin_memory()

    def e2e_step():
        # CFG-pair call exactly like the trainers': latents [half], embeddings [2*half] (uncond ; cond)
        l_d = lat_h[:half].to(dev, non_blocking=True)
        e_d = ehs_h[:2 * half].to(dev, non_blocking=True)
        p_d = pooled_h[:2 * half].to(dev, non_blocking=True)
        t_d = tids_h[:2 * half].to(dev, non_blocking=True)
        eps = train_util.predict_noise_xl(unet, sched, 500, l_d, e_d, p_d, t_d, guidance_scale=3.0)
        eps_host[:half].copy_(eps, non_blocking=True)

    with torch.no_grad():
        e2e_ms = timed(e2e_step, args.steps, args.warmup, dm)
    record("e2e_guided_eps", lambda: eps_host[:half].clone())
    h2d = (lat_h[:half].numel() * 4 + ehs_h[:2 * half].numel() * 2 + pooled_h[:2 * half].numel() * 2
           + tids_h[:2 * half].numel() * 4)
    e2e = {"value": world * 2 * half / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": eps_host[:half].numel() * 4, "ms_per_step": e2e_ms,
           "api": "sliders_b200.train_util.predict_noise_xl (CFG pair, guidance 3) with pinned host buffers"}

    extra = {}
    # ---- BASELINE config 5 (N = 1): inference sweep, 50 DDIM steps, batch 16 (32 passes per step), slider scales
    if world == 1 and not args.no_extra:
        scales = (-5.0, 5.0)
        g5 = torch.Generator().manual_seed(5)
        lat16 = torch.randn(16, 4, 128, 128, generator=g5).to(dev, torch.bfloat16)
        pe = torch.randn(32, 77, 2048, generator=g5).to(dev, torch.bfloat16)
        ae = torch.randn(32, 1280, generator=g5).to(dev, torch.bfloat16)
        at = torch.tensor([[1024., 1024., 0., 0., 1024., 1024.]] * 32, device=dev)
        s5 = create_noise_scheduler("ddim")
        sweep = lambda sc, n: generate.scale_sweep(unet, net, s5, lat16, pe, ae, at, scales=sc, num_inference_steps=n,
                                                   guidance_scale=5.0, start_noise=750)
        with torch.no_grad():
            sweep((1.0,), 2)                 # captures the two 32-pass graphs (adaptors gated off / on)
            ms5 = timed(keep("sweep", lambda: sweep(scales, 50)), 1, 0)
        record("config5_sweep_latents", lambda: torch.stack([x.float().cpu() for x in last["sweep"]]))
        per_scale_s = ms5 * 1e-3 / len(scales)
        extra["config5_inference_sweep"] = {
            "what": "eval denoise loop (generate_images_xl.py:325-364): batch 16, CFG 5, 50 DDIM steps, slider gated on "
                    "t <= 750; timed sample = scales (-5, +5) of the 11 of the sweep (-5..+5), same graphs serve every scale",
            "images_per_s": 16 / per_scale_s, "s_per_scale": per_scale_s, "full_sweep_s_extrapolated": 11 * per_scale_s,
            "passes_per_s": 32 * 50 / per_scale_s,
            "frac_of_sustained": 32 * 50 / per_scale_s * (FLOPS_PER_PASS["sdxl"] + FLOPS_LORA[("sdxl", 4)]) / 1e12 / peaks["sustained"]}
        del lat16, pe, ae, at
    net.__exit__(None, None, None)

    # ---- training paths: BASELINE config 3 (text slider, one condition per GPU + one LoRA-grad all-reduce) and
    # config 4 (image slider, rank 8, +scale / -scale on rank parity); whole iterations through sliders_b200.trainer
    train = None
    if not args.no_train:
        net.requires_grad_(True)
        # more than 4 GPUs: independent sliders side by side, 4 ranks each (the iteration does not shard further)
        sgroup, sidx, n_sliders = parallel.slider_groups(4) if world > 4 else (None, 0, 1)
        parallel.broadcast_lora_params(net, sgroup)
        opt = train_util.get_optimizer("AdamW")(net.prepare_optimizer_params(), lr=2e-4)
        gtr = torch.Generator().manual_seed(77 + sidx)
        mk = lambda: trainer.PromptEmbedsXL(torch.randn(1, 77, 2048, generator=gtr).to(dev, torch.bfloat16),
                                            torch.randn(1, 1280, generator=gtr).to(dev, torch.bfloat16))
        unc, tgt, pos = mk(), mk(), mk()
        pair = trainer.PromptEmbedsPair(torch.nn.MSELoss(), tgt, pos, unc, unc,
                                        trainer.PromptSettings(guidance_scale=4.0, resolution=1024, batch_size=1,
                                                               action="enhance"))
        tsched = create_noise_scheduler("ddim")
        state = {"it": 0, "loss": None}

        def text_it():
            state["loss"] = trainer.text_slider_step_xl(unet, net, tsched, opt, None, pair, timesteps_to=25, device=dev,
                                                        weight_dtype=torch.bfloat16, group=sgroup,
                                                        generator=torch.Generator().manual_seed(1000 + state["it"]))
            state["it"] += 1

        n_it = 3
        it_ms = timed(text_it, n_it, 1, dm)
        record("config3_text_slider_loss", lambda: torch.tensor([float(state["loss"])]))
        parallel.assert_replicas_equal(list(net.parameters()), sgroup)
        passes = 2 * (25 + 4)  # CFG pairs: 25 denoise steps + positive / neutral / unconditional / target
        gw = world // n_sliders  # ranks per slider
        train = {"what": "BASELINE config 3 — text-slider iteration, SDXL 1024 px, batch 1, rank-4 LoRA "
                         "(train_lora_xl.py:162-356): 25 DDIM denoise steps (guidance 3) + 4 CFG-pair predictions + "
                         "backward-to-LoRA + AdamW(692 tensors)",
                 "ms_per_iteration": it_ms, "iterations_timed": n_it, "passes_per_iteration": passes,
                 "sliders_in_parallel": n_sliders, "ranks_per_slider": gw,
                 "iterations_per_s": n_sliders / (it_ms * 1e-3),
                 "passes_per_s": n_sliders * passes / (it_ms * 1e-3), "loss": float(state["loss"]),
                 "replicas_equal_after": True,
                 "sharding": ("single GPU" if world == 1 else
                              (f"{n_sliders} independent sliders x {gw} ranks; within a slider: " if n_sliders > 1 else "") +
                              f"denoise CFG-split over rank parity (1 all-gather of 64 KiB per step), target prediction on rank "
                              f"{gw - 1}, frozen predictions over ranks 0..{max(gw - 2, 0)}, 1 LoRA-grad all-reduce")}
        net.requires_grad_(False)
        opt = None
        unet.reset_graphs() if hasattr(unet, "reset_graphs") else None

        # config 4: a rank-8 network on a second module tree that shares the 5 GB of UNet parameters
        unet8, net8 = build_product(dev, "sdxl", 8, share=unet)
        unet8.use_cuda_graph = True
        net8.requires_grad_(True)
        parallel.broadcast_lora_params(net8)
        opt8 = train_util.get_optimizer("AdamW")(net8.prepare_optimizer_params(), lr=2e-4)
        g4 = torch.Generator().manual_seed(4)
        x_low = torch.randn(1, 4, 128, 128, generator=g4)
        x_high = x_low + 0.3 * torch.randn(1, 4, 128, 128, generator=g4)
        st4 = {"l": None}

        def image_it():
            st4["l"] = trainer.image_slider_step_xl(unet8, net8, tsched, opt8, None, pair, x_low, x_high, 2.0,
                                                    timesteps_to=20, seed=4, device=dev, weight_dtype=torch.bfloat16)

        im_ms = timed(image_it, n_it, 1, dm)
        record("config4_image_slider_losses", lambda: torch.tensor([float(x) for x in st4["l"]]))
        parallel.assert_replicas_equal(list(net8.parameters()))
        extra["config4_image_slider"] = {
            "what": "BASELINE config 4 — image-slider step, SDXL, rank-8 LoRA, paired synthetic latents [1,4,128,128] with shared "
                    "noise (train_lora-scale-xl.py:311-375): 2 grad-carrying CFG-pair predictions (+scale / -scale), 2 "
                    "backward passes accumulated, AdamW",
            "ms_per_step": im_ms, "steps_timed": n_it, "loss_high": float(st4["l"][0]), "loss_low": float(st4["l"][1]),
            "replicas_equal_after": True,
            "sharding": "single GPU" if world == 1 else "+scale prediction on even ranks, -scale on odd ranks, 1 LoRA-grad "
                                                        "all-reduce (17.3 MB); batch 1 leaves ranks >= 2 idle"}
        del unet8, net8, opt8
    unet.use_cuda_graph = False

    # ---- BASELINE config 2 (N = 1): SD-1.5, rank 4, 512 px, bf16, B in {1, 2, 8}
    if world == 1 and not args.no_extra:
        u15, n15 = build_product(dev, "sd15", 4)
        u15.use_cuda_graph = True
        rows = {}
        with torch.no_grad(), n15:
            for b in (1, 2, 8):
                l15, e15, _, _ = make_host_inputs(b, "sd15", seed=b, pin=False)
                l15, e15 = l15.to(dev), e15.to(dev)
                ms15 = timed(keep("sd15", lambda: u15(l15, 500, e15).sample), args.steps, args.warmup)
                record(f"config2_sd15_fwd_sample_B{b}", lambda: last["sd15"].float().cpu())
                pps = b / (ms15 * 1e-3)
                rows[f"B{b}"] = {"ms_per_forward": ms15, "passes_per_s": pps,
                                 "frac_of_sustained": pps * (FLOPS_PER_PASS["sd15"] + FLOPS_LORA[("sd15", 4)]) / 1e12 / peaks["sustained"]}
        extra["config2_sd15_bf16"] = {"what": "SD-1.5 UNet forward, rank-4 LoRA (150 adaptors), latents [B,4,64,64], CUDA-graph "
                                              "replay; 100 % of sustained = 1775 passes/s", **rows}
        del u15, n15

    # ---- CPU legs (rank 0, N == 1 only): the headline workload's CPU baseline + BASELINE config 1
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        torch.set_num_threads(threads)
        t0 = time.time()
        call, kind, what, (lat1, ehs2, pooled2, tids2) = cpu_pair_call("sdxl", lora_state=net.state_dict(),
                                                                        unet_state=unet.state_dict())
        eps_cpu = call()                      # warm-up
        times = []
        while not times or (time.time() - t0 < args.cpu_seconds and len(times) < 3):
            t1 = time.time()
            eps_cpu = call()
            times.append(time.time() - t1)
        # parity of the kernel path against this very CPU run (same weights, same LoRA, same inputs, same call)
        net.set_lora_slider(1.0)   # the config-5 sweep above leaves its last slider scale behind
        net.__enter__()
        with torch.no_grad():
            got = train_util.predict_noise_xl(unet, sched, 500, lat1.to(dev), ehs2.to(dev), pooled2.to(dev),
                                              tids2.to(dev), guidance_scale=3.0)
        net.__exit__(None, None, None)
        rel = ((got.float().cpu() - eps_cpu).norm() / eps_cpu.norm()).item()
        dt = statistics.mean(times)
        cpu_baseline = {"value": 2.0 / dt, "unit": UNIT, "cores": threads, "kind": kind,
                        "sample": f"{len(times)} timed (+1 warm-up) CFG-pair calls (predict_noise_xl, batch 1 = 2 passes, guidance "
                                  f"3, LoRA hook live) of the same SDXL@128x128 workload, fp32, {threads} torch threads, "
                                  f"{time.time() - t0:.0f}s wall incl. build; {what}",
                        "eps_rel_rms_kernels_vs_this_cpu_run": rel}
        del call
        if not args.no_extra:
            extra["config1_sd15_cpu_iteration"] = cpu_config1(threads)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_fwd * args.steps,
                "launches_per_step": launches_per_fwd, "roofline": roofline, "cpu_baseline": cpu_baseline,
                "train": train, "configs": extra}
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dump)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
