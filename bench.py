#!/usr/bin/env python
"""Benchmark of the hot path: bf16 forward of ViT-B/16 224^2 (BASELINE.json configs[1]), images/sec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 512]            # this repo's fused sm_100a path
    python bench.py --impl reference [...]                                       # UNMODIFIED reference on host cores
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...             # one rank per GPU (weak scaling)
    python bench.py --model vit_l16|vit_h14|navit [--dim-head 80]                # the other BASELINE.json configs
    python bench.py --dump-outputs DIR [...]     # also write the logits of the last timed step to DIR/logits.npy

One "step" = one forward of a synthetic batch per GPU (+ the all-gather of the logits when N > 1).  Prints ONE JSON
line on rank 0 (see DESIGN.md "Measurement" for every field).

Baselines carried by the GPU arm's line (rank 0, N = 1):
  * `cpu_baseline`        the unmodified reference (baseline/_ref, kind "reference") on the host cores, bounded sample;
  * `gpu_eager_baseline`  the unmodified reference's eager bf16 forward on the SAME GPU, same weights, same batch,
                          same CUDA-event protocol (the on-box bar of BASELINE.md section 5), plus the max |logit|
                          difference between it and the fused path.
Both legs need the unmodified reference installed under baseline/_ref/, which is not part of the repository: without
it `gpu_eager_baseline` reports "unavailable" and `cpu_baseline` times the oracle port instead (kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "baseline", "_ref")

VIT_B16 = dict(image_size=224, patch_size=16, num_classes=1000, dim=768, depth=12, heads=12, mlp_dim=3072)
METRIC = "images/sec ViT-B/16 224^2 bf16 fwd"
# BASELINE.json configs[1..4]; the headline metric is ViT-B/16
MODELS = {
    "vit_b16": VIT_B16,
    "vit_l16": dict(image_size=224, patch_size=16, num_classes=1000, dim=1024, depth=24, heads=16, mlp_dim=4096),
    "vit_h14": dict(image_size=224, patch_size=14, num_classes=1000, dim=1280, depth=32, heads=16, mlp_dim=5120),
    "navit": dict(image_size=512, patch_size=16, num_classes=1000, dim=1024, depth=6, heads=16, mlp_dim=4096),
}
PRETTY = {"vit_b16": "ViT-B/16", "vit_l16": "ViT-L/16", "vit_h14": "ViT-H/14", "navit": "NaViT"}
DEFAULT_BATCH = {"vit_b16": 512, "vit_l16": 256, "vit_h14": 128, "navit": 256}


def metric_name(model: str) -> str:
    if model == "navit":
        return "images/sec NaViT packed variable-res (256 img, dim 1024, depth 6) bf16 fwd"
    return METRIC.replace("ViT-B/16", PRETTY[model])


def workload_name(model: str, cfg: dict, batch: int) -> str:
    if model == "navit":
        return ("NaViT forward, BASELINE.json configs[4]: %d images/GPU, H,W = 16*randrange(4,33) (random.seed(rank)), "
                "dim 1024, depth 6, heads 16, mlp 4096, padding-free" % batch)
    tag = {"vit_b16": "configs[1]", "vit_l16": "configs[2] (per-GPU share)", "vit_h14": "configs[3] (per-GPU share)"}
    return "%s 224^2 forward, dim_head %d (BASELINE.json %s)" % (PRETTY[model], cfg.get("dim_head", 64), tag[model])


class stdout_to_stderr:
    """fd-level redirect: library chatter (e.g. NCCL's version banner) must not pollute the one-JSON-line stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    # fallback stated in /opt/skills/guides/B200_PROFILING.md
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def cpu_model_string() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------------------------------
# clocks / power: sample nvidia-smi DURING the timed region
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.index = index
        self.proc = None
        self.path = None

    def start(self) -> None:
        try:
            fd, self.path = tempfile.mkstemp(prefix=f"b200vit_clocks_{self.index}_", suffix=".csv")
            self.f = os.fdopen(fd, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
            if self.path:
                self.f.close()
                os.unlink(self.path)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()          # exact PID we started
        try:
            self.proc.wait(5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as f:
            lines = f.readlines()
        os.unlink(self.path)
        for line in lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "power_w_median": statistics.median(pw), "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------------------
def model_cfg(args) -> dict:
    cfg = dict(MODELS[args.model])
    if args.dim_head != 64:
        cfg["dim_head"] = args.dim_head
    return cfg


def navit_sizes(batch: int, seed: int):
    """SURVEY.md 8d config 5: H, W = 16 * randrange(4, 33) per image."""
    rng = random.Random(seed)
    return [(16 * rng.randrange(4, 33), 16 * rng.randrange(4, 33)) for _ in range(batch)]


def navit_flops(cfg: dict, sizes) -> tuple:
    """(GEMM FLOPs, algorithmic attention FLOPs) of one NaViT forward: 2 x MACs, attention only within an image."""
    D, L, H, mlp, C, p, ncls = cfg["dim"], cfg["depth"], cfg["heads"], cfg["mlp_dim"], 3, cfg["patch_size"], cfg["num_classes"]
    dh = cfg.get("dim_head", 64)
    I = H * dh
    ns = [(h // p) * (w // p) for h, w in sizes]
    T, S = sum(ns), len(ns)
    gemm = T * (2 * C * p * p * D + L * (2 * D * 3 * I + 2 * I * D + 4 * D * mlp) + 2 * D * 2 * I) + S * (2 * I * D + 2 * D * ncls)
    attn = L * sum(4 * H * n * n * dh for n in ns) + sum(4 * H * n * dh for n in ns)
    return float(gemm), float(attn)


def import_reference():
    """The UNMODIFIED reference package installed into baseline/_ref (pip --target, see DESIGN.md); None if absent."""
    if not os.path.isdir(os.path.join(REF_DIR, "vit_pytorch")):
        return None
    sys.dont_write_bytecode = True
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import importlib
    return importlib.import_module("vit_pytorch")


def build_reference_model(model: str, cfg: dict):
    """Reference constructor under torch.manual_seed(0) (same RNG stream as this repo's drop-in), or None."""
    ref = import_reference()
    if ref is None:
        return None
    torch.manual_seed(0)
    if model == "navit":
        from vit_pytorch.na_vit import NaViT as RefNaViT
        return RefNaViT(**cfg).eval()
    return ref.ViT(**cfg).eval()


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference on the host cores (bounded sample)
# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_runner(model: str, cfg: dict, sample: int, dtype: torch.dtype):
    """fn() = one forward of `sample` images through the reference (baseline/_ref) -- or, when that install is
    missing, the oracle port -- on the host.  Returns (fn, kind)."""
    ref_model = build_reference_model(model, cfg)
    kind = "reference"
    if model == "navit":
        sizes = navit_sizes(sample, 0)
        torch.manual_seed(1)
        imgs = [torch.randn(3, h, w).to(dtype) for h, w in sizes]
        if ref_model is None:
            from oracle import navit_oracle as NO
            from oracle import vit_oracle as O
            from vit_pytorch_b200 import NaViT
            torch.manual_seed(0)
            sd = O.upcast(NaViT(**cfg).state_dict(), dtype)
            return (lambda: NO.navit_forward(sd, cfg, [imgs])), "port"
        m = ref_model.to(dtype)
        return (lambda: m(imgs, group_images=True, group_max_seq_len=4096)), kind
    torch.manual_seed(1)
    img = torch.randn(sample, 3, cfg["image_size"], cfg["image_size"]).to(dtype)
    if ref_model is None:
        from oracle import vit_oracle as O
        from vit_pytorch_b200 import ViT
        torch.manual_seed(0)
        sd = O.upcast(ViT(**cfg).state_dict(), dtype)
        return (lambda: O.vit_forward(sd, cfg, img)), "port"
    m = ref_model.to(dtype)
    return (lambda: m(img)), kind


def time_cpu(fn, steps: int, warmup: int) -> float:
    """seconds per forward: `warmup` untimed calls, then the mean of `steps` calls."""
    with torch.inference_mode():
        for _ in range(warmup):
            fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        return (time.perf_counter() - t0) / steps


def cpu_matrix(model: str, cfg: dict, budget_s: float) -> list:
    """BASELINE.md section 4 protocol: fp32 and bf16, B = 16 and 64, all host threads, 1 warm-up + best of 3."""
    out = []
    t_end = time.perf_counter() + budget_s
    for dt_name, dt in (("bf16", torch.bfloat16), ("fp32", torch.float32)):
        for b in (16, 64):
            if time.perf_counter() > t_end:
                out.append({"dtype": dt_name, "batch": b, "skipped": "time budget"})
                continue
            fn, kind = cpu_reference_runner(model, cfg, b, dt)
            with torch.inference_mode():
                fn()
                best = None
                for _ in range(3):
                    t0 = time.perf_counter(); fn(); t = time.perf_counter() - t0
                    best = t if best is None else min(best, t)
                    if time.perf_counter() > t_end:
                        break
            out.append({"dtype": dt_name, "batch": b, "s_per_fwd": best, "images_per_sec": b / best, "kind": kind})
    return out


def run_reference_arm(args, rank: int, world: int) -> None:
    """`--impl reference`: the reference's own CPU implementation of the path (unmodified package from baseline/_ref)
    with every host thread, bf16 (the metric's dtype), a bounded sample per step.  Rank 0 only."""
    if rank != 0:
        return
    cfg = model_cfg(args)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sb = args.cpu_batch
    fn, kind = cpu_reference_runner(args.model, cfg, sb, torch.bfloat16)
    nwarm = max(1, min(args.warmup, 2)) if args.warmup > 0 else 0
    # bounded sample: the whole --steps/--warmup run has to end within a few minutes on whatever host this is (the
    # protocol fixes threads = all cores, where a 16-image forward can take seconds): halve the sample until the
    # estimate from one probe forward fits args.cpu_budget seconds
    with torch.inference_mode():
        fn()
        while sb > 1:
            t0 = time.perf_counter(); fn(); probe = time.perf_counter() - t0
            if probe * (args.steps + nwarm) <= args.cpu_budget:
                break
            sb = max(1, sb // 2)
            fn, kind = cpu_reference_runner(args.model, cfg, sb, torch.bfloat16)
            fn()
    sec = time_cpu(fn, args.steps, nwarm)
    val = sb / sec
    matrix = None if args.no_matrix else cpu_matrix(args.model, cfg, args.matrix_budget)
    src = "baseline/_ref/vit_pytorch (unmodified lucidrains/vit-pytorch 1.23.6)" if kind == "reference" \
        else "oracle port (baseline/_ref missing)"
    line = {
        "impl": "reference", "metric": metric_name(args.model), "value": val, "unit": "images/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(args.model, cfg, args.batch or DEFAULT_BATCH[args.model]),
                   "sample": f"{sb} images per step on the host CPU", "threads": cores, "cpu": cpu_model_string()},
        "cpu_baseline": {"value": val, "unit": "images/sec", "cores": cores, "kind": kind,
                         "sample": f"{src}, bf16, {sb}-image forwards, {args.steps} steps, "
                                   f"torch.set_num_threads({cores}), {cpu_model_string()}",
                         "matrix": matrix},
        "e2e": {"value": val, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
class PackedImages:
    """A list of [3, H, W] image views into ONE contiguous buffer (device, or pinned host), so that a whole
    variable-resolution batch crosses PCIe as a single copy."""

    def __init__(self, sizes, device=None, pinned: bool = False) -> None:
        n = sum(3 * h * w for h, w in sizes)
        self.flat = torch.empty(n, dtype=torch.bfloat16, device=device) if device is not None else \
            (torch.empty(n, dtype=torch.bfloat16).pin_memory() if pinned else torch.empty(n, dtype=torch.bfloat16))
        self.views, o = [], 0
        for h, w in sizes:
            self.views.append(self.flat[o:o + 3 * h * w].view(3, h, w))
            o += 3 * h * w


def run_gpu_arm(args, rank: int, local_rank: int, world: int) -> None:
    import torch.distributed as dist
    from oracle import vit_oracle as O
    from vit_pytorch_b200 import NaViT, ViT, _lib
    from vit_pytorch_b200.parallel import all_gather_logits

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        with stdout_to_stderr():
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()                       # NCCL prints its version banner on the first collective
    if not _lib.device_ok(local_rank):
        raise SystemExit("bench.py: libb200vit.so cannot run on this device: " +
                         _lib.lib().b200vit_last_error().decode())

    is_navit = args.model == "navit"
    B = args.batch or DEFAULT_BATCH[args.model]
    CFG = model_cfg(args)
    torch.manual_seed(0)
    model = (NaViT if is_navit else ViT)(**CFG).eval().to(dev, torch.bfloat16)
    torch.manual_seed(1 + rank)
    if is_navit:
        sizes = navit_sizes(B, rank)
        packed = PackedImages(sizes, device=dev)
        packed.flat.copy_(torch.randn(packed.flat.numel(), device=dev).bfloat16())
        img = packed.views
        tokens = sum((h // 16) * (w // 16) for h, w in sizes)
    else:
        img = torch.randn(B, 3, CFG["image_size"], CFG["image_size"], device=dev).bfloat16()
    with torch.inference_mode():
        assert model.fused_reason(img) is None, model.fused_reason(img)

    def step(x):
        with torch.inference_mode():
            out = model(x)
            return all_gather_logits(out) if world > 1 else out

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_ranks(ms: float) -> list:
        if world == 1:
            return [ms]
        t = torch.zeros(world, device=dev, dtype=torch.float64)
        t[rank] = ms
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    W = max(args.warmup, 3)
    for _ in range(W):
        step(img)
    sync_all()

    # ---- device-resident timing (the `value`) ----
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    try:                                         # the nvidia-smi sampler never outlives the timed region
        if sampler:
            time.sleep(0.3)
        _lib.reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        for _ in range(args.steps):
            out = step(img)
        e1.record()
        torch.cuda.synchronize()
        launches = _lib.launch_count()
        per_rank_ms = all_ranks(e0.elapsed_time(e1))
        ms_total = max(per_rank_ms)
        sync_all()
    finally:
        clocks = sampler.stop() if sampler else None
    value = world * B * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:         # outside the sampled window; `out` is still the last timed step's
        dump_outputs(args.dump_outputs, {"logits": out})

    # ---- per-rank compute without the collective (N > 1): which GPU sets the pace of the coupled step ----
    per_rank_compute_ms = None
    if world > 1:
        sync_all()
        e0.record()
        for _ in range(args.steps):
            with torch.inference_mode():
                model(img)
        e1.record()
        torch.cuda.synchronize()
        per_rank_compute_ms = [m / args.steps for m in all_ranks(e0.elapsed_time(e1))]
        sync_all()

    # ---- the collective on its own (N > 1): CUDA events around `steps` all-gathers of the logits ----
    allgather_ms = None
    if world > 1:
        local_logits = out[:B].contiguous()
        sync_all()
        e0.record()
        for _ in range(args.steps):
            all_gather_logits(local_logits)
        e1.record()
        torch.cuda.synchronize()
        allgather_ms = max(all_ranks(e0.elapsed_time(e1))) / args.steps
        sync_all()

    # ---- end to end through the public API with host buffers (H2D of the batch + D2H of the logits every step) ----
    ncls = CFG["num_classes"]
    host_out = torch.empty(world * B, ncls, dtype=torch.bfloat16).pin_memory()
    if is_navit:
        host_packed = PackedImages(sizes, pinned=True)
        host_packed.flat.copy_(packed.flat)
        dev_bufs = [PackedImages(sizes, device=dev) for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        copied = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        state = {"i": 0}

        def start_copy(slot):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                dev_bufs[slot].flat.copy_(host_packed.flat, non_blocking=True)
                copied[slot].record(copy_stream)

        start_copy(0)

        def e2e_step():
            slot = state["i"] & 1
            torch.cuda.current_stream().wait_event(copied[slot])
            start_copy(slot ^ 1)               # the copy of step i+1 overlaps the forward of step i
            o = step(dev_bufs[slot].views)
            consumed[slot].record(torch.cuda.current_stream())
            host_out.copy_(o, non_blocking=True)
            state["i"] += 1

        h2d_bytes = host_packed.flat.numel() * 2
    else:
        from vit_pytorch_b200.io import DeviceFeeder
        host_img = torch.empty(tuple(img.shape), dtype=torch.bfloat16).pin_memory()
        host_img.copy_(img)
        feeder = DeviceFeeder(tuple(img.shape), torch.bfloat16, dev)

        def e2e_step():
            # every step copies its own batch host -> device (the copy of step i+1 overlaps the forward of step i)
            x = feeder.push(host_img, next_host=host_img)
            o = step(x)
            feeder.done(x)
            host_out.copy_(o, non_blocking=True)

        h2d_bytes = host_img.numel() * 2

    for _ in range(3):
        e2e_step()
    sync_all()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = max(all_ranks(e0.elapsed_time(e1)))
    sync_all()
    e2e = {"value": world * B * args.steps / (ms_e2e / 1e3), "unit": "images/sec",
           "h2d_bytes_per_step": h2d_bytes * world, "d2h_bytes_per_step": host_out.numel() * 2 * world}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the tcgen05 GEMM): CUDA events around every launch of a few more steps ----
    peaks, peak_src = read_peaks()
    nprof = min(args.steps, 5)
    _lib.profile_start()
    for _ in range(nprof):
        with torch.inference_mode():
            model(img)
    rec = _lib.profile_stop()
    by = {}
    for name, meta, ms in rec:
        d = by.setdefault(name, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
        d["ms"] += ms; d["flops"] += meta.get("flops", 0.0); d["bytes"] += meta.get("bytes", 0.0); d["launches"] += 1
    tot_ms = sum(d["ms"] for d in by.values())
    breakdown = {k: {"ms_per_step": v["ms"] / nprof, "share": v["ms"] / tot_ms, "launches_per_step": v["launches"] // nprof,
                     **({"tflops": v["flops"] / v["ms"] / 1e9} if v["flops"] else {}),
                     **({"gbps": v["bytes"] / v["ms"] / 1e6} if v["bytes"] else {})}
                 for k, v in sorted(by.items(), key=lambda kv: -kv[1]["ms"])}
    g = by["gemm"]
    achieved = g["flops"] / g["ms"] / 1e9                     # TFLOP/s over the GEMM launches of the step
    peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))   # kernel timed inside a long step
    # dram traffic of the dominant kernel: only from an ncu capture of THIS round's library (profiles/gemm_traffic.json
    # carries the library version it was taken with); otherwise null
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        if tj.get("lib_version") == int(_lib.lib().b200vit_version()) and tj.get("model", "vit_b16") == args.model:
            traffic = tj.get("dram_bytes_per_launch")
    roofline = {"bound": "tensor", "kernel": "gemm2_kernel (tcgen05 cta_group::2)", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "peak_source": f"{peak_src} sustained",
                "avg_launch_ms": g["ms"] / g["launches"], "launches_per_step": g["launches"] // nprof}
    attn_key = "attention_varlen" if "attention_varlen" in by else ("attention" if "attention" in by else None)
    roofline_attention = None
    if attn_key:
        a = by[attn_key]
        gbps = a["bytes"] / a["ms"] / 1e6
        roofline_attention = {"bound": "hbm", "kernel": attn_key, "achieved": gbps, "peak": float(peaks["hbm_gbs"]),
                              "unit": "GB/s", "frac": gbps / float(peaks["hbm_gbs"]), "traffic": None,
                              "avg_launch_ms": a["ms"] / a["launches"]}

    if is_navit:
        gf, af = navit_flops(CFG, sizes)
        flops_step = gf + af
        extra_cfg = {"tokens_per_gpu": tokens, "gemm_tflop_per_step": gf / 1e12, "attention_tflop_per_step_algorithmic": af / 1e12}
    else:
        flops_step = O.flops_per_image(**CFG) * B
        extra_cfg = {}
    tf = flops_step / (ms_total / args.steps / 1e3) / 1e12

    # ---- on-box GPU bar: the unmodified reference, eager bf16, same weights / batch / protocol ----
    gpu_eager = None
    if world == 1 and not args.no_eager:
        gpu_eager = gpu_eager_baseline(args, CFG, model, img, out, dev, B)

    cpu_baseline = None
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        fn, kind = cpu_reference_runner(args.model, CFG, args.cpu_batch, torch.bfloat16)
        with torch.inference_mode():
            fn()
            t0 = time.perf_counter(); n = 0
            while n < 3 or (time.perf_counter() - t0 < 10.0 and n < 50):
                fn(); n += 1
            dt_s = time.perf_counter() - t0
        cpu_baseline = {"value": args.cpu_batch * n / dt_s, "unit": "images/sec", "cores": cores, "kind": kind,
                        "sample": f"baseline/_ref reference, bf16, {n} forwards of {args.cpu_batch} images, "
                                  f"{cores} threads, {cpu_model_string()}"}

    energy = None
    if clocks and clocks.get("power_w_median"):
        energy = clocks["power_w_median"] * (ms_total / args.steps / 1e3) / B

    line = {
        "metric": metric_name(args.model), "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
        "warmup": W, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(args.model, CFG, B), "batch_per_gpu": B,
                   "global_batch": B * world, "parallelism": f"dp{world}",
                   "l2_policy": "inputs and activations (GBs/step) exceed the 126 MB L2",
                   "ln_mode": os.environ.get("B200VIT_LN_MODE", "fold"),
                   "weights": "random init, torch.manual_seed(0)", **extra_cfg},
        "tflops_per_gpu": tf,
        "frac_of_bf16_burst_peak": tf / float(peaks["bf16_tflops"]),
        "frac_of_bf16_sustained_peak": tf / peak,
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "joules_per_image": energy,
        "per_rank_ms_per_step": [m / args.steps for m in per_rank_ms],
        "per_rank_compute_ms": per_rank_compute_ms, "allgather_ms": allgather_ms,
        "roofline": roofline, "roofline_attention": roofline_attention,
        "cpu_baseline": cpu_baseline, "gpu_eager_baseline": gpu_eager, "breakdown": breakdown,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict) -> None:
    """Each array as float32 `directory/<name>.npy`.  An array larger than its share of DUMP_BYTES keeps a fixed,
    seeded sample of its rows (in order), so that two builds can be compared output for output."""
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        row_bytes = a[0].numel() * 4 if a.dim() > 1 else 4
        if a.numel() * 4 > share:
            keep = max(1, share // row_bytes)
            rows = torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            a = a[rows]
        np.save(os.path.join(directory, name + ".npy"), a.numpy())


def gpu_eager_baseline(args, CFG, model, img, our_out, dev, B):
    """Reference eager bf16 forward on this GPU (cuBLASLt + ATen kernels, what a user of the reference gets today)."""
    ref = build_reference_model(args.model, CFG)
    if ref is None:
        return {"unavailable": "baseline/_ref not installed"}
    try:
        ref = ref.to(dev, torch.bfloat16)
        ref.load_state_dict(model.state_dict())
        if args.model == "navit":
            call = lambda: ref(img, group_images=True, group_max_seq_len=4096)
        else:
            call = lambda: ref(img)
        with torch.inference_mode():
            for _ in range(3):
                ro = call()
            torch.cuda.synchronize()
            n = max(3, min(args.steps, 10))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                ro = call()
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        diff = (ro.float() - our_out[: ro.shape[0]].float()).abs()
        return {"value": B / ms * 1e3, "unit": "images/sec", "ms_per_step": ms, "steps": n,
                "impl": "baseline/_ref vit_pytorch (unmodified), torch eager bf16, inference_mode, same weights and batch",
                "max_abs_logit_diff_vs_fused": float(diff.max()), "mean_abs_logit_diff_vs_fused": float(diff.mean())}
    except Exception as e:  # noqa: BLE001  (the baseline must never take the benchmark down)
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    finally:
        del ref
        torch.cuda.empty_cache()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (weak scaling); 0 = the model's default")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-batch", type=int, default=16, help="images per CPU-baseline forward (bounded sample)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-eager", action="store_true", help="skip the gpu_eager_baseline leg")
    ap.add_argument("--no-matrix", action="store_true", help="reference arm: skip the fp32/bf16 x B=16/64 matrix")
    ap.add_argument("--matrix-budget", type=float, default=60.0, help="seconds the reference arm may spend on the matrix")
    ap.add_argument("--cpu-budget", type=float, default=120.0,
                    help="reference arm: seconds the timed steps may take; the per-step sample is halved until they fit")
    ap.add_argument("--model", default="vit_b16", choices=sorted(MODELS), help="vit_b16 is the headline config")
    ap.add_argument("--dim-head", type=int, default=64, help="ViT-H/14 canonical is 80")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the logits of the last timed step to DIR/logits.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "b200":
            ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
        try:                                     # fail before any GPU work, not after the timed steps
            os.makedirs(args.dump_outputs, exist_ok=True)
        except OSError as e:
            ap.error(f"--dump-outputs {args.dump_outputs}: {e}")
        if not os.access(args.dump_outputs, os.W_OK | os.X_OK):
            ap.error(f"--dump-outputs {args.dump_outputs}: directory is not writable")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world != args.gpus:
        if args.gpus > 1 and world == 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun --nproc-per-node {args.gpus}")
    run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
