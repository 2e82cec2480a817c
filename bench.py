#!/usr/bin/env python
"""Headline benchmark: clips/sec of one SlowFast-8x8-R50 training step on N B200s (BASELINE.json configs[1]), with the
other configs of the metric (MViTv2-S, X3D-M, MaskFeat-S, MaskFeat on MViTv2-B 32x224x224) as secondary legs.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the UNMODIFIED reference (oracle/_ref) on the box's host cores
    python bench.py ... --dump-outputs DIR   # also write the headline leg's last timed step's outputs as DIR/*.npy

A step = zero_grad -> forward (engine kernels) -> loss -> backward (engine kernels) -> [one NCCL all-reduce of the flat
gradient bucket when N > 1] -> optimizer step, on the recipe's per-GPU batch of synthetic Kinetics-shaped input, random
init, parity mode (split-bf16 operands, fp32 accumulate / storage) unless --nsplit 1.  Rank 0 prints ONE JSON line;
DESIGN.md "Measurement" describes every field.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# name -> (preset, per-GPU batch of the published recipe, forward GFLOP per clip (SURVEY.md 8d), ideal fwd MB per clip)
LEGS = {
    "slowfast": dict(preset="SLOWFAST_8x8_R50", batch=8, gflop=100.62, mb=571.8, opt="sgd", seed=1234,
                     what="SlowFast-8x8-R50 (configs/Kinetics/SLOWFAST_8x8_R50.yaml) train step: fwd + CE loss + bwd + "
                          "grad all-reduce (N>1) + SGD-nesterov, 32x224x224 fast / 8x224x224 slow, random init"),
    "mvitv2_s": dict(preset="MVITv2_S_16x4", batch=4, gflop=128.45, mb=647.0, opt="adamw", seed=4321,
                     what="MViTv2-S 16x4 (configs/Kinetics/MVITv2_S_16x4.yaml) train step, drop-path 0.2 + head dropout "
                          "0.5 on, AdamW, 16x224x224"),
    "x3d_m": dict(preset="X3D_M", batch=16, gflop=9.47, mb=365.6, opt="sgd", seed=5321,
                  what="X3D-M (configs/Kinetics/X3D_M.yaml) train step, head dropout 0.5 on, SGD-nesterov, 16x224x224"),
    "maskfeat_s": dict(preset="MVITv2_S_16x4_MaskFeat_PT", batch=4, gflop=173.0, mb=None, opt="adamw", seed=6321,
                       what="MaskFeat pre-training step on MViTv2-S (configs/masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml): "
                            "mask-token encoder fwd + HOG targets + MultipleMSELoss + bwd + AdamW, 40 % cube mask"),
    "maskfeat_b": dict(preset="MVITv2_B_32x3_MaskFeat_PT", batch=2, gflop=None, mb=None, opt="adamw", seed=7321,
                       what="BASELINE config 5: MaskFeat pre-training step on MViTv2-B 32x224x224 (MVIT block of "
                            "configs/Kinetics/MVITv2_B_32x3.yaml composed with the masked_ssl MaskFeat recipe, SURVEY 3.5)"),
}


TORCH_OPTIM = False  # --torch-optim


def host_threads() -> int:
    """Threads of the CPU legs: the cores this process may run on (cgroup / affinity mask), at most 64.  torchrun exports
    OMP_NUM_THREADS=1, so torch's own default is NOT consulted: the count is set explicitly with set_num_threads."""
    try:
        allowed = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        allowed = os.cpu_count() or 1
    return max(1, min(allowed, 64))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tflops_burst=p["bf16_tflops"],
                    tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback")


def load_traffic():
    """DRAM bytes per launch of each kernel class from the committed ncu pass (profiles/*traffic*.json, written by
    tests/probes/summarize_traffic.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum`)."""
    path = os.path.join(ROOT, "profiles", "r2_traffic_summary.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------ the reference itself
REF_YAML = {"SLOWFAST_8x8_R50": "Kinetics/SLOWFAST_8x8_R50.yaml", "MVITv2_S_16x4": "Kinetics/MVITv2_S_16x4.yaml",
            "X3D_M": "Kinetics/X3D_M.yaml"}


def reference_model(preset: str, overrides=()):
    """The UNMODIFIED reference module (slowfast.models.build_model on the reference's own yaml) from oracle/_ref (copied
    there by build()) through oracle/refshim.py.  Returns (cfg, model) or raises if no reference tree exists."""
    from oracle import refshim
    if not refshim.reference_available():
        raise RuntimeError("no reference tree (build() copies it into oracle/_ref when a checkout is readable)")
    cfg = refshim.load_cfg(REF_YAML[preset], list(overrides))
    return cfg, refshim.build_reference_model(cfg)


def synthetic_batch(cfg, batch: int, seed: int):
    """randn clips packed per pathway (datasets/utils.py:78 pack_pathway_output) + integer labels (SURVEY.md 8d)."""
    g = torch.Generator().manual_seed(seed)
    T = cfg.DATA.NUM_FRAMES
    clip = torch.randn(batch, 3, T, cfg.DATA.TRAIN_CROP_SIZE, cfg.DATA.TRAIN_CROP_SIZE, generator=g)
    if cfg.MODEL.ARCH == "slowfast":
        idx = torch.linspace(0, T - 1, T // cfg.SLOWFAST.ALPHA).long()
        x = [clip.index_select(2, idx).contiguous(), clip]
    else:
        x = [clip]
    y = torch.randint(0, cfg.MODEL.NUM_CLASSES, (batch,), generator=g)
    return x, y


def time_reference_cpu(preset: str, batch: int, steps: int, warm: int, budget_s: float):
    """fwd + CE + bwd of ``batch`` clips through the reference's own nn.Module on the host cores (fp32 ATen CPU kernels)."""
    import torch.nn.functional as F
    threads = host_threads()
    torch.set_num_threads(threads)
    cfg, model = reference_model(preset, ["MODEL.DROPOUT_RATE", 0.0] + (["MVIT.DROPPATH_RATE", 0.0] if "MVIT" in preset else []))
    model.train()
    x, y = synthetic_batch(cfg, batch, 1234)

    def one():
        model.zero_grad(set_to_none=True)
        F.cross_entropy(model([t.clone() for t in x]), y).backward()

    for _ in range(warm):
        one()
    n, t0 = 0, time.perf_counter()
    while n < steps and (n < 1 or time.perf_counter() - t0 < budget_s):
        one()
        n += 1
    dt = (time.perf_counter() - t0) / n
    return dict(clips_per_s=batch / dt, ms_per_step=dt * 1e3, steps=n, threads=threads, batch=batch)


def reference_arm(args):
    """``--impl reference``: the reference's OWN CPU implementation of the path (its nn.Conv3d / BatchNorm3d / ... modules,
    unmodified, from oracle/_ref) on this box's host cores, all the threads the process may use, on the same workload
    (SlowFast-8x8-R50 train step, the same per-step batch); steps are bounded so that the run ends within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    leg = LEGS["slowfast"]
    steps, warm = max(1, min(args.steps, 3)), 1
    try:
        r = time_reference_cpu(leg["preset"], args.batch, steps, warm, budget_s=150.0)
        kind = "reference"
    except RuntimeError as e:
        print(json.dumps(dict(impl="reference", unavailable=str(e)[:200])), flush=True)
        return
    v = r["clips_per_s"]
    line = dict(metric="clips/sec (fwd+bwd) SlowFast-8x8-R50", value=v, unit="clips/s", n_gpus=args.gpus, steps=r["steps"],
                warmup=warm, ms_per_step=r["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", impl="reference",
                config=dict(workload=leg["what"], per_gpu_batch=args.batch, global_batch=args.batch,
                            parallelism="host CPU", threads=r["threads"],
                            note="unmodified reference modules (oracle/_ref) on the host cores; fwd + CE + bwd, no "
                                 "optimizer step"),
                cpu_baseline=dict(value=v, unit="clips/s", cores=r["threads"], kind=kind,
                                  sample=f"{r['steps']} x fwd+bwd of {args.batch} clips through slowfast.models.build_model "
                                         f"(fp32 ATen CPU kernels), {r['ms_per_step']:.0f} ms/step"),
                e2e=dict(value=v, unit="clips/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def aten_gpu_leg(preset: str, dev, batch: int, iters: int = 3):
    """The comparator SURVEY.md 8(d) names as the one that matters: the reference's OWN modules (nn.Conv3d / BatchNorm3d /
    MultiScaleAttention ... = ATen + cuDNN / cuBLAS kernels) on the SAME device: fwd + CE + bwd of the same batch in fp32
    (TF32 off: the reference's parity setting), with TF32 allowed (torch's cuDNN default), and under bf16 autocast."""
    import torch.nn.functional as F
    over = ["NUM_GPUS", 1, "MODEL.DROPOUT_RATE", 0.0] + (["MVIT.DROPPATH_RATE", 0.0] if "MVIT" in preset else [])
    cfg, model = reference_model(preset, over)
    model = model.to(dev).train()
    x, y = synthetic_batch(cfg, batch, 1234)
    x, y = [t.to(dev) for t in x], y.to(dev)
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    out = {}
    try:
        torch.backends.cudnn.benchmark = True
        for mode in ("fp32", "tf32", "bf16_autocast"):
            torch.backends.cudnn.allow_tf32 = mode != "fp32"
            torch.backends.cuda.matmul.allow_tf32 = mode != "fp32"

            def one():
                model.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=mode == "bf16_autocast"):
                    loss = F.cross_entropy(model([t for t in x]), y)
                loss.backward()

            for _ in range(2):
                one()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                one()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            out[mode] = dict(ms_per_step=ms, clips_per_s=batch / (ms * 1e-3))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
        del model
        torch.cuda.empty_cache()
    out["what"] = (f"fwd+CE+bwd (no optimizer step) of {batch} clips through the UNMODIFIED reference modules "
                   f"({REF_YAML[preset]}) on this GPU: ATen / cuDNN / cuBLAS kernels")
    return out


# ------------------------------------------------------------------------------------------------ engine legs
def build_leg(name: str, nsplit: int, dev, rank: int, batch=None):
    import torch.nn.functional as F

    from slowfast_b200.config import get_cfg
    leg = LEGS[name]
    cfg = get_cfg(leg["preset"], B200={"NSPLIT": nsplit})
    mname = cfg.MODEL.MODEL_NAME
    if mname == "SlowFast":
        from slowfast_b200.nets.resnet import B200SlowFast as M
    elif mname == "MViT":
        from slowfast_b200.nets.mvit import B200MViT as M
    elif mname == "X3D":
        from slowfast_b200.nets.x3d import B200X3D as M
    else:
        from slowfast_b200.nets.maskfeat import B200MaskMViT as M
    torch.manual_seed(cfg.RNG_SEED)
    model = M(cfg).to(dev).train()
    if TORCH_OPTIM:   # A/B: the optimizers the reference's construct_optimizer builds, on param.grad
        if leg["opt"] == "sgd":
            opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
        else:
            opt = torch.optim.AdamW(model.parameters(), lr=1e-5, weight_decay=0.05)
    else:             # the same updates fused on the flat gradient bucket (slowfast_b200/optim.py, csrc/optim.cu)
        from slowfast_b200.optim import FlatOptimizer
        model.flat_grad_only = True
        if leg["opt"] == "sgd":
            opt = FlatOptimizer(model, "sgd", lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
        else:
            opt = FlatOptimizer(model, "adamw", lr=1e-5, weight_decay=0.05)
    B = batch or leg["batch"]
    g = torch.Generator().manual_seed(leg["seed"] + rank)
    T = cfg.DATA.NUM_FRAMES
    clip = torch.randn(B, 3, T, 224, 224, generator=g)
    if mname == "SlowFast":
        idx = torch.linspace(0, T - 1, T // cfg.SLOWFAST.ALPHA).long()   # pack_pathway_output (datasets/utils.py:95-103)
        host = [clip.index_select(2, idx).contiguous(), clip]
    elif mname == "MaskMViT":
        tt = T // cfg.MVIT.PATCH_STRIDE[0]
        host = [clip, (torch.rand(B, tt, 7, 7, generator=g) < 0.4).float()]
    else:
        host = [clip]
    labels = torch.randint(0, cfg.MODEL.NUM_CLASSES, (B,), generator=g)
    host = [t.pin_memory() for t in host]
    labels = labels.pin_memory()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    meta = torch.Tensor()
    last = {}   # the model output of the latest step (--dump-outputs)

    def step(x, y):
        opt.zero_grad(set_to_none=True)
        if mname == "MaskMViT":
            preds, labs = model([x[0], meta, x[1]])
            last["logits"] = preds[0]
            loss = sum(F.mse_loss(p, l[0]) * l[1] for p, l in zip(preds, labs))   # losses.py:38-62 MultipleMSELoss
        else:
            last["logits"] = model(x)
            loss = F.cross_entropy(last["logits"], y)
        loss.backward()
        if world > 1:
            model.allreduce_gradients()
        opt.step()
        return loss

    return dict(name=name, cfg=cfg, model=model, step=step, host=host, labels=labels, B=B, leg=leg, last=last)


DUMP_SAMPLE = 1 << 21   # parameter / gradient elements written by --dump-outputs (8 MiB each in float32)


def dump_outputs(out_dir: str, model, loss, logits) -> None:
    """What the caller of a training step receives, as float32 .npy files: the loss, the logits, and the same seeded
    sample of DUMP_SAMPLE elements of the updated parameters and of their gradients (all parameters flattened in
    model.parameters() order; all of them when there are fewer).  The kernels accumulate some sums with atomics, so two
    runs agree to rounding, not bit for bit: compare with a tolerance (two runs of the 10 + 3 step headline on a B200 at
    1000 W: loss 8e-7, logits 1e-5, parameters 2e-6, gradients 4e-3 relative L2)."""
    import numpy as np
    params = list(model.parameters())
    if getattr(model, "flat_grad_only", False):   # no param.grad: read the bucket where FlatOptimizer reads it
        from slowfast_b200.engine import flat_offsets
        offsets, _ = flat_offsets(params)
        grads = [model.ctx.flat_grad[o:o + p.numel()] for p, o in zip(params, offsets)]
    else:
        grads = [p.grad for p in params]
    flat_p = torch.cat([p.detach().flatten() for p in params])
    flat_g = torch.cat([g.detach().flatten() for g in grads])
    n = flat_p.numel()
    idx = torch.arange(n) if n <= DUMP_SAMPLE else \
        torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    idx = idx.to(flat_p.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("loss", loss.detach().reshape(1)), ("logits", logits.detach()),
                    ("params_sample", flat_p[idx]), ("grads_sample", flat_g[idx])):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def measure_leg(L, args, dev, world, barrier, max_over_ranks, clock_index=None, dump_dir=None):
    """(1) device-resident clips/s, (2) end-to-end clips/s with pinned H2D + loss read-back inside the timed region,
    (3) per-class roofline of the implicit-GEMM kernels.  With ``dump_dir``, the outputs of the last step of (1) are
    written there before anything else runs.  Returns a dict."""
    from slowfast_b200 import ops
    step, host, labels_h, B = L["step"], L["host"], L["labels"], L["B"]
    resident = [t.to(dev) for t in host]
    labels = labels_h.to(dev)
    for _ in range(max(args.warmup, 3)):
        step(resident, labels)
    barrier()
    sampler = ClockSampler(clock_index) if clock_index is not None else None
    if sampler:
        sampler.start()
    l0 = ops.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        loss = step(resident, labels)
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = ops.launches() - l0
    clocks = sampler.stop() if sampler else None
    value = B * world * args.steps / (ms_total * 1e-3)
    if dump_dir:
        dump_outputs(dump_dir, L["model"], loss, L["last"]["logits"])

    # end to end through the public call with HOST buffers: pinned H2D every step (prefetched on a copy stream, as a
    # loader with non_blocking copies does) + D2H read of the loss every step
    copy_stream = torch.cuda.Stream()
    bufs = [[torch.empty_like(t, device=dev) for t in host] for _ in range(2)]
    lab_bufs = [torch.empty_like(labels_h, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            for d, s in zip(bufs[slot], host):
                d.copy_(s, non_blocking=True)
            lab_bufs[slot].copy_(labels_h, non_blocking=True)
            ready[slot].record(copy_stream)

    for s in range(2):
        consumed[s].record()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    prefetch(0)
    last = 0.0
    for i in range(args.steps):
        slot = i & 1
        if i + 1 < args.steps:
            prefetch(slot ^ 1)
        torch.cuda.current_stream().wait_event(ready[slot])
        loss = step(bufs[slot], lab_bufs[slot])
        consumed[slot].record()
        last = loss.item()  # device -> host read of the step's result
    t1.record()
    barrier()
    ms_e2e = max_over_ranks(t0.elapsed_time(t1))
    e2e_value = B * world * args.steps / (ms_e2e * 1e-3)
    h2d = sum(t.numel() * t.element_size() for t in host) + labels_h.numel() * labels_h.element_size()
    # end to end with the device-side input pipeline (SURVEY.md 8f-3, slowfast_b200/data.py): the H2D copy carries the uint8
    # clip [B, T, 224, 224, 3]; normalisation, THWC -> CTHW and the pathway packing run as kernels on the GPU
    e2e_u8 = None
    if L["name"] == "slowfast":
        from slowfast_b200.data import pack_pathways_u8
        cfg = L["cfg"]
        g = torch.Generator().manual_seed(99)
        host_u8 = torch.randint(0, 256, (B, cfg.DATA.NUM_FRAMES, 224, 224, 3), generator=g, dtype=torch.uint8).pin_memory()
        ubufs = [torch.empty_like(host_u8, device=dev) for _ in range(2)]

        def prefetch_u8(slot):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                ubufs[slot].copy_(host_u8, non_blocking=True)
                lab_bufs[slot].copy_(labels_h, non_blocking=True)
                ready[slot].record(copy_stream)

        for warm in range(3):   # the u8 path has its own input tensors: warm the program up on them
            step(pack_pathways_u8(ubufs[0].copy_(host_u8), cfg), labels)
        for s_ in range(2):
            consumed[s_].record()
        barrier()
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record()
        prefetch_u8(0)
        for i in range(args.steps):
            slot = i & 1
            if i + 1 < args.steps:
                prefetch_u8(slot ^ 1)
            torch.cuda.current_stream().wait_event(ready[slot])
            loss = step(pack_pathways_u8(ubufs[slot], cfg), lab_bufs[slot])
            consumed[slot].record()
            loss.item()
        u1.record()
        barrier()
        ms_u8 = max_over_ranks(u0.elapsed_time(u1))
        e2e_u8 = dict(value=B * world * args.steps / (ms_u8 * 1e-3), unit="clips/s", ms_per_step=ms_u8 / args.steps,
                      h2d_bytes_per_step=host_u8.numel() + labels_h.numel() * labels_h.element_size(), d2h_bytes_per_step=4,
                      note="uint8 clip H2D + sfb_clip_normalize_pack (normalise, permute, slow-pathway sub-sampling) on the GPU")
        del ubufs
    # (every rank runs the profiled extra step: it contains the gradient all-reduce)
    roofline = profile_conv_kernels(L["model"], step, resident, labels, load_peaks(), L["name"])
    out = dict(value=value, unit="clips/s", ms_per_step=ms_total / args.steps, per_gpu_batch=B, gpu_launches=launches,
               e2e=dict(value=e2e_value, unit="clips/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=4,
                        ms_per_step=ms_e2e / args.steps, last_loss=last),
               roofline=roofline, clocks=clocks, e2e_uint8_input=e2e_u8)
    gf = L["leg"]["gflop"]
    if gf:
        out["algorithmic_tflops"] = value * 3 * gf * 1e9 / 1e12
    if L["leg"]["mb"]:
        out["ideal_traffic_gbps"] = value * 3 * L["leg"]["mb"] * 1e6 / 1e9
    del bufs, lab_bufs, resident
    return out


def profile_conv_kernels(model, step, resident, labels, peaks, leg_name):
    """Time every implicit-GEMM launch of one step with CUDA events on the launching stream and aggregate per kernel
    class; the roofline object describes the class with the largest share of the step.  ``achieved`` = algorithmic
    bytes (operands once at the precision they are stored in + fp32 output) or algorithmic 2*M*N*K FLOPs / the sum of
    launch durations; ``traffic`` = average DRAM bytes per launch of the same class from the committed ncu pass."""
    from slowfast_b200 import ops
    recs = []
    orig_conv, orig_wgrad = ops.conv_igemm, ops.conv_wgrad

    def timed(kind, fn, flops_fn, bytes_fn):
        def wrapper(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a, **k)
            e.record()
            recs.append((kind, s, e, flops_fn(*a, **k), bytes_fn(*a, **k)))
            return r
        return wrapper

    def conv_flops(x, f, geom, out, strides, **k):
        m = x.n * geom.out[0] * geom.out[1] * geom.out[2]
        return 2.0 * m * f.rows * f.ntaps * f.cols_pad

    def conv_bytes(x, f, geom, out, strides, **k):
        m = x.n * geom.out[0] * geom.out[1] * geom.out[2]
        planes = 2 if x.lo is not None else 1
        return x.rows * x.c * 2 * planes + f.rows * f.ntaps * f.cols_pad * 2 * planes + m * f.rows * 4

    def wg_flops(x, dy, geom, dwm, **k):
        taps = geom.k[0] * geom.k[1] * geom.k[2]
        return 2.0 * dy.rows * dy.c * taps * x.c

    def wg_bytes(x, dy, geom, dwm, **k):
        planes = 2 if x.lo is not None else 1
        return (x.rows * x.c + dy.rows * dy.c) * 2 * planes + dwm.numel() * 4

    ops.conv_igemm = timed("conv_igemm(fprop+dgrad)", orig_conv, conv_flops, conv_bytes)
    ops.conv_wgrad = timed("conv_wgrad", orig_wgrad, wg_flops, wg_bytes)
    graphs_were = model.cuda_graphs
    model.cuda_graphs = False  # replays bypass the python wrappers: time the same launches eagerly
    try:
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        step(resident, labels)
        s1.record()
        torch.cuda.synchronize()
    finally:
        ops.conv_igemm, ops.conv_wgrad = orig_conv, orig_wgrad
        model.cuda_graphs = graphs_were
    step_ms = s0.elapsed_time(s1)
    agg = {}
    for kind, s, e, fl, by in recs:
        a = agg.setdefault(kind, dict(ms=0.0, flops=0.0, bytes=0.0, launches=0))
        a["ms"] += s.elapsed_time(e)
        a["flops"] += fl
        a["bytes"] += by
        a["launches"] += 1
    if not agg:
        return None
    top = max(agg, key=lambda k: agg[k]["ms"])
    a = agg[top]
    tf = a["flops"] / (a["ms"] * 1e-3) / 1e12
    gbs = a["bytes"] / (a["ms"] * 1e-3) / 1e9
    tensor_frac = tf / peaks["tflops_sustained"]
    hbm_frac = gbs / peaks["hbm_gbs"]
    bound = "tensor" if tensor_frac >= hbm_frac else "hbm"
    tr = load_traffic().get(leg_name, {}).get(top.split("(")[0])
    traffic = None
    if tr:
        traffic = tr["dram_bytes_per_launch"]
    return dict(kernel=top, bound=bound,
                achieved=tf if bound == "tensor" else gbs, peak=peaks["tflops_sustained"] if bound == "tensor" else peaks["hbm_gbs"],
                unit="TFLOP/s" if bound == "tensor" else "GB/s", frac=max(tensor_frac, hbm_frac), traffic=traffic,
                algorithmic_bytes_per_launch=a["bytes"] / a["launches"],
                traffic_source=(tr or {}).get("source"),
                peak_source=peaks["source"] + (" (sustained bf16: kernel timed inside a long step)" if bound == "tensor" else ""),
                per_class={k: dict(launches=v["launches"], ms=round(v["ms"], 3), share_of_step=round(v["ms"] / step_ms, 4),
                                   algorithmic_tflops=round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2),
                                   algorithmic_gbs=round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1)) for k, v in agg.items()},
                profiled_step_ms=round(step_ms, 3),
                note="achieved = sum of algorithmic bytes / 2*M*N*K FLOPs (operand-split passes NOT counted) over the sum of "
                     "CUDA-event launch durations of the class in one eager step; events add launch gaps: a lower bound")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nsplit", type=int, default=3, choices=[1, 3])
    ap.add_argument("--batch", type=int, default=LEGS["slowfast"]["batch"])
    ap.add_argument("--legs", default="mvitv2_s,x3d_m,maskfeat_s,maskfeat_b,mvitv2_s_bf16",
                    help="secondary legs to run (comma separated; '' = headline only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aten-gpu", action="store_true",
                    help="skip timing the reference's own modules (ATen / cuDNN) on this GPU (N=1 only)")
    ap.add_argument("--torch-optim", action="store_true",
                    help="step torch.optim.SGD / AdamW on param.grad instead of the fused flat-bucket optimizer")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, logits and a seeded sample of the updated parameters and their gradients "
                         "after the headline leg's last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global TORCH_OPTIM
    TORCH_OPTIM = args.torch_optim
    if args.impl == "reference":
        reference_arm(args)
        return
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=600))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    peaks = load_peaks()
    # ---- headline: SlowFast-8x8-R50 ------------------------------------------------------------------------------
    L = build_leg("slowfast", args.nsplit, dev, rank, batch=args.batch)
    head = measure_leg(L, args, dev, world, barrier, max_over_ranks, clock_index=local if rank == 0 else None,
                       dump_dir=args.dump_outputs if rank == 0 else None)
    cfg = L["cfg"]
    del L
    torch.cuda.empty_cache()

    # ---- CPU baseline: the UNMODIFIED reference on this box's host cores, bounded sample (rank 0, N == 1 only)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            r = time_reference_cpu("SLOWFAST_8x8_R50", 4, steps=3, warm=1, budget_s=25.0)
            cpu_baseline = dict(value=r["clips_per_s"], unit="clips/s", cores=r["threads"], kind="reference",
                                sample=f"{r['steps']} x fwd+CE+bwd of {r['batch']} clips through the unmodified reference "
                                       f"modules (oracle/_ref, fp32 ATen CPU kernels), {r['ms_per_step']:.0f} ms/step")
        except Exception as e:  # noqa: BLE001
            cpu_baseline = dict(error=repr(e)[:300])

    # ---- secondary legs: the other configs of BASELINE.json's metric --------------------------------------------
    extra = {}
    for name in [s for s in args.legs.split(",") if s]:
        try:
            if name == "mvitv2_s_bf16":   # BASELINE config 4 says bf16: the same leg in fast mode (bf16 operands)
                LL = build_leg("mvitv2_s", 1, dev, rank)
                r = measure_leg(LL, args, dev, world, barrier, max_over_ranks)
                r["precision_mode"] = "nsplit1 (bf16 operands, fp32 accumulate)"
            else:
                LL = build_leg(name, args.nsplit, dev, rank)
                r = measure_leg(LL, args, dev, world, barrier, max_over_ranks)
            r["metric"] = f"clips/sec (fwd+bwd) {name}"
            r["config"] = LL["leg"]["what"] + ", synthetic"
            extra[name] = r
            del LL
        except Exception as e:  # noqa: BLE001 - the headline line must still be printed
            extra[name] = dict(error=repr(e)[:300])
        torch.cuda.empty_cache()

    # ---- the reference's own GPU code path on this device (N == 1 only; a reported baseline) ---------------------
    aten_gpu = None
    if rank == 0 and world == 1 and not args.no_aten_gpu:
        aten_gpu = {}
        for name, preset in (("slowfast", "SLOWFAST_8x8_R50"), ("mvitv2_s", "MVITv2_S_16x4"), ("x3d_m", "X3D_M")):
            try:
                aten_gpu[name] = aten_gpu_leg(preset, dev, batch=LEGS[name]["batch"] if name != "slowfast" else args.batch)
            except Exception as e:  # noqa: BLE001
                aten_gpu[name] = dict(error=repr(e)[:300])

    if rank == 0:
        value = head["value"]
        step_flops = 3.0 * LEGS["slowfast"]["gflop"] * 1e9  # training step ~ 3x forward (SURVEY 8d)
        line = dict(
            metric="clips/sec (fwd+bwd) SlowFast-8x8-R50", value=value, unit="clips/s", n_gpus=world,
            steps=args.steps, warmup=args.warmup, ms_per_step=head["ms_per_step"], higher_is_better=True,
            scaling="weak", vs_baseline=None,
            dtype="bf16x3-split operands, f32 accumulate/storage" if args.nsplit == 3 else "bf16 operands, f32 accumulate",
            data="synthetic",
            config=dict(workload=LEGS["slowfast"]["what"], per_gpu_batch=args.batch, global_batch=args.batch * world,
                        parallelism=f"dp{world}", precision_mode=f"nsplit{args.nsplit}",
                        optimizer="torch.optim on param.grad" if TORCH_OPTIM else "fused SGD-nesterov / AdamW on the flat bucket",
                        l2_policy="per-step working set (inputs 193 MB + activations > 10 GB) exceeds the 126 MB L2; no flush needed"),
            e2e=head["e2e"], e2e_uint8_input=head["e2e_uint8_input"], gpu_launches=head["gpu_launches"],
            clocks=head["clocks"], roofline=head["roofline"],
            cpu_baseline=cpu_baseline,
            aten_gpu_baseline=aten_gpu,
            model_tflops=dict(algorithmic_tflops=value * step_flops / 1e12,
                              frac_of_bf16_sustained=value * step_flops / 1e12 / world / peaks["tflops_sustained"],
                              peaks=peaks["source"]),
        )
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
