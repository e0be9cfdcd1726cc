#!/usr/bin/env python
"""bench.py — headline benchmark of the argus_b200 hot path.

    python bench.py --gpus N --steps K --warmup W              # our B200 path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle port)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also save what the last timed step computed

Workload (BASELINE.json configs[1]): one data-parallel training step of NCameraCNN on a synthetic 2-view batch of
256 image pairs per GPU at 256x256 — uint8 images -> GPU augmentation -> forward (bf16, fp32 accumulate) ->
SE(3) pose loss -> backward -> clip_grad_norm_ + Adam.  Metric: training image-pairs/s over all GPUs.

`value` is timed on the device with the uint8 batch already resident in HBM; `e2e` is the same step through the
public engine API with pinned HOST buffers (H2D of the images/targets and D2H of the loss inside the timed region).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

PAIR_FLOPS_FWD = 21.362e9          # SURVEY.md §8(d): forward GEMM FLOPs per image pair at 256x256
PAIR_FLOPS_TRAIN = 63.47e9         # forward + dgrad + wgrad (no stem dgrad)
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
# pairs per CPU step in BOTH CPU legs (`cpu_baseline` of our line and `--impl reference`): the largest sample of the
# 256-pair workload that keeps `--steps 20 --warmup 5` within a few minutes on the box's host cores (~8 pairs/s)
CPU_SAMPLE_PAIRS = 32
# --dump-outputs keeps this many positions of each 25.9 M-element arena (parameters, gradients): 16 MiB apiece in fp32
DUMP_SAMPLE = 1 << 22


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return json.loads(p.read_text()), "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.index = index
        self.samples: list[list[str]] = []
        self.proc = None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self) -> None:
        for line in self.proc.stdout:
            self.samples.append([c.strip() for c in line.split(",")])

    def mark(self) -> None:
        """Samples before this call (start-up, warm-up) are dropped from the summary."""
        self.first = len(self.samples)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples[getattr(self, "first", 0):]:
            if len(s) < 7:
                continue
            try:
                sm.append(float(s[0]))
                smax = float(s[1])
            except ValueError:
                continue
            for n, v in zip(names, s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def synthetic_batch(B: int, n_cams: int, H: int, W: int, seed: int):
    """uint8 HWC image pairs (what a decoded PNG pair is, reference tests/conftest.py:35-41) and SE3 targets."""
    import torch

    g = torch.Generator().manual_seed(seed)
    images = torch.randint(0, 256, (B, n_cams, H, W, 3), dtype=torch.uint8, generator=g)
    q = torch.randn(B, 4, generator=g)
    targets = torch.cat([torch.randn(B, 3, generator=g), q / q.norm(dim=-1, keepdim=True)], -1)
    return images, targets


def dump_step_outputs(directory: str, model, engine, loss) -> None:
    """Saves what the last training step handed its caller, as float32 .npy files: the mean loss it returned, the
    gradient norm before clipping, and the state the next step starts from (the updated parameters and the batch-norm
    running statistics) together with the gradients of the step. Parameters and gradients are the same fixed, seeded
    sample of DUMP_SAMPLE positions, so that two builds can be compared output for output."""
    import numpy as np
    import torch

    params = model.flat_params
    idx = torch.randperm(params.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    idx = idx.to(params.device)
    arrays = {"loss": loss.reshape(1), "grad_norm": engine.last_grad_norm.reshape(1), "params_sample": params[idx],
              "grads_sample": model.flat_grads[idx], "bn_running_stats": model._flat_buffers}
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(out / f"{name}.npy", t.detach().float().cpu().numpy())


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args) -> None:
    os.environ.setdefault("ARGUS_PROFILE_DETAIL", "1")   # instrumented pass: tensor-core launches keyed by layer shape
    import torch
    import torch.distributed as dist

    from argus_b200 import _lib
    from argus_b200.engine import TrainEngine
    from argus_b200.models import NCameraCNN

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime

        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev,
                                timeout=datetime.timedelta(seconds=180))
    B, H, W, n_cams = args.batch, args.size, args.size, 2
    if os.environ.get("ARGUS_HIGH_PRIORITY_STREAM", "0") == "1":
        # Experiment (off by default): the step on a high-priority stream, so that the look-ahead augmentation (engine side
        # stream, default priority) only fills what the step's kernels leave free instead of competing with them at every
        # kernel boundary. Measured 40.3 -> 39.8 ms/step, but one of several runs then diverged in the last digits of
        # the loss (profiles/experiments/stream_determinism.py), so the reproducible default-stream configuration stays.
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=-1))

    torch.manual_seed(42)
    model = NCameraCNN().to(dev)
    from argus_b200.data import Augmentation, AugmentationConfig

    # the training loop's configuration (argus_b200/train.py defaults): the reference's default-on kornia chain AND its
    # spaghetti arcs (drawn on every training image, data.py:212-215), both on the device
    augmentation = Augmentation(AugmentationConfig(), train=True, seed=42, gpu_spaghetti=True).to(dev)
    if args.no_augmentation:
        augmentation = None
    engine = TrainEngine(model, lr=1e-4, max_grad_norm=1.0, augmentation=augmentation)

    ring = 3
    host_batches = []
    dev_batches = []
    for i in range(ring):
        imgs, tgt = synthetic_batch(B, n_cams, H, W, seed=1000 * rank + i)
        host_batches.append((imgs.pin_memory(), tgt.pin_memory()))
        dev_batches.append((imgs.to(dev), tgt.to(dev)))
    lib = _lib.load()
    lib.argus_launch_count.restype = ctypes.c_int64

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up, then the device-resident timed region (nvidia-smi needs ~1 s to start: launch it first)
    sampler = ClockSampler(local_rank)
    sampler.start()
    trace = [] if os.environ.get("ARGUS_BENCH_TRACE") in ("1", "2") else None   # debugging aid: every step's loss to stderr
    if os.environ.get("ARGUS_BENCH_TRACE") == "2":
        # ... and checksums of the pooled stem output (the staged input), the gradient arena and the updated parameters
        sigs = []
        pooled_buf = torch.empty(B * n_cams * (H // 4) * (W // 4) * 64, dtype=torch.bfloat16, device=dev)

        infos_ = list(model._param_infos)
        untraced_step = engine.step

        def traced_step(images, targets):
            # nothing is inserted between backward and optimizer (that hides the effect): everything is read afterwards
            loss_ = untraced_step(images, targets)
            _lib.check(lib_.argus_model_copy_activation(model._handle.ptr, ctypes.c_int(-1), _lib.ptr(pooled_buf),
                                                        ctypes.c_int64(pooled_buf.numel()), None, None, _lib.stream_ptr()))
            a = pooled_buf.float().abs().sum().double()
            g_ = model.flat_grads
            per = torch.stack([g_[o:o + k].double().abs().sum() for (_n, o, k, _s) in infos_])
            c = model.flat_params.double().abs().sum()
            sigs.append(torch.cat([torch.stack([a, per.sum(), c]), per]))
            return loss_

        lib_ = _lib.load()
        engine.step = traced_step
    for i in range(args.warmup):
        l_ = engine.step(*dev_batches[i % ring])
        if trace is not None:
            trace.append(l_.clone())
    barrier()
    t_wait = time.time()
    while not sampler.samples and time.time() - t_wait < 5.0:
        time.sleep(0.05)                      # (no collective in this loop: ranks may wait different amounts)
    for i in range(2):                        # back under load before the timed region
        l_ = engine.step(*dev_batches[i % ring])
        if trace is not None:
            trace.append(l_.clone())
    engine.prefetch(dev_batches[0][0])        # look-ahead staging, as the training loop does (argus_b200/train.py)
    barrier()
    sampler.mark()
    launches0 = lib.argus_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    loss = None
    for i in range(args.steps):
        loss = engine.step(*dev_batches[i % ring])
        if trace is not None:
            trace.append(loss.clone())
        # augmentation + staging of the next batch on the engine's side stream, overlapping this step
        engine.prefetch(dev_batches[(i + 1) % ring][0])
    ev1.record()
    barrier()
    launches = lib.argus_launch_count() - launches0
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * B * args.steps / (ms_total / 1e3)
    final_loss = float(loss.item())
    if args.dump_outputs and rank == 0:
        dump_step_outputs(args.dump_outputs, model, engine, loss)   # before the passes below change the model
    if trace is not None and rank == 0:
        print("LOSS_TRACE " + " ".join(repr(float(x)) for x in trace), file=sys.stderr, flush=True)
        if os.environ.get("ARGUS_BENCH_TRACE") == "2":
            for k, sg in enumerate(sigs[:len(trace)]):
                print(f"SIG {k} in={float(sg[0])!r} grad={float(sg[1])!r} par={float(sg[2])!r}", file=sys.stderr, flush=True)
            import json as json_
            json_.dump({"names": [n for (n, _o, _k, _s) in infos_], "sig": [[float(v) for v in sg] for sg in sigs]},
                       open(os.environ.get("ARGUS_BENCH_TRACE_FILE", "/tmp/bench_trace.json"), "w"))

    # ---- end-to-end: pinned host buffers -> H2D -> step -> loss D2H, every step
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()
    stage_img = [torch.empty_like(dev_batches[0][0]) for _ in range(2)]
    stage_tgt = [torch.empty_like(dev_batches[0][1]) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    for i in range(2):  # warm the path
        stage_img[0].copy_(host_batches[i % ring][0], non_blocking=True)
        stage_tgt[0].copy_(host_batches[i % ring][1], non_blocking=True)
        engine.step(stage_img[0], stage_tgt[0])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    # double-buffered: the copy of batch i+1 runs on a side stream while batch i trains
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    with torch.cuda.stream(copy_stream):
        stage_img[0].copy_(host_batches[0][0], non_blocking=True)
        stage_tgt[0].copy_(host_batches[0][1], non_blocking=True)
        ready[0].record(copy_stream)
    for i in range(args.steps):
        cur, nxt = i % 2, (i + 1) % 2
        if i + 1 < args.steps:
            with torch.cuda.stream(copy_stream):
                if i >= 1:
                    copy_stream.wait_event(consumed[nxt])
                stage_img[nxt].copy_(host_batches[(i + 1) % ring][0], non_blocking=True)
                stage_tgt[nxt].copy_(host_batches[(i + 1) % ring][1], non_blocking=True)
                ready[nxt].record(copy_stream)
        torch.cuda.current_stream().wait_event(ready[cur])
        l = engine.step(stage_img[cur], stage_tgt[cur])
        if i + 1 < args.steps:
            engine.prefetch(stage_img[nxt], after=ready[nxt])
        consumed[cur].record()
        loss_host.copy_(l.reshape(1), non_blocking=True)
    e1.record()
    barrier()
    t2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t2.item()) / 1e3)
    h2d = host_batches[0][0].numel() + host_batches[0][1].numel() * 4

    # ---- per-kernel-family timing with CUDA events (separate pass: the headline numbers above are un-instrumented)
    families = {}
    _lib.call("argus_model_set_wgrad_overlap", model._handle.ptr, 0)  # isolated kernel times for the roofline
    if rank == 0:
        lib.argus_profile_enable(1)
    for i in range(2):  # every rank steps (the steps contain collectives); only rank 0 records events
        engine.step(*dev_batches[i % ring])
    torch.cuda.synchronize()
    if rank == 0:
        buf = ctypes.create_string_buffer(1 << 19)
        _lib.check(lib.argus_profile_report(buf, ctypes.c_int(1 << 19)))
        lib.argus_profile_enable(0)
        families = json.loads(buf.value.decode())
        for f in families.values():
            f["launches"] //= 2
            f["ms"] /= 2
            f["flops"] /= 2
            f["bytes"] /= 2
    barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_kind = load_peaks()
    # the instrumented pass keys tensor-core launches by layer shape ("conv_fwd:M.._N.._K.._t.."); fold them back into
    # kernel families for the summary and keep the per-shape groups for the roofline of the dominant kernel
    shapes = {k: f for k, f in families.items() if ":" in k}
    folded: dict = {}
    for k, f in families.items():
        base = k.split(":")[0]
        agg = folded.setdefault(base, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
        for key in agg:
            agg[key] += f[key]
    families = folded
    conv = [families[k] for k in ("conv_fwd", "conv_dgrad", "conv_wgrad", "conv_wgradx") if k in families]
    conv_ms = sum(f["ms"] for f in conv)
    conv_flops = sum(f["flops"] for f in conv)
    conv_launches = sum(f["launches"] for f in conv)
    total_ms = sum(f["ms"] for f in families.values()) or 1.0
    algorithmic_flops = PAIR_FLOPS_TRAIN * B  # per step, all tensor-core launches together
    achieved = algorithmic_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
    peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    ridge = peak * 1e12 / (peaks["hbm_gbs"] * 1e9)       # flop / byte above which a launch is tensor-bound
    roofline_aggregate = {
        "bound": "tensor", "kernel": "conv_gemm_kernel + wgrad_kernel + wgrad_xpose_kernel (tcgen05 implicit GEMM, all "
                                     "launches of a step, HBM-bound and tensor-bound shapes together)",
        "achieved": round(achieved, 2), "peak": peak, "unit": "TFLOP/s", "frac": round(achieved / peak, 4),
        "peak_kind": f"{peak_kind} sustained cuBLAS bf16", "traffic": None, "algorithmic_bytes_per_launch": None,
        "launches_per_step": conv_launches, "avg_launch_ms": round(conv_ms / max(conv_launches, 1), 4),
        "issued_flops_per_step": conv_flops, "algorithmic_flops_per_step": algorithmic_flops,
        "share_of_step": round(conv_ms / total_ms, 4),
    }
    # DRAM traffic of the same launches from the committed ncu capture (profiles/capture.sh), per launch like `achieved`
    conv_bytes = sum(f["bytes"] for f in conv)
    roofline_aggregate["algorithmic_bytes_per_launch"] = round(conv_bytes / max(conv_launches, 1))
    traffic_files = sorted(Path(__file__).resolve().parent.glob("profiles/*_conv_traffic.json"))
    if traffic_files and B == 256 and args.size == 256:
        tr = json.loads(traffic_files[-1].read_text())
        roofline_aggregate["traffic"] = round(tr["dram_bytes_per_launch"])
        roofline_aggregate["traffic_source"] = (f"committed: profiles/{traffic_files[-1].name} ({tr['launches']} launches "
                                                "of one step under ncu; not re-measured in this run)")
    # launches split by what bounds their SHAPE (arithmetic intensity against the ridge of the measured peaks)
    split = {"tensor": {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0},
             "hbm": {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0}}
    for k, f in shapes.items():
        if not k.startswith("conv_") or f["bytes"] <= 0:
            continue
        b = "tensor" if f["flops"] / f["bytes"] >= ridge else "hbm"
        for key in split[b]:
            split[b][key] += f[key]
    by_bound = {}
    if split["tensor"]["ms"] > 0:
        tf = split["tensor"]["flops"] / (split["tensor"]["ms"] / 1e3) / 1e12
        by_bound["tensor_bound_shapes"] = {"ms": round(split["tensor"]["ms"], 3), "launches": split["tensor"]["launches"],
                                           "achieved": round(tf, 1), "unit": "TFLOP/s (issued)", "peak": peak,
                                           "frac": round(tf / peak, 4)}
    if split["hbm"]["ms"] > 0:
        gb = split["hbm"]["bytes"] / (split["hbm"]["ms"] / 1e3) / 1e9
        by_bound["hbm_bound_shapes"] = {"ms": round(split["hbm"]["ms"], 3), "launches": split["hbm"]["launches"],
                                        "achieved": round(gb, 1), "unit": "GB/s", "peak": peaks["hbm_gbs"],
                                        "frac": round(gb / peaks["hbm_gbs"], 4)}
    roofline_aggregate["by_bound"] = by_bound
    # `roofline` proper: the single dominant tensor-core launch group (one kernel instantiation on one layer shape, the
    # largest share of the step), against the roofline that bounds THAT shape
    roofline = dict(roofline_aggregate)
    top = max(((k, f) for k, f in shapes.items() if k.startswith("conv_") and f["bytes"] > 0), key=lambda kv: kv[1]["ms"],
              default=None)
    if top is not None:
        k, f = top
        n_l = max(f["launches"], 1)
        ai = f["flops"] / f["bytes"]
        if ai >= ridge:
            ach, pk, unit, bound = f["flops"] / (f["ms"] / 1e3) / 1e12, peak, "TFLOP/s", "tensor"
            pk_kind = f"{peak_kind} sustained cuBLAS bf16"
        else:
            ach, pk, unit, bound = f["bytes"] / (f["ms"] / 1e3) / 1e9, peaks["hbm_gbs"], "GB/s", "hbm"
            pk_kind = f"{peak_kind} copy bandwidth"
        roofline = {"bound": bound, "kernel": f"tcgen05 implicit GEMM, {k} ({n_l} launches / step)",
                    "achieved": round(ach, 1), "peak": pk, "unit": unit, "frac": round(ach / pk, 4), "peak_kind": pk_kind,
                    "traffic": None, "algorithmic_bytes_per_launch": round(f["bytes"] / n_l),
                    "algorithmic_flops_per_launch": round(f["flops"] / n_l), "avg_launch_ms": round(f["ms"] / n_l, 4),
                    "arithmetic_intensity": round(ai, 1), "ridge": round(ridge, 1),
                    "share_of_step": round(f["ms"] / total_ms, 4),
                    "traffic_note": "per-shape DRAM traffic is in profiles/ (ncu --set full captures); not re-measured here"}
        # dram__bytes_read.sum + dram__bytes_write.sum per launch of this family from the committed `ncu --set full` capture
        # (profiles/*_family_traffic.json, written from the capture of the same code), when the shape was captured
        fam_files = sorted(Path(__file__).resolve().parent.glob("profiles/*_family_traffic.json"))
        if fam_files and B == 256 and args.size == 256:
            ft = json.loads(fam_files[-1].read_text()).get(k)
            if ft:
                roofline["traffic"] = round(ft["dram_bytes_per_launch"])
                roofline["traffic_note"] = f"committed: profiles/{fam_files[-1].name} -- {ft['source']}"
    # whole-step HBM view: algorithmic bytes of every launch (each operand tensor counted once) over the step time
    step_bytes = sum(f["bytes"] for f in families.values())
    step_ms = ms_total / args.steps
    hbm_step = {"algorithmic_gb_per_step": round(step_bytes / 1e9, 2),
                "achieved_gbs": round(step_bytes / (step_ms / 1e3) / 1e9, 1), "peak_gbs": peaks["hbm_gbs"],
                "frac": round(step_bytes / (step_ms / 1e3) / 1e9 / peaks["hbm_gbs"], 4),
                "note": "sum over all kernels of one step of the bytes each must move at least once, divided by the "
                        "un-instrumented step time; the step as a whole is HBM-bound"}
    mem = {}
    for k, f in families.items():
        if f["bytes"] > 0 and f["ms"] > 0 and k not in ("conv_fwd", "conv_dgrad", "conv_wgrad"):
            gbs = f["bytes"] / (f["ms"] / 1e3) / 1e9
            mem[k] = {"ms": round(f["ms"], 3), "launches": f["launches"], "GB/s": round(gbs, 1),
                      "frac_hbm": round(gbs / peaks["hbm_gbs"], 3)}
    inference = None
    torch_cuda = None
    del engine
    torch.cuda.empty_cache()
    if world == 1 and not args.no_inference:
        inference = measure_inference(dev, args.size)
    if world == 1 and not args.no_torch_baseline:
        del model
        torch.cuda.empty_cache()
        torch_cuda = torch_cuda_baseline(dev, B, args.size)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_throughput(sample_pairs=CPU_SAMPLE_PAIRS, iters=2, warmup=1, size=args.size,
                                       augmentation=augmentation is not None)

    line = {
        "metric": "train image-pairs/sec", "value": round(value, 2), "unit": "pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "configs[1]: train step, synthetic 2-view batch 256/GPU at 256x256, bf16 + fp32 accumulate, "
                               "augmentation + geometric pose loss + clip + Adam",
                   "per_gpu_batch_pairs": B, "global_batch_pairs": B * world, "image_size": [H, W], "n_cams": n_cams,
                   "augmentation": augmentation is not None,
                   "spaghetti": bool(augmentation is not None and augmentation.gpu_spaghetti), "parallelism": f"dp{world}",
                   "l2_note": "no explicit flush: every step streams >30 GB of activations (>> 126 MB L2) and rotates 3 input batches"},
        "e2e": {"value": round(e2e_value, 2), "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "note": "pinned host uint8 batch -> H2D on a side stream (double buffered) -> engine.step -> loss D2H"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "roofline_aggregate": roofline_aggregate,
        "hbm_step": hbm_step,
        "kernel_families_ms": {k: round(f["ms"], 3) for k, f in families.items()},
        "memory_bound_kernels": mem,
        "final_loss": final_loss,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if inference is not None:
        line["inference"] = inference
    if torch_cuda is not None:
        line["torch_cuda_baseline"] = torch_cuda
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def measure_inference(dev, size: int) -> dict:
    """BASELINE.json configs[2]: eval-mode `get_pose` latency at batch 1 and 64 (protocol of the reference's
    scripts/timing.py:13-45: 100 timed trials after warm-up, CUDA events per trial), eager C-ABI calls and the
    CUDA-graph PoseEstimator; input = uint8 pair(s) in pinned HOST memory (H2D inside the timed region)."""
    import torch

    from argus_b200.models import NCameraCNN
    from argus_b200.utils import PoseEstimator, get_pose

    torch.manual_seed(42)
    model = NCameraCNN().to(dev).eval()
    out = {}
    for B in (1, 64):
        host = synthetic_batch(B, 2, size, size, seed=7)[0].pin_memory()
        est = PoseEstimator(model, B, size, size, uint8_input=True)
        dev_in = host.to(dev)

        def eager():
            return get_pose(dev_in.copy_(host, non_blocking=True), model)

        def graph():
            return est(host)

        res = {}
        for name, fn in (("eager", eager), ("cuda_graph", graph)):
            for _ in range(10):
                fn()
            torch.cuda.synchronize()
            times = []
            for _ in range(100):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                e1.synchronize()
                times.append(e0.elapsed_time(e1))
            times.sort()
            res[name] = {"p50_ms": round(times[50], 4), "p99_ms": round(times[98], 4)}
        res["pairs_per_s_graph"] = round(B / (res["cuda_graph"]["p50_ms"] / 1e3), 1)
        out[f"batch{B}"] = res
    # algorithmic HBM bytes of one batch-64 eval forward (every operand tensor of every kernel once), from the library's
    # own launch accounting: the forward at this batch is an HBM-bound chain of wide 1x1 convolutions, not tensor-bound
    import ctypes as ct

    from argus_b200 import _lib

    lib = _lib.load()
    x64 = synthetic_batch(64, 2, size, size, seed=7)[0].to(dev)
    lib.argus_profile_enable(1)
    with torch.no_grad():
        model._forward_impl(x64, False)
    torch.cuda.synchronize()
    buf = ct.create_string_buffer(1 << 18)
    _lib.check(lib.argus_profile_report(buf, ct.c_int(1 << 18)))
    lib.argus_profile_enable(0)
    fam = json.loads(buf.value.decode())
    fwd_bytes64 = sum(f["bytes"] for f in fam.values())
    # floors (SURVEY.md §8d): batch 1 is bound by reading the 51.8 MB of bf16 weights once plus the forward FLOPs
    # (>= 25 us together); large batches by the forward FLOPs alone (65.6 k pairs/s at the sustained tensor peak)
    peaks, _ = load_peaks()
    floor_b1_us = 51.8e6 / (peaks["hbm_gbs"] * 1e9) * 1e6 + PAIR_FLOPS_FWD / (peaks["bf16_tflops_sustained"] * 1e12) * 1e6
    ceil_pairs = peaks["bf16_tflops_sustained"] * 1e12 / PAIR_FLOPS_FWD
    out["roofline"] = {
        "batch1": {"floor_us": round(floor_b1_us, 1), "p50_us": round(out["batch1"]["cuda_graph"]["p50_ms"] * 1e3, 1),
                   "frac": round(floor_b1_us / (out["batch1"]["cuda_graph"]["p50_ms"] * 1e3), 4),
                   "bound": "launch latency (> 60 dependent kernels), not HBM or tensor"},
        "batch64": {"ceiling_pairs_per_s": round(min(ceil_pairs, 64 / (fwd_bytes64 / (peaks["hbm_gbs"] * 1e9))), 1),
                    "tensor_ceiling_pairs_per_s": round(ceil_pairs, 1),
                    "hbm_ceiling_pairs_per_s": round(64 / (fwd_bytes64 / (peaks["hbm_gbs"] * 1e9)), 1),
                    "algorithmic_gb_per_forward": round(fwd_bytes64 / 1e9, 2),
                    "pairs_per_s": out["batch64"]["pairs_per_s_graph"],
                    "frac": round(out["batch64"]["pairs_per_s_graph"] /
                                  min(ceil_pairs, 64 / (fwd_bytes64 / (peaks["hbm_gbs"] * 1e9))), 4),
                    "bound": "hbm" if fwd_bytes64 / (peaks["hbm_gbs"] * 1e9) > 64 / ceil_pairs else "tensor"}}
    return out


def torch_cuda_baseline(dev, B: int, size: int) -> dict:
    """The library path this repo replaces, on the SAME B200 in the same run (SURVEY.md §8d "the real bar"): the
    reference model (oracle/ref_model.py == argus/models.py on torchvision's ResNet-50, random init) under PyTorch CUDA
    -- cuDNN convolutions, channels_last, bf16 autocast, torch's fused Adam -- for the same training step (forward, pose
    loss, backward, clip_grad_norm_, Adam) on a device-resident fp32 batch (no augmentation: kornia is not installed;
    the reference augments on CPU workers anyway), and eval-mode forward latency at batch 1 / 64. Informative baseline,
    measured after our own timed regions; nothing of it is on the product path."""
    import torch

    from oracle.ref_model import make_reference_model, torch_loss

    out = {}
    try:
        torch.backends.cudnn.benchmark = True
        model = make_reference_model(42).to(dev).to(memory_format=torch.channels_last)
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)
        imgs, tgt = synthetic_batch(B, 2, size, size, seed=0)
        x = (imgs.permute(0, 1, 4, 2, 3).reshape(B, 6, size, size).float() / 255.0).to(dev)
        tgt = tgt.to(dev)

        def step():
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                pred = model(x)
            loss = torch_loss(pred.float(), tgt).mean()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
            return loss

        model.train()
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 8
        e0.record()
        for _ in range(n):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        out["train"] = {"ms_per_step": round(ms, 2), "pairs_per_s": round(B / (ms / 1e3), 1), "batch_pairs": B,
                        "what": "reference NCameraCNN, torch CUDA: cuDNN + channels_last + bf16 autocast + fused Adam, "
                                "device-resident fp32 input, no augmentation"}
        del opt
        model.eval()
        for b in (1, 64):
            xb = x[:b].contiguous()
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                for _ in range(10):
                    model(xb)
                torch.cuda.synchronize()
                times = []
                for _ in range(50):
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record()
                    model(xb)
                    a1.record()
                    a1.synchronize()
                    times.append(a0.elapsed_time(a1))
            times.sort()
            out[f"infer_batch{b}"] = {"p50_ms": round(times[25], 4), "pairs_per_s": round(b / (times[25] / 1e3), 1),
                                      "what": "eval forward, eager, bf16 autocast, channels_last"}
    except Exception as exc:  # the baseline must never take the product's bench line down with it
        out["error"] = f"{type(exc).__name__}: {exc}"[:300]
    finally:
        torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own algorithm on the host cores (oracle port; the reference is pure PyTorch/CPU)
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_step_fn(sample_pairs: int, size: int, augmentation: bool):
    import numpy as np
    import torch

    from oracle.ref_model import make_reference_model, torch_loss

    torch.set_num_threads(os.cpu_count() or 1)
    model = make_reference_model(42)
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    images_u8, targets = synthetic_batch(sample_pairs, 2, size, size, seed=0)
    aug = None
    if augmentation:
        try:
            from oracle import augment as oracle_aug
            aug = oracle_aug
        except ImportError:
            aug = None

    def step(i: int) -> float:
        if aug is not None:
            x = aug.augment_batch_u8(images_u8.numpy(), seed=i)          # (B, n_cams, 3, H, W) float32
            x = torch.from_numpy(np.ascontiguousarray(x)).reshape(sample_pairs, 6, size, size)
        else:
            x = (images_u8.permute(0, 1, 4, 2, 3).reshape(sample_pairs, 6, size, size).float() / 255.0)
        opt.zero_grad()
        loss = torch_loss(model(x), targets).mean().float()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        return float(loss)

    return step


def cpu_reference_throughput(sample_pairs: int, iters: int, warmup: int, size: int, augmentation: bool) -> dict:
    step = cpu_reference_step_fn(sample_pairs, size, augmentation)
    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(iters):
        step(warmup + i)
    dt = time.perf_counter() - t0
    return {"value": round(sample_pairs * iters / dt, 3), "unit": "pairs/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"{iters} steps of {sample_pairs} pairs at {size}x{size} (fp32 PyTorch CPU: oracle/ref_model.py = "
                      f"argus/models.py + loss + clip + Adam{' + oracle augmentation' if augmentation else ''}), after {warmup} warm-up"}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = CPU_SAMPLE_PAIRS
    aug_available = (ROOT / "oracle" / "augment.py").exists() and not args.no_augmentation
    step = cpu_reference_step_fn(sample, args.size, aug_available)
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": "train image-pairs/sec", "value": round(value, 3), "unit": "pairs/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"configs[1] train step (bounded sample: {sample} pairs per step on the host cores)",
                   "per_step_pairs": sample, "image_size": [args.size, args.size], "augmentation": aug_available},
        "cpu_baseline": {"value": round(value, 3), "unit": "pairs/s", "cores": os.cpu_count(), "kind": "port",
                         "sample": f"{args.steps} steps of {sample} pairs, fp32 PyTorch CPU port of the reference path"},
        "e2e": {"value": round(value, 3), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="image pairs per GPU")
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--no-augmentation", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-inference", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, about 34 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
