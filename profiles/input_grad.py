"""Cost of the input gradient at the bench configuration (B = 256 pairs, 256 x 256, N = 512 images).

(a) argus_stem_dgrad alone: CUDA events around >= 50 launches after warm-up, algorithmic bytes / FLOPs and the share of
    the HBM floor (the 1.47 GB the kernel must move at the 6.46 TB/s a 1:1 copy reaches, profiles/r1e_hbm_mix.txt);
(b) the autograd forward + backward of NCameraCNN on an fp32 batch, with and without x.requires_grad, alternated in one
    process over several repetitions: the difference is what asking for x.grad costs a training step.

Writes one JSON object (with the device name and power limit read in the same run) to --out.
    python profiles/input_grad.py --out profiles/input_grad.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

HBM_COPY_TBPS = 6.46   # measured 1:1 read/write rate of a B200 (profiles/r1e_hbm_mix.txt)


def device_info() -> dict:
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        info.update({"nvidia_smi_name": name, "power_limit": power, "max_sm_clock": clock})
    except Exception as e:  # the timing is still worth recording; say why the settings are missing
        info["nvidia_smi_error"] = repr(e)
    return info


def time_kernel(B: int, H: int, W: int, launches: int) -> dict:
    from argus_b200 import _lib

    dev = torch.device("cuda", 0)
    N = 2 * B
    g = torch.Generator(device=dev).manual_seed(0)
    dy = torch.randn(N, H // 2, W // 2, 64, device=dev, generator=g).to(torch.bfloat16)
    wp = (torch.randn(64, 256, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    dx = torch.empty(N, 3, H, W, device=dev)
    args = (dy, wp, dx, N, H, W, _lib.stream_ptr())
    for _ in range(10):
        _lib.call("argus_stem_dgrad", *args)
    torch.cuda.synchronize()
    times = []
    for _ in range(launches):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.call("argus_stem_dgrad", *args)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = statistics.median(times)
    pixels = N * (H // 2) * (W // 2)
    bytes_rd, bytes_wr = pixels * 64 * 2, N * 3 * H * W * 4
    flops_alg = 2.0 * pixels * 64 * 147          # every (dy element, 7x7x3 weight) product
    flops_mma = 2.0 * pixels * 64 * 256          # what the padded 16-tap x 16-channel GEMM issues
    floor_ms = (bytes_rd + bytes_wr) / (HBM_COPY_TBPS * 1e12) * 1e3
    return {"N_images": N, "H": H, "W": W, "launches": launches, "ms_median": round(ms, 4),
            "ms_min": round(min(times), 4), "ms_max": round(max(times), 4),
            "bytes_read": bytes_rd, "bytes_written": bytes_wr, "achieved_TBps": round((bytes_rd + bytes_wr) / ms / 1e9, 3),
            "flops_algorithmic": flops_alg, "flops_mma": flops_mma,
            "achieved_TFLOPs_algorithmic": round(flops_alg / ms / 1e9, 1),
            "hbm_floor_ms_at_6.46TBps": round(floor_ms, 4), "share_of_hbm_floor": round(floor_ms / ms, 3)}


def time_autograd(B: int, H: int, W: int, reps: int, iters: int) -> dict:
    from argus_b200.loss import geometric_loss_fn
    from argus_b200.models import NCameraCNN

    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1)
    model = NCameraCNN().to(dev).train()
    x = torch.rand(B, 6, H, W, device=dev, generator=g)
    q = torch.randn(B, 4, device=dev, generator=g)
    target = torch.cat([torch.randn(B, 3, device=dev, generator=g), q / q.norm(dim=-1, keepdim=True)], -1)

    def step(need_x: bool) -> float:
        xi = x.detach().requires_grad_(need_x)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        loss = geometric_loss_fn(model(xi), target).mean()
        loss.backward()
        e1.record()
        e1.synchronize()
        for p in model.parameters():
            p.grad = None
        return e0.elapsed_time(e1)

    for need in (False, True, False, True):
        step(need)   # warm-up: plans, tensor maps, allocator
    per_rep = []
    for _ in range(reps):
        base = statistics.median(step(False) for _ in range(iters))
        with_x = statistics.median(step(True) for _ in range(iters))
        per_rep.append((base, with_x))
    diffs = [w - b for b, w in per_rep]
    return {"B": B, "H": H, "W": W, "reps": reps, "iters_per_rep": iters,
            "ms_without_x_grad": [round(b, 3) for b, _ in per_rep], "ms_with_x_grad": [round(w, 3) for _, w in per_rep],
            "diff_ms_mean": round(statistics.mean(diffs), 3), "diff_ms_stdev": round(statistics.stdev(diffs), 3),
            "diff_ms_min": round(min(diffs), 3), "diff_ms_max": round(max(diffs), 3)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256, help="image pairs")
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: timings are only meaningful on the B200")
    res = {"what": "input gradient (argus_stem_dgrad + argus_model_input_grad) at the bench configuration"}
    res.update(device_info())
    res["stem_dgrad_kernel"] = time_kernel(args.batch, args.size, args.size, args.launches)
    res["autograd_fwd_bwd"] = time_autograd(args.batch, args.size, args.size, args.reps, args.iters)
    text = json.dumps(res, indent=1)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
