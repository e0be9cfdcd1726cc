"""Cost of the frozen-statistics (differentiable eval-mode) path at B = 1, 64 and 256 image pairs, 256 x 256.

Per batch size, with CUDA events around each call after warm-up (median of --iters):
  eval_forward_ms      the no-grad eval forward (argus_model_forward, training = 0)
  frozen_forward_ms    the same forward with bit masks and arg-max bytes (argus_model_forward_frozen)
  frozen_backward_ms   argus_model_backward of that forward, all four stages
  train_fwd_bwd_ms     a training forward + backward for comparison (not at B = 1: train mode rejects it)
and the un-pool kernel of the stem (argus_stem_unpool_relu) against the two-term HBM model of DESIGN.md section 4,
t = R / 7.2 TB/s + W / 5.0 TB/s.

Writes one JSON object (with the device name and power limit read in the same run) to --out.
    python profiles/frozen_bn.py --out profiles/frozen_bn.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from input_grad import device_info  # noqa: E402

READ_TBPS, WRITE_TBPS = 7.2, 5.0


def timed(fn, iters: int) -> float:
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times)


def time_model(B: int, H: int, iters: int) -> dict:
    from argus_b200 import _lib
    from argus_b200.models import NCameraCNN

    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(B)
    x = torch.rand(B, 6, H, H, device=dev, generator=g)
    d_out = torch.randn(B, 6, device=dev, generator=g)
    model = NCameraCNN().to(dev).eval()
    ptr, st = model._handle.ptr, _lib.stream_ptr()

    def backward():
        _lib.call("argus_model_zero_grads", ptr, st)
        _lib.call("argus_model_backward", ptr, d_out, 0, 4, st)

    res = {"B": B, "H": H, "W": H}
    with torch.no_grad():
        for _ in range(3):
            model._forward_impl(x, False)
            model._forward_impl(x, False, frozen=True)
            backward()
        res["eval_forward_ms"] = round(timed(lambda: model._forward_impl(x, False), iters), 3)
        res["frozen_forward_ms"] = round(timed(lambda: model._forward_impl(x, False, frozen=True), iters), 3)
        bwd = []
        for _ in range(iters):
            model._forward_impl(x, False, frozen=True)
            bwd.append(timed(backward, 1))
        res["frozen_backward_ms"] = round(statistics.median(bwd), 3)
        if B > 1:
            tm = NCameraCNN().to(dev).train()
            tptr = tm._handle.ptr

            def train_step():
                tm._forward_impl(x, True)
                _lib.call("argus_model_zero_grads", tptr, st)
                _lib.call("argus_model_backward", tptr, d_out, 0, 4, st)

            for _ in range(3):
                train_step()
            res["train_fwd_bwd_ms"] = round(timed(train_step, iters), 3)
            del tm
    del model
    torch.cuda.empty_cache()
    return res


def time_unpool(B: int, H: int, launches: int) -> dict:
    from argus_b200 import _lib

    dev = torch.device("cuda", 0)
    N, H1 = 2 * B, H // 2
    g = torch.Generator(device=dev).manual_seed(3)
    act = torch.relu(torch.randn(N, H1, H1, 64, device=dev, generator=g)).to(torch.bfloat16)
    pooled = torch.empty(N, H1 // 2, H1 // 2, 64, dtype=torch.bfloat16, device=dev)
    idx = torch.empty(N, H1 // 2, H1 // 2, 64, dtype=torch.uint8, device=dev)
    st = _lib.stream_ptr()
    _lib.call("argus_maxpool_forward", act, None, None, pooled, idx, N, H1, H1, 64, st)
    dpool = torch.randn(N, H1 // 2, H1 // 2, 64, device=dev, generator=g).to(torch.bfloat16)
    g0 = torch.empty_like(act)
    sums = torch.empty(64, device=dev)
    call = lambda: _lib.call("argus_stem_unpool_relu", dpool, idx, pooled, g0, N, H1, H1, sums, st)
    for _ in range(10):
        call()
    ms = timed(call, launches)
    pix = N * H1 * H1
    rd = pix // 4 * 64 * (2 + 2 + 1)
    wr = pix * 64 * 2
    model_ms = (rd / (READ_TBPS * 1e12) + wr / (WRITE_TBPS * 1e12)) * 1e3
    return {"N_images": N, "stem_H": H1, "stem_W": H1, "launches": launches, "ms_median": round(ms, 4),
            "bytes_read": rd, "bytes_written": wr, "hbm_model_ms": round(model_ms, 4),
            "share_of_hbm_model": round(model_ms / ms, 3)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 64, 256])
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: timings are only meaningful on the B200")
    res = {"what": "frozen-statistics forward / backward (argus_model_forward_frozen) against the eval forward and a "
                   "training step"}
    res.update(device_info())
    res["model"] = [time_model(B, args.size, args.iters) for B in args.batches]
    res["stem_unpool_relu"] = time_unpool(max(args.batches), args.size, args.launches)
    text = json.dumps(res, indent=1)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
