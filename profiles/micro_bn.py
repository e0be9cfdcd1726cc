"""Micro-benchmark: batch-norm backward (reduce + apply) and the statistics-carrying wide 1x1 forward convolutions at
the bench shapes (B=256 pairs -> 512 images), through the C ABI, per kernel family with the library's own CUDA-event
profiler. A/B: MICRO_LIB=path runs another build of the library (e.g. the parent commit's) instead of the in-tree one.
Usage: python profiles/micro_bn.py [reps]"""
import ctypes
import json
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from argus_b200 import _lib  # noqa: E402

if os.environ.get("MICRO_LIB"):   # A/B against another build of the library
    _lib.LIB_PATH = Path(os.environ["MICRO_LIB"]).resolve()

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
dev = torch.device("cuda", 0)
lib = _lib.load()
PEAK = 6456.5


def families(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    lib.argus_profile_enable(1)
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    _lib.check(lib.argus_profile_report(buf, ctypes.c_int(1 << 16)))
    lib.argus_profile_enable(0)
    return json.loads(buf.value.decode())


def show(tag, rep):
    for fam, f in rep.items():
        ms = f["ms"] / max(1, f["launches"])
        gbs = f["bytes"] / max(1, f["launches"]) / ms / 1e6 if f["bytes"] else 0.0
        tf = f["flops"] / max(1, f["launches"]) / ms / 1e9 if f["flops"] else 0.0
        print(f"{tag:34s} {fam:16s} {ms * 1e3:9.1f} us  {gbs:8.1f} GB/s ({gbs / PEAK:5.1%})  {tf:7.1f} TF/s", flush=True)


def bf(*shape):
    return torch.randn(*shape, device=dev).bfloat16()


# batch-norm backward at the shapes of one training step (rows, C, mask_mode)
for rows, C, mask in [(2097152, 64, 1), (524288, 128, 1), (131072, 256, 1), (32768, 512, 1), (32768, 2048, 0),
                      (2097152, 128, 1), (131072, 1024, 0), (524288, 512, 3)]:
    dy = bf(rows, C); x = bf(rows, C); dx = torch.empty_like(x)
    sc = torch.rand(C, device=dev) + 0.5; sh = torch.randn(C, device=dev)
    mean = torch.randn(C, device=dev) * 0.1; invstd = torch.rand(C, device=dev) + 0.5
    dgamma = torch.zeros(C, device=dev); dbeta = torch.zeros(C, device=dev)
    out = torch.randint(0, 256, (rows, C // 8), device=dev, dtype=torch.uint8) if mask == 3 else None
    rep = families(lambda: _lib.call("argus_bn_backward", dy, x, out, sc, sh, mean, invstd, dgamma, dbeta, dx,
                                     _lib.c_int64(rows), C, mask, _lib.stream_ptr()))
    show(f"bn_bwd R{rows} C{C} m{mask}", rep)
    del dy, x, dx, out

# forward 1x1 / 3x3 convolutions that carry the BN statistics in their epilogue (HBM-bound wide outputs)
N = 512
for H, Cin, Cout, k in [(64, 64, 256, 1), (32, 128, 512, 1), (16, 256, 1024, 1), (64, 256, 64, 1), (64, 64, 64, 3),
                        (32, 128, 128, 3)]:
    x = bf(N, H, H, Cin); w = bf(Cout, k, k, Cin); y = torch.empty(N, H, H, Cout, device=dev, dtype=torch.bfloat16)
    slots = ctypes.c_int(0)
    _lib.check(lib.argus_conv2d_stat_slots(N, H, H, Cin, Cout, k, 1, 0, ctypes.byref(slots)))
    stat = torch.zeros(slots.value, 2, Cout, device=dev)
    for use_stats in (0, 1):
        rep = families(lambda: _lib.call("argus_conv2d_forward", x, w, y, N, H, H, Cin, Cout, k, 1, 0, None, None, None, 0,
                                         stat if use_stats else None, slots.value if use_stats else 0, _lib.stream_ptr()))
        for f in rep.values():   # report HBM bytes for the conv too
            f["bytes"] = f["launches"] * 2.0 * N * H * H * (Cin + Cout)
        show(f"conv{k}x{k} {Cin}->{Cout} @{H} stats={use_stats}", rep)
    del x, w, y, stat
