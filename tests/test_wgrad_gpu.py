"""Every weight-gradient GEMM path (wgrad_kernel<64|128|256>, wgrad_xpose_kernel<4|10>, wgrad_reduce_kernel) against
the float64 reference of tests/wgrad_ref.py, element by element, through every split-K geometry the planner produces.

Each case pins the kernel instance it must reach and, where the geometry is the point of the case, the split-K
geometry: a predicate on the plan. Geometries depend on the SM count, so such cases search their shape at run time with
the planning mirror over a fixed candidate list, and every case asserts that argus_conv2d_wgrad_launch_info reports
exactly what the mirror planned. Every case runs an exact-integer variant (bit for bit against float64) and a real bf16
variant (rounding bound), each from dW = 0 three times (bitwise reproducible) and once from a random start D (must be
fl(D + result from 0) bit for bit: every path adds into dW with one rounding). dW sits between two 4 KB sentinels, and
the split-K scratch is filled with NaN (0xff bytes) through the library's own scratch before every launch.
"""
import ctypes
import itertools
import time
import zlib

import pytest
import torch

import wgrad_ref as wr
from argus_b200 import _lib

pytestmark = pytest.mark.gpu


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------------------------
# geometry predicates (p = wr.plan(...))
# ------------------------------------------------------------------------------------------------------------------
def one_split(p, S):
    return p["splits"] == 1 and p["kblocks"] >= 2


def ragged_splits(p, S):   # several splits, the last one shorter than the others
    return 1 < p["splits"] and p["kblocks"] - p["per"] * (p["splits"] - 1) < p["per"] and p["capped"] == p["splits"]


def capped_by_kblocks(p, S):   # the SM count asked for more splits than kblocks / 4 allows
    return 2 <= p["capped"] < p["uncapped"] and p["splits"] == p["capped"]


def shrunk(p, S):   # the no-empty-split loop lowered the count
    return 1 < p["splits"] < p["capped"]


def many_splits(p, S):   # the reduce's 8-way unrolled loop plus its 4-group tail
    return p["splits"] >= 32 and p["splits"] % 4 != 0


def grid_stride(p, S):   # the reduce's grid is capped at 4 x SMs blocks of 64 float4: each block loops
    return p["splits"] > 1 and -(-p["rows"] * p["ktot"] // 4 // 64) > 4 * S


def fewer_than_sms(p, S):
    return 1 < p["splits"] < S


def all_sms_ragged(p, S):
    return p["splits"] == S and p["kblocks"] % S != 0


def tile_candidates(cin):
    """1x1 / 3x3 shapes with Cin = cin, cheapest first (the planner picks BLOCK_N from Cin alone)."""
    out = []
    for N, H, cout, k, s in itertools.product((1, 2, 3, 4, 5, 6, 8, 12, 16, 20, 24, 33, 40, 48, 64),
                                              (1, 2, 4, 8, 16, 32, 64), (128, 256, 512, 1024), (1, 3), (1, 2)):
        if H % s or (k == 3 and H < 2):
            continue
        out.append((N, H, H, cin, cout, k, s, 0))
    return out


def xpose_candidates(stem):
    # all SMs with a ragged last split and no shrink needs kblocks = S m + r with r > S - 1 - m: m of about S / 2, so
    # the largest candidates reach 16 384 k-blocks (layer1 at batch 256)
    Ns = (1, 2, 3, 4, 5, 6, 8, 12, 16, 24, 32, 48, 64, 128, 200, 256)
    if stem:
        return [(N, H, H, 3, 64, 7, 2, 1) for N in Ns for H in (32, 64, 128, 256)]
    return [(N, H, H, 64, 64, 3, 1, 0) for N in Ns for H in (8, 16, 32, 64)]


def cost(mode, shape, S):
    p = wr.plan(mode, shape, S)
    return p["pixels"] * p["rows"] * p["ktot"] + 64 * p["scratch"], shape


def C(name, mode, inst, shape=None, geometry=None, candidates=None, data=None):
    """inst: (xpose, n) the launch must run; geometry: predicate on the plan; candidates: shapes to search."""
    return dict(name=name, mode=mode, inst=inst, shape=shape, geometry=geometry, candidates=candidates, data=data)


CASES = []
for bn, cin in ((64, 64), (128, 128), (256, 256)):
    for label, pred in (("one_split", one_split), ("ragged_splits", ragged_splits), ("capped", capped_by_kblocks),
                        ("shrunk", shrunk), ("many_splits", many_splits), ("reduce_grid_stride", grid_stride)):
        CASES.append(C(f"tile{bn}_{label}", "conv", (0, bn), geometry=pred, candidates=tile_candidates(cin)))
CASES += [
    # tile kernel shapes (N, H, W, Cin, Cout, k, stride, kind)
    C("cout64_1x1_halfM", "conv", (0, 256), (2, 64, 64, 256, 64, 1, 1, 0)),
    C("cout64_1x1_single_box", "conv", (0, 64), (3, 32, 32, 64, 64, 1, 1, 0)),
    C("cout64_1x1_many", "conv", (0, 256), (8, 64, 64, 256, 64, 1, 1, 0)),
    C("down_1x1_s2", "conv", (0, 256), (2, 64, 64, 256, 512, 1, 2, 0)),
    C("c1x1_64_256", "conv", (0, 64), (4, 64, 64, 64, 256, 1, 1, 0)),
    C("c1x1_64_256_b8", "conv", (0, 64), (8, 64, 64, 64, 256, 1, 1, 0)),
    C("c1x1_1024_256", "conv", (0, 256), (2, 16, 16, 1024, 256, 1, 1, 0)),
    C("c1x1_512_2048", "conv", (0, 256), (4, 8, 8, 512, 2048, 1, 1, 0)),
    C("c1x1_128_512", "conv", (0, 128), (16, 32, 32, 128, 512, 1, 1, 0)),
    C("c3x3_s1_512", "conv", (0, 256), (2, 8, 8, 512, 512, 3, 1, 0)),
    C("c3x3_s1_128", "conv", (0, 128), (20, 32, 32, 128, 128, 3, 1, 0)),
    C("c3x3_s1_64_128", "conv", (0, 64), (3, 16, 16, 64, 128, 3, 1, 0)),
    C("c3x3_s1_128_64", "conv", (0, 128), (2, 8, 16, 128, 64, 3, 1, 0)),
    C("c3x3_s2_128", "conv", (0, 128), (2, 64, 64, 128, 128, 3, 2, 0)),
    C("c3x3_s2_256", "conv", (0, 256), (6, 16, 16, 256, 256, 3, 2, 0)),
    C("c3x3_s2_512", "conv", (0, 256), (2, 16, 16, 512, 512, 3, 2, 0)),
    C("howo4_ragged_kblock", "conv", (0, 256), (5, 2, 2, 256, 256, 3, 1, 0)),          # 16 images per box, N = 5
    C("howo16_ragged_kblock", "conv", (0, 256), (2, 4, 4, 512, 512, 3, 1, 0)),         # 4 images per box, N = 2
    C("howo16_s2_ragged_kblock", "conv", (0, 128), (7, 8, 8, 128, 256, 3, 2, 0)),
    C("wo128", "conv", (0, 128), (1, 128, 128, 128, 128, 3, 1, 0)),                      # 64-pixel row segments
    C("fc_ragged_m", "conv", (0, 256), (300, 1, 1, 2048, 1024, 1, 1, 0)),
    # stacked [dy | x]^T x and the pure Gram matrix
    C("stacked_cin64", "stacked", (0, 64), (4, 16, 16, 64, 256, 1, 1, 0)),              # second x box out of bounds
    C("stacked_cin256_s2", "stacked", (0, 256), (2, 16, 16, 256, 512, 1, 2, 0)),
    C("stacked_cin128", "stacked", (0, 128), (20, 32, 32, 128, 512, 1, 1, 0)),
    C("stacked_cin512_s2", "stacked", (0, 256), (4, 16, 16, 512, 1024, 1, 2, 0)),
    C("gram_s1", "gram", (0, 128), (2, 32, 32, 128, 128, 1, 1, 0)),
    C("gram_s2", "gram", (0, 256), (4, 16, 16, 256, 256, 1, 2, 0)),
    C("gram_cin256_splits", "gram", (0, 256), (4, 32, 32, 256, 256, 1, 1, 0)),   # the fused block tail's Gram
    C("gram_cin64_s1", "gram", (0, 64), (4, 16, 16, 64, 64, 1, 1, 0)),
    # transposed all-taps kernel
    C("stem_small", "conv", (1, 4), (2, 64, 64, 3, 64, 7, 2, 1)),
    C("stem_256", "conv", (1, 4), (3, 256, 256, 3, 64, 7, 2, 1)),
    C("stem_one_split", "conv", (1, 4), geometry=one_split, candidates=xpose_candidates(True)),
    C("stem_fewer_than_sms", "conv", (1, 4), geometry=fewer_than_sms, candidates=xpose_candidates(True)),
    C("stem_all_sms_ragged", "conv", (1, 4), geometry=all_sms_ragged, candidates=xpose_candidates(True)),
    C("l1_3x3", "conv", (1, 10), (4, 64, 64, 64, 64, 3, 1, 0)),
    C("l1_3x3_one_split", "conv", (1, 10), geometry=one_split, candidates=xpose_candidates(False)),
    C("l1_3x3_fewer_than_sms", "conv", (1, 10), geometry=fewer_than_sms, candidates=xpose_candidates(False)),
    C("l1_3x3_all_sms_ragged", "conv", (1, 10), geometry=all_sms_ragged, candidates=xpose_candidates(False)),
    C("l1_3x3_model_b256", "conv", (1, 10), (256, 64, 64, 64, 64, 3, 1, 0)),
]
BY_NAME = {c["name"]: c for c in CASES}
_resolved = {}


def resolve(case):
    """(shape, plan) of a case on this device's SM count."""
    name = case["name"]
    if name not in _resolved:
        S = sms()
        if case["shape"] is not None:
            shape = case["shape"]
        else:
            fits = [s for s in case["candidates"] if case["geometry"](wr.plan(case["mode"], s, S), S)
                    and (wr.plan(case["mode"], s, S)["xpose"], wr.plan(case["mode"], s, S)["n"]) == case["inst"]]
            assert fits, f"{name}: no candidate shape reaches this geometry on {S} SMs"
            shape = min(fits, key=lambda s: cost(case["mode"], s, S))
        _resolved[name] = (shape, wr.plan(case["mode"], shape, S))
    return _resolved[name]


def query(mode, shape):
    N, H, W, Cin, Cout, k, s, kind = shape
    out = (ctypes.c_int * 11)()
    _lib.call("argus_conv2d_wgrad_launch_info", wr.MODES[mode], N, H, W, Cin, Cout, k, s, kind, out, 11)
    return tuple(out)


def key_of(p):   # what launch_wgrad records: (xpose, n, stacked, co_split > 0, splits > 1)
    return (p["xpose"], p["n"], p["stacked"], int(p["co_split"] > 0), int(p["splits"] > 1))


def recorded_wgrad_keys():
    n = ctypes.c_int()
    _lib.call("argus_wgrad_instances_get", None, 0, ctypes.byref(n))
    buf = (ctypes.c_int * (5 * n.value))()
    _lib.call("argus_wgrad_instances_get", buf, 5 * n.value, ctypes.byref(n))
    return {tuple(buf[5 * i:5 * i + 5]) for i in range(n.value)}


def compiled_wgrad_instances():
    n = ctypes.c_int()
    _lib.call("argus_wgrad_instances_all", None, 0, ctypes.byref(n))
    buf = (ctypes.c_int * (2 * n.value))()
    _lib.call("argus_wgrad_instances_all", buf, 2 * n.value, ctypes.byref(n))
    return {tuple(buf[2 * i:2 * i + 2]) for i in range(n.value)}


def launch(mode, shape, dy, x, p, start):
    """One launch into a fresh [sentinel | dW = start | sentinel] buffer, after filling the scratch with NaN."""
    N, H, W, Cin, Cout, k, s, kind = shape
    n = p["rows"] * p["ktot"]
    buf = torch.full((2 * wr.SENTINEL + n,), wr.SENTINEL_VALUE, device=x.device)
    buf[wr.SENTINEL:wr.SENTINEL + n] = start.reshape(-1)
    dw = buf[wr.SENTINEL:wr.SENTINEL + n]
    st = _lib.stream_ptr()
    _lib.call("argus_lib_scratch_fill", _lib.c_int64(p["scratch"]), 0xff, st)
    if mode == "conv":
        _lib.call("argus_conv2d_wgrad", dy, x, dw, N, H, W, Cin, Cout, k, s, kind, st)
    elif mode == "stacked":
        _lib.call("argus_conv2d_wgrad_gram", dy, x, dw, N, H, W, Cin, Cout, s, st)
    else:
        _lib.call("argus_conv2d_gram", x, dw, N, H, W, Cin, Cout, s, st)
    torch.cuda.synchronize()
    wr.check_sentinels(buf, n, p, f"{mode} {shape}")
    return dw.view(p["rows"], p["ktot"]).clone()


@pytest.mark.parametrize("name", list(BY_NAME))
def test_wgrad_case(cuda_device, name):
    case = BY_NAME[name]
    mode = case["mode"]
    shape, p = resolve(case)
    info = query(mode, shape)
    assert info == wr.info_tuple(p), f"{name} {shape}: library plans {info}, mirror {wr.info_tuple(p)}"
    assert (p["xpose"], p["n"]) == case["inst"], f"{name}: reaches {(p['xpose'], p['n'])}"
    if case["geometry"] is not None:
        assert case["geometry"](p, sms()), f"{name}: geometry {p}"
    t0 = time.perf_counter()
    gen = torch.Generator(device=cuda_device).manual_seed(zlib.crc32(name.encode()))
    worst = None
    _lib.call("argus_conv_instances_record", 1)
    try:
        for exact in (True, False):
            what = f"{name} {shape} {'exact' if exact else 'real'}"
            dy, x = wr.make_operands(mode, shape, exact, gen, cuda_device)
            prob = wr.Problem(mode, shape, dy, x)
            ref, A = prob.reference()
            zero = torch.zeros(p["rows"], p["ktot"], device=cuda_device)
            runs = [launch(mode, shape, dy, x, p, zero) for _ in range(3)]
            for r in runs[1:]:
                assert torch.equal(r.view(torch.int32), runs[0].view(torch.int32)), f"{what}: not reproducible"
            if exact:
                wr.check_exact(prob, runs[0], ref, A, p, what)
            else:
                worst = wr.check_bound(prob, runs[0], ref, A, p, what)
            D = torch.randn(p["rows"], p["ktot"], generator=gen, device=cuda_device)
            wr.check_accumulated(launch(mode, shape, dy, x, p, D), D, runs[0], p, what + " from D")
            del dy, x, prob, ref, A, runs
    finally:
        _lib.call("argus_conv_instances_record", 0)
    assert recorded_wgrad_keys() == {key_of(p)}
    print(f"{name}: shape {shape} {'xpose' if p['xpose'] else 'tile'} n={p['n']} splits {p['splits']} "
          f"(asked {p['uncapped']}, capped {p['capped']}) k-blocks {p['kblocks']} per split {p['per']} "
          f"grid {p['grid']} scratch {p['scratch']}: exact bit for bit, largest err/bound {worst:.3f} "
          f"({time.perf_counter() - t0:.2f} s)")
    torch.cuda.empty_cache()


def test_plan_mirror_matches_library(cuda_device):
    S = sms()
    shapes = [(N, H, H, cin, cout, k, s, 0) for N in (1, 3, 40) for H in (2, 8, 32) for cin in (64, 128, 256, 512)
              for cout in (64, 128, 256, 2048) for k in (1, 3) for s in (1, 2)]
    shapes += [(N, H, H, 3, 64, 7, 2, 1) for N in (1, 2, 5, 16) for H in (32, 64, 128, 256)]
    for shape in shapes:
        assert query("conv", shape) == wr.info_tuple(wr.plan("conv", shape, S)), shape
        if shape[7] == 0 and shape[5] == 1:
            if shape[4] % 128 == 0:
                assert query("stacked", shape) == wr.info_tuple(wr.plan("stacked", shape, S)), shape
            assert query("gram", shape) == wr.info_tuple(wr.plan("gram", shape, S)), shape


def test_model_launches_only_pinned_wgrad_keys(cuda_device):
    """Every weight-gradient key a training step, a frozen-statistics backward and the algebraic conv + BN backward
    launch is one a case above pins, and every compiled instance has a case."""
    from argus_b200.engine import TrainEngine
    from argus_b200.models import NCameraCNN
    from gpu_util import random_targets, structured_images

    table = {key_of(resolve(c)[1]) for c in CASES}
    insts = {c["inst"] for c in CASES}
    assert compiled_wgrad_instances() <= insts, sorted(compiled_wgrad_instances() - insts)
    seen = {}

    def record(label, fn):
        _lib.call("argus_conv_instances_record", 1)
        try:
            fn()
            torch.cuda.synchronize()
        finally:
            _lib.call("argus_conv_instances_record", 0)
        seen[label] = recorded_wgrad_keys()

    for B, H, frozen in ((256, 256, False), (8, 128, False), (16, 256, True)):
        model = NCameraCNN().to(cuda_device)
        model.eval() if frozen else model.train()
        eng = TrainEngine(model, lr=1e-4, max_grad_norm=1.0, distributed=False, frozen_bn=frozen)
        x = structured_images(B, 6, H, H, 1, cuda_device)
        record(f"{'frozen' if frozen else 'train'} B={B} {H}x{H}",
               lambda: eng.forward_backward(x, random_targets(B, 2, cuda_device)))
        del model, eng, x
        torch.cuda.empty_cache()

    N, H, W, C, O = 4, 16, 16, 64, 256
    g = torch.Generator(device=cuda_device).manual_seed(0)
    up = torch.randn(N * H * W, O, generator=g, device=cuda_device).bfloat16()
    act = torch.randn(N, H, W, C, generator=g, device=cuda_device).relu().bfloat16()
    w = torch.randn(O, C, generator=g, device=cuda_device).bfloat16()
    ones, zeros = torch.ones(O, device=cuda_device), torch.zeros(O, device=cuda_device)
    record("argus_conv_bn_backward_algebraic", lambda: _lib.call(
        "argus_conv_bn_backward_algebraic", up, act, w, up.float().sum(0), ones, zeros, ones, torch.zeros(O, device=cuda_device),
        torch.zeros(O, device=cuda_device), torch.zeros(O, C, device=cuda_device), torch.empty_like(act), N, H, W, C, O, 1,
        _lib.stream_ptr()))
    for label, keys in seen.items():
        print(f"{label}: wgrad keys (xpose, n, stacked, co_split > 0, splits > 1) {sorted(keys)}")
        assert keys, f"{label}: no weight-gradient launch recorded"
    missing = {k: sorted(v - table) for k, v in seen.items() if v - table}
    assert not missing, f"weight-gradient keys launched that no case pins: {missing}"
