"""Every conv_gemm_kernel instance (csrc/conv_gemm.cuh, dispatched by launch_conv in csrc/conv_ops.cu) against a
float64 reference of its epilogue, element by element (tests/epilogue_ref.py), and the Gram-matrix batch statistics of
the fused forward block tail against float64 batch norm.

Each case names the instance it must reach (BLOCK_N, option mask, halo, weights resident), asserted through
argus_conv2d_launch_info before it runs. Outputs are NaN-filled before the launch and followed by a 4 KB sentinel that
must stay untouched; every case runs three times (twice plainly, once with early_trigger where the instance honours it)
and must reproduce output, bit mask and statistics slots bit for bit.
"""
import ctypes
import zlib

import pytest
import torch
import torch.nn.functional as F

import epilogue_ref as er
from argus_b200 import _lib
from test_conv_gpu import s2d_pack, stem_pack_w

pytestmark = pytest.mark.gpu

SCALE, SHIFT, RES, RES_AFF, RELU, BITS, OUT_BITS, RES_BITS, STATS, BN_RAW, EARLY = (
    1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024)
TAIL = 1 | 2 | 8        # kOptAffine | kOptRes | kOptRelu
AFF_RELU, AFF, PLAIN, RES_OB, AFF_OB, BNRED, BNRED_B, GENERIC = 9, 1, 0, 6, 5, 34, 35, 31



def C(name, launch, shape, flags, expect, **kw):
    """launch: fwd | stem | dgrad (1x1 dgrad_ex) | dgrad_k (any k, no extras) | dgrad_bits | concat | bnred |
    bnred_concat; shape (N,H,W,Cin,Cout,k,stride); expect (block_n, opt, halo, b_resident)."""
    return dict(name=name, launch=launch, shape=shape, flags=flags, expect=expect, **kw)


S256 = (5, 64, 64, 64, 256, 1, 1)    # 160 M tiles x 1: BLOCK_N 256, tiles just above the grid
S128 = (3, 64, 64, 64, 256, 1, 1)    # 96 x 2 tiles: BLOCK_N 128
S64 = (3, 4, 4, 64, 64, 1, 1)        # 48 rows: one partial M tile, Cout = 64 (one bit-mask word per half chunk)
D256, D128 = (5, 64, 64, 256, 64, 1, 1), (3, 64, 64, 256, 64, 1, 1)   # dgrads: output = the 256 input channels
TB = SCALE | SHIFT | RES | RELU | BITS

CASES = [
    # folded BN, fused block tail (BN + identity + ReLU + bits) and without the bit mask
    C("tail_bits_256", "fwd", S256, TB, (256, TAIL, 0, 0)),
    C("tail_256", "fwd", S256, TB & ~BITS, (256, TAIL, 0, 0)),
    C("tail_bits_128", "fwd", S128, TB, (128, TAIL, 0, 0)),
    C("tail_bits_64_ragged", "fwd", S64, TB, (64, TAIL, 0, 0)),
    C("tail_3x3_halo_resident", "fwd", (2, 32, 32, 64, 64, 3, 1), TB, (64, TAIL, 1, 1)),
    # 156 tiles over 148 CTAs with three N tiles: grid % num_n_tiles != 0, so the weights cannot stay resident
    C("tail_3x3_halo_grid_mod", "fwd", (26, 16, 16, 64, 192, 3, 1), TB, (64, TAIL, 1, 0)),
    C("tail_3x3_halo_128", "fwd", (20, 32, 32, 64, 128, 3, 1), TB & ~BITS, (128, TAIL, 1, 0)),
    # eval-mode folded BN (+ ReLU): conv1 / conv2 / stem / downsample
    C("affrelu_256", "fwd", S256, SCALE | SHIFT | RELU, (256, AFF_RELU, 0, 0)),
    C("affrelu_128_3x3s2", "fwd", (20, 64, 64, 64, 128, 3, 2), SCALE | SHIFT | RELU, (128, AFF_RELU, 0, 0)),
    C("affrelu_64_halo", "fwd", (2, 32, 32, 64, 64, 3, 1), SCALE | SHIFT | RELU, (64, AFF_RELU, 1, 1)),
    C("affrelu_stem", "stem", (2, 128, 128, 3, 64, 7, 2), SCALE | SHIFT | RELU, (64, AFF_RELU, 0, 0)),
    C("affrelu_stem_many_tiles", "stem", (40, 128, 128, 3, 64, 7, 2), SCALE | SHIFT | RELU, (64, AFF_RELU, 0, 0)),
    C("affrelu_halo_grid_mod", "fwd", (26, 16, 16, 64, 192, 3, 1), SCALE | SHIFT | RELU, (64, AFF_RELU, 1, 0)),
    C("affrelu_halo_128", "fwd", (20, 32, 32, 64, 128, 3, 1), SCALE | SHIFT | RELU, (128, AFF_RELU, 1, 0)),
    C("aff_256_s2", "fwd", (5, 128, 128, 64, 256, 1, 2), SCALE | SHIFT, (256, AFF, 0, 0)),
    C("aff_128_s2", "fwd", (3, 128, 128, 64, 256, 1, 2), SCALE | SHIFT, (128, AFF, 0, 0)),
    C("aff_64_s2", "fwd", (2, 32, 32, 256, 64, 1, 2), SCALE | SHIFT, (64, AFF, 0, 0)),
    # generic kernel: block tail whose downsample is normalised on the fly (first blocks of layers 3 and 4)
    C("generic_layer3_tail_256", "fwd", (20, 16, 16, 256, 1024, 1, 1), TB | RES_AFF, (256, GENERIC, 0, 0)),
    C("generic_layer3_tail_64", "fwd", (4, 16, 16, 256, 1024, 1, 1), TB | RES_AFF, (64, GENERIC, 0, 0)),
    C("generic_layer4_tail_128", "fwd", (20, 8, 8, 512, 2048, 1, 1), TB | RES_AFF, (128, GENERIC, 0, 0)),
    C("generic_fc_bias", "fwd", (300, 1, 1, 2048, 512, 1, 1), SHIFT, (64, GENERIC, 0, 0)),
    # plain forward with statistics (every training-forward convolution)
    C("plain_fwd_256", "fwd", S256, STATS, (256, PLAIN, 0, 0)),
    C("plain_fwd_128", "fwd", S128, STATS, (128, PLAIN, 0, 0)),
    C("plain_fwd_64_ragged", "fwd", S64, STATS, (64, PLAIN, 0, 0)),
    C("plain_fwd_halo", "fwd", (2, 32, 32, 64, 64, 3, 1), STATS, (64, PLAIN, 1, 1)),
    C("plain_fwd_halo_128", "fwd", (20, 32, 32, 64, 128, 3, 1), STATS, (128, PLAIN, 1, 0)),
    C("plain_fwd_stem", "stem", (3, 64, 64, 3, 64, 7, 2), STATS, (64, PLAIN, 0, 0)),
    # dgrads
    C("plain_dgrad_256", "dgrad", D256, STATS, (256, PLAIN, 0, 0)),
    C("plain_dgrad_128", "dgrad", D128, STATS, (128, PLAIN, 0, 0)),
    C("plain_dgrad_64_ragged", "dgrad", S64, STATS, (64, PLAIN, 0, 0)),
    C("plain_dgrad_3x3_halo", "dgrad_k", (2, 32, 32, 64, 64, 3, 1), 0, (64, PLAIN, 1, 1)),
    C("plain_dgrad_3x3_halo_128", "dgrad_k", (20, 32, 32, 128, 128, 3, 1), 0, (128, PLAIN, 1, 0)),
    C("res_ob_dgrad_256", "dgrad", D256, RES | OUT_BITS, (256, RES_OB, 0, 0)),
    C("res_ob_dgrad_128", "dgrad", D128, RES | OUT_BITS, (128, RES_OB, 0, 0)),
    C("res_ob_dgrad_64_ragged", "dgrad", S64, RES | OUT_BITS, (64, RES_OB, 0, 0)),
    C("concat_ob_256", "concat", D256, SHIFT | OUT_BITS, (256, AFF_OB, 0, 0), c1=64),
    C("concat_ob_128", "concat", D128, SHIFT | OUT_BITS, (128, AFF_OB, 0, 0), c1=64),
    C("concat_ob_64_ragged", "concat", S64, SHIFT | OUT_BITS, (64, AFF_OB, 0, 0), c1=128),
    C("concat_s2", "concat", (4, 32, 32, 256, 128, 1, 2), SHIFT, (64, AFF_OB, 0, 0), c1=256),
    C("generic_dgrad_res_bits_256", "dgrad_bits", D256, RES | RES_BITS, (256, GENERIC, 0, 0)),
    C("generic_dgrad_res_bits_128", "dgrad_bits", D128, RES | RES_BITS, (128, GENERIC, 0, 0)),
    C("generic_dgrad_res_bits_64", "dgrad_bits", S64, RES | RES_BITS, (64, GENERIC, 0, 0)),
    # fused BN-backward reduction (ARGUS_BN_REDUCE_FUSED)
    C("bnred_256", "bnred", D256, BN_RAW | STATS, (256, BNRED, 0, 0)),
    C("bnred_128", "bnred", D128, BN_RAW | STATS, (128, BNRED, 0, 0)),
    C("bnred_64_ragged", "bnred", S64, BN_RAW | STATS, (64, BNRED, 0, 0)),
    C("bnred_3x3_halo", "bnred", (2, 32, 32, 64, 64, 3, 1), BN_RAW | STATS, (64, BNRED, 1, 1)),
    C("bnred_3x3_halo_128", "bnred", (20, 32, 32, 128, 128, 3, 1), BN_RAW | STATS, (128, BNRED, 1, 0)),
    C("bnred_concat_256", "bnred_concat", D256, SHIFT | BN_RAW | STATS, (256, BNRED_B, 0, 0), c1=64),
    C("bnred_concat_128", "bnred_concat", D128, SHIFT | BN_RAW | STATS, (128, BNRED_B, 0, 0), c1=64),
    C("bnred_concat_64", "bnred_concat", S64, SHIFT | BN_RAW | STATS, (64, BNRED_B, 0, 0), c1=64),
]
EARLY_OPTS = {TAIL, AFF_RELU, AFF}   # the eval-mode chain sets early_trigger on these


def launch_info(launch, shape, flags, kind=0, c1=0):
    N, H, W, Cin, Cout, k, s = shape
    code = {"fwd": 0, "stem": 0, "dgrad": 1, "dgrad_k": 1, "dgrad_bits": 1, "bnred": 1, "concat": 2, "bnred_concat": 2}[launch]
    out = (ctypes.c_int * 40)()
    n = ctypes.c_int()
    _lib.call("argus_conv2d_launch_info", code, N, H, W, Cin, Cout, k, s, kind, c1, flags, out, 40, ctypes.byref(n))
    return [tuple(out[10 * i:10 * i + 10]) for i in range(n.value)]


def case_info(case):
    return launch_info(case["launch"], case["shape"], case["flags"], 1 if case["launch"] == "stem" else 0,
                       case.get("c1", 0))


def all_instances():
    """(block_n, b_mn, opt) of every instance launch_conv can dispatch to, from the library's own table."""
    n = ctypes.c_int()
    _lib.call("argus_conv_instances_all", None, 0, ctypes.byref(n))
    buf = (ctypes.c_int * (3 * n.value))()
    _lib.call("argus_conv_instances_all", buf, 3 * n.value, ctypes.byref(n))
    return [tuple(buf[3 * i:3 * i + 3]) for i in range(n.value)]


def recorded_keys():
    n = ctypes.c_int()
    _lib.call("argus_conv_instances_get", None, 0, ctypes.byref(n))
    buf = (ctypes.c_int * (5 * n.value))()
    _lib.call("argus_conv_instances_get", buf, 5 * n.value, ctypes.byref(n))
    return {tuple(buf[5 * i:5 * i + 5]) for i in range(n.value)}


def b_mn_of(case):   # forward launches read the weights K-major, dgrads MN-major
    return 0 if case["launch"] in ("fwd", "stem") else 1


def key_of(info):   # the key launch_conv records: (block_n, b_mn, opt, halo, b_resident)
    return info[:5]


def guarded(shape, dtype, dev):
    """Tensor of `shape` followed by a 4 KB sentinel; returns (view, whole buffer)."""
    n = 1
    for d in shape:
        n *= d
    per = 4096 // torch.tensor([], dtype=dtype).element_size()
    buf = torch.empty(n + per, dtype=dtype, device=dev)
    if dtype == torch.uint8:
        buf.fill_(0xA5)
    else:
        buf.view(torch.int16).fill_(0x7FA5)   # a NaN
    return buf[:n].view(shape), buf


def check_sentinel(buf, n, what):
    tail = buf[n:]
    want = 0xA5 if buf.dtype == torch.uint8 else 0x7FA5
    v = tail if buf.dtype == torch.uint8 else tail.view(torch.int16)
    assert bool((v == want).all()), f"{what}: the 4 KB after the tensor were written"


def make_inputs(case, dev, g):
    N, H, W, Cin, Cout, k, s = case["shape"]
    f, launch = case["flags"], case["launch"]
    rnd = lambda *sz: torch.randn(*sz, generator=g).to(dev)
    t = {}
    Cres = Cout if launch in ("fwd", "stem") else Cin          # channels of the result
    rows_out = N * (H // s) * (W // s) if launch in ("fwd", "stem") else N * H * W
    zero_ch = torch.arange(Cres, device=dev) % 5 == 0          # shift 0 here: rows of a zero image give pre == 0
    if launch == "stem":
        img = torch.rand(N, 3, H, W, generator=g).to(dev)
        img[0] = 0
        wt = rnd(64, 3, 7, 7) / 147 ** 0.5
        t["x"], t["w"] = s2d_pack(img), stem_pack_w(wt)
        ib, wb = img.to(torch.bfloat16).double(), wt.to(torch.bfloat16).double()
        acc = F.conv2d(ib, wb, stride=2, padding=3).permute(0, 2, 3, 1).reshape(-1, 64)
        absacc = F.conv2d(ib.abs(), wb.abs(), stride=2, padding=3).permute(0, 2, 3, 1).reshape(-1, 64)
    elif launch == "fwd":
        x = rnd(N, H, W, Cin).to(torch.bfloat16)
        x[0] = 0
        w = (rnd(Cout, k, k, Cin) / (Cin * k * k) ** 0.5).to(torch.bfloat16)
        t["x"], t["w"] = x, w
        acc, absacc = er.conv_nhwc_f64(x, w, k, s)
    else:
        Ho, Wo = H // s, W // s
        dy = rnd(N, Ho, Wo, Cout).to(torch.bfloat16)
        dy[0] = 0
        w = (rnd(Cout, k, k, Cin) / (Cout * k * k) ** 0.5).to(torch.bfloat16)
        acc, absacc = er.dgrad_nhwc_f64(dy, w, k, s)
        if launch in ("concat", "bnred_concat"):
            c1 = case["c1"]
            a1 = rnd(N, H, W, c1).to(torch.bfloat16)
            a1[0] = 0
            b1 = (rnd(c1, Cin) / c1 ** 0.5).to(torch.bfloat16)
            t["a1"] = a1
            wstack = torch.cat([w.reshape(Cout, Cin), b1], 0).contiguous()
            a_s = a1[:, ::s, ::s, :].double().reshape(-1, c1)
            extra = torch.zeros(N, H, W, Cin, dtype=torch.float64, device=dev)
            extra[:, ::s, ::s, :] = (a_s @ b1.double()).reshape(N, H // s, W // s, Cin)
            extra_abs = torch.zeros_like(extra)
            extra_abs[:, ::s, ::s, :] = (a_s.abs() @ b1.double().abs()).reshape(N, H // s, W // s, Cin)
            acc, absacc = acc + extra.reshape(-1, Cin), absacc + extra_abs.reshape(-1, Cin)
            t["w"] = wstack
        else:
            t["w"] = w
        t["dy"] = dy
    t["acc"], t["absacc"] = acc, absacc
    if f & SCALE:
        sc = torch.rand(Cres, generator=g).to(dev) + 0.5
        sc[1::3] *= -1                                          # negative BN scales
        t["scale"] = sc
    if f & SHIFT:
        sh = rnd(Cres)
        sh[zero_ch] = 0
        t["shift"] = sh
    if f & RES:
        r = rnd(rows_out, Cres).to(torch.bfloat16)
        r[:rows_out // N] = 0                                   # image 0
        t["res"] = r
    if f & RES_AFF:
        t["res_scale"] = rnd(Cres)
        rs = rnd(Cres)
        rs[zero_ch] = 0
        t["res_shift"] = rs
    if f & (OUT_BITS | RES_BITS):
        t["in_bits"] = er.bool_to_bits(torch.rand(rows_out, Cres, generator=g).to(dev) > 0.4)
    if f & BN_RAW:
        t["raw"] = rnd(rows_out, Cres).to(torch.bfloat16)
        t["bn_scale"] = rnd(Cres)
        t["bn_shift"] = rnd(Cres) * 0.5
        t["bn_shift"][zero_ch] = 0
        t["raw"][: rows_out // N, :][:, zero_ch] = 0           # raw * s + t == 0 exactly: masked out
    t["rows"], t["C"] = rows_out, Cres
    return t


def run_case(case, t, dev, info, early):
    N, H, W, Cin, Cout, k, s = case["shape"]
    f, launch = case["flags"], case["launch"]
    rows, Cr = t["rows"], t["C"]
    y, ybuf = guarded((rows, Cr), torch.bfloat16, dev)
    bits, bbuf = guarded((rows, Cr // 8), torch.uint8, dev) if f & BITS else (None, None)
    slots = info[9]
    partial = torch.zeros(slots, 2, Cr, device=dev) if f & STATS else None
    st = _lib.stream_ptr()
    if launch in ("fwd", "stem"):
        _lib.call("argus_conv2d_forward_full", t["x"], t["w"], y, N, H, W, Cin, Cout, k, s, int(launch == "stem"),
                  t.get("scale"), t.get("shift"), t.get("res"), t.get("res_scale"), t.get("res_shift"),
                  int(bool(f & RELU)), bits, partial, slots, int(early), st)
    elif launch in ("dgrad", "concat"):
        _lib.call("argus_conv2d_dgrad_ex", t["dy"], t["w"], y, N, H, W, Cin, Cout, s, t.get("a1"),
                  case.get("c1", 0), t.get("shift"), t.get("res"), t.get("in_bits"), partial, slots, st)
    elif launch == "dgrad_k":
        _lib.call("argus_conv2d_dgrad", t["dy"], t["w"], y, N, H, W, Cin, Cout, k, s, None, st)
    elif launch == "dgrad_bits":
        _lib.call("argus_conv2d_dgrad_bits", t["dy"], t["w"], y, N, H, W, Cin, Cout, k, t["res"], t["in_bits"], st)
    else:
        _lib.call("argus_conv2d_dgrad_bnred", t["dy"], t["w"], y, N, H, W, Cin, Cout, k, s, t.get("a1"),
                  case.get("c1", 0), t.get("shift"), t["raw"], t["bn_scale"], t["bn_shift"], partial, slots, st)
    torch.cuda.synchronize()
    check_sentinel(ybuf, rows * Cr, "output")
    if bits is not None:
        check_sentinel(bbuf, rows * Cr // 8, "ReLU bits")
    return y, bits, partial


def reference(case, t):
    f, launch = case["flags"], case["launch"]
    res = t.get("res")
    if launch == "dgrad_bits":
        res = res.double() * er.bits_to_bool(t["in_bits"], t["C"])
    pre, ref, E = er.epilogue_ref(t["acc"], t["absacc"], t.get("scale"), t.get("shift"), res, t.get("res_scale"),
                                  t.get("res_shift"), relu=bool(f & RELU))
    keep = None
    if f & OUT_BITS:
        keep = er.bits_to_bool(t["in_bits"], t["C"])
    if f & BN_RAW:
        keep = (t["raw"].double() * t["bn_scale"].double() + t["bn_shift"].double()) > 0
    if keep is not None:   # masked elements are stored as exact zeros
        ref, E = ref * keep, E * keep
    return pre, ref, E


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_epilogue_instance(cuda_device, case):
    dev = cuda_device
    info = case_info(case)
    assert len(info) == 1
    info = info[0]
    bn, opt, halo, bres = case["expect"]
    assert (info[0], info[1], info[2], info[3], info[4]) == (bn, b_mn_of(case), opt, halo, bres), f"dispatch: {info}"
    g = torch.Generator().manual_seed(zlib.crc32(case["name"].encode()))
    t = make_inputs(case, dev, g)
    N, H, W, Cin, Cout, k, s = case["shape"]
    strided_dgrad = case["launch"] in ("concat",) and s == 2
    # the entry point must launch exactly the instance the planning query predicts
    _lib.call("argus_conv_instances_record", 1)
    try:
        runs = [run_case(case, t, dev, info, False), run_case(case, t, dev, info, False)]
        if opt in EARLY_OPTS:
            early_info = case_info(dict(case, flags=case["flags"] | EARLY))[0]
            assert early_info[:5] == info[:5]
            runs.append(run_case(case, t, dev, info, True))
    finally:
        _lib.call("argus_conv_instances_record", 0)
    assert recorded_keys() == {key_of(info)}
    y, bits, partial = runs[0]
    for y2, bits2, partial2 in runs[1:]:
        assert torch.equal(y.view(torch.int16), y2.view(torch.int16)), "output not reproducible"
        if bits is not None:
            assert torch.equal(bits, bits2), "bit mask not reproducible"
        if partial is not None:
            assert torch.equal(partial, partial2), "statistics slots not reproducible"
    pre, ref, E = reference(case, t)
    if strided_dgrad:
        # pixels no tap reaches are never written (the caller zero-fills): they keep the NaN fill
        even = torch.zeros(N, H, W, dtype=torch.bool, device=dev)
        even[:, ::2, ::2] = True
        even = even.reshape(-1)
        assert bool(torch.isnan(y[~even].float()).all()), "stride-2 dgrad wrote a pixel of another parity class"
        y, pre, ref, E = y[even], pre[even], ref[even], E[even]
    excess = ((y.double() - ref).abs() - er.REL * ref.abs()).clamp_min(0)
    need = float((excess / (E / er.C_ACC).clamp_min(1e-300)).max())
    print(f"{case['name']}: accumulation constant needed {need:.3e} (C_ACC = {er.C_ACC:.3e})")
    worst = er.check_values(y, ref, E, case["name"])
    print(f"{case['name']}: info {info} largest err/bound {worst:.3f}")
    if bits is not None:
        er.check_bits(bits, y, pre, E)
        zero_pre = (pre == 0) & (E == 0)
        assert bool(zero_pre.any()), "case lacks exactly-zero pre-activations"
        assert not bool(er.bits_to_bool(bits, t["C"])[zero_pre].any())
        assert bool((y.float()[zero_pre] <= 0).all())
    if partial is not None:
        if case["flags"] & BN_RAW:
            er.check_stat_slots(partial, y, t["C"], second=t["raw"], what=case["name"] + " sums")
        else:
            er.check_stat_slots(partial, y, t["C"], what=case["name"] + " statistics")


def test_every_instance_has_a_case(cuda_device):
    table = all_instances()
    assert len(table) == len(set(table)) == 33
    hit = {(c["expect"][0], b_mn_of(c), c["expect"][1]) for c in CASES}
    assert hit == set(table), sorted(set(table) - hit)


# ------------------------------------------------------------------------------------------------------------------
# Gram statistics of the fused block tail
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [64, 256, 2048])
@pytest.mark.parametrize("stride", [1, 2])
def test_colsum_pixels(cuda_device, C, stride):
    g = torch.Generator().manual_seed(C + stride)
    N, H, W = 3, 6, 10                               # 180 / 45 rows: the last block is partial
    x = torch.randn(N, H, W, C, generator=g).to(cuda_device).to(torch.bfloat16) + 3
    out = torch.full((C,), float("nan"), device=cuda_device)
    scratch = torch.empty(4 * 148 * C, device=cuda_device)
    _lib.call("argus_colsum_pixels", x, N, H, W, C, stride, scratch, out, _lib.stream_ptr())
    torch.cuda.synchronize()
    xs = x[:, ::stride, ::stride, :].double().reshape(-1, C)
    want = xs.sum(0)
    assert bool(((out.double() - want).abs() <= 1e-6 * xs.abs().sum(0)).all())


@pytest.mark.parametrize("shape", [(4, 16, 16, 64, 1), (4, 16, 16, 256, 2), (2, 32, 32, 128, 1)])
def test_conv2d_gram(cuda_device, shape):
    N, H, W, C, s = shape
    g = torch.Generator().manual_seed(C)
    x = torch.randn(N, H, W, C, generator=g).to(cuda_device).to(torch.bfloat16)
    G = torch.zeros(C, C, device=cuda_device)
    _lib.call("argus_conv2d_gram", x, G, N, H, W, C, C, s, _lib.stream_ptr())
    torch.cuda.synchronize()
    xs = x[:, ::s, ::s, :].double().reshape(-1, C)
    want, scale = xs.t() @ xs, xs.abs().t() @ xs.abs()
    err = (G.double() - want).abs() / scale
    print(f"gram {shape}: largest |err| / (|x|^T |x|) = {float(err.max()):.3e}")
    assert float(err.max()) < 2.0 ** -16


def _gram_stats(x, Wt, gamma, beta, rm, rv, dev):
    """Gram path: G, colsum, bn_stats_from_gram. Returns dict of fp32 outputs."""
    N, H, W, Cc = x.shape
    O = Wt.shape[0]
    G = torch.zeros(Cc, Cc, device=dev)
    s = torch.empty(Cc, device=dev)
    st = _lib.stream_ptr()
    _lib.call("argus_conv2d_gram", x, G, N, H, W, Cc, O, 1, st)
    _lib.call("argus_colsum_pixels", x, N, H, W, Cc, 1, torch.empty(4 * 148 * Cc, device=dev), s, st)
    out = {k: torch.empty(O, device=dev) for k in ("scale", "shift", "mean", "invstd")}
    out["rm"], out["rv"] = rm.clone(), rv.clone()
    _lib.call("argus_bn_stats_from_gram", Wt, G, s, _lib.c_double(N * H * W), gamma, beta, out["rm"], out["rv"], 0.1,
              1e-5, out["scale"], out["shift"], out["mean"], out["invstd"], torch.empty(O * Cc // 16, device=dev), O,
              Cc, st)
    return out


def _separate_stats(x, Wt, gamma, beta, rm, rv, dev):
    """Yardstick: plain conv with fp32 statistics slots, then bn_finalize."""
    N, H, W, Cc = x.shape
    O = Wt.shape[0]
    info = launch_info("fwd", (N, H, W, Cc, O, 1, 1), STATS)[0]
    y = torch.empty(N, H, W, O, device=dev, dtype=torch.bfloat16)
    partial = torch.zeros(info[9], 2, O, device=dev)
    st = _lib.stream_ptr()
    _lib.call("argus_conv2d_forward", x, Wt.reshape(O, 1, 1, Cc), y, N, H, W, Cc, O, 1, 1, 0, None, None, None, 0,
              partial, info[9], st)
    out = {k: torch.empty(O, device=dev) for k in ("scale", "shift", "mean", "invstd")}
    out["rm"], out["rv"] = rm.clone(), rv.clone()
    _lib.call("argus_bn_finalize", partial, info[9], _lib.c_double(N * H * W), gamma, beta, out["rm"], out["rv"], 0.1,
              1e-5, out["scale"], out["shift"], out["mean"], out["invstd"], O, st)
    del y
    return out


@pytest.fixture(scope="module")
def gram_report(cuda_device):
    """bn3 statistics of the fused block tail at the real layer-1 size (512 images of 64 x 64 = 2 M rows, 64 -> 256
    channels), on post-ReLU inputs with a large common offset and output channels whose mean / std ratio is swept from 1
    to 30 (var = E[y^2] - mean^2 cancels). Truth: float64 batch norm of the unrounded y = x W^T. Yardstick: the
    separate-pass formula (bf16 y, fp32 slot sums, bn_finalize) on the same data."""
    dev = cuda_device
    g = torch.Generator().manual_seed(7)
    N, H, W, Cc, O = 512, 64, 64, 64, 256
    x = (torch.relu(torch.randn(N, H, W, Cc, generator=g)) + 4.0).to(torch.bfloat16).to(dev)
    xs = x.reshape(-1, Cc)
    P = xs.shape[0]
    m_x = xs.double().sum(0) / P
    G64 = xs.double().t() @ xs.double()
    cov = G64 / P - torch.outer(m_x, m_x)
    # W_o = v_o + beta_o u: v_o random with zero sum, u = ones / C; beta_o picked on a grid to hit the target ratio
    targets = torch.tensor([1.0, 3.0, 10.0, 30.0], dtype=torch.float64)
    v = torch.randn(O, Cc, generator=g, dtype=torch.float64) / Cc ** 0.5
    v = (v - v.mean(1, keepdim=True)).to(dev)
    u = torch.full((Cc,), 1.0 / Cc, dtype=torch.float64, device=dev)
    betas = torch.logspace(-3, 2, 4000, dtype=torch.float64, device=dev)
    want_ratio = targets.repeat_interleave(O // 4).to(dev)
    Wc = v.unsqueeze(1) + betas.view(1, -1, 1) * u                   # O x grid x C
    mean = Wc @ m_x
    var = torch.einsum("ogc,cd,ogd->og", Wc, cov, Wc)
    ratio = mean.abs() / var.sqrt()
    pick = (ratio.log() - want_ratio.log().unsqueeze(1)).abs().argmin(1)
    Wt = (v + betas[pick].unsqueeze(1) * u).to(torch.bfloat16).contiguous()
    Wd = Wt.double()
    mean_t = Wd @ m_x
    ey2 = torch.einsum("oc,cd,od->o", Wd, G64 / P, Wd)
    var_t = ey2 - mean_t ** 2
    ratio_t = mean_t.abs() / var_t.sqrt()
    gamma = torch.randn(O, generator=g).to(dev)
    beta = torch.randn(O, generator=g).to(dev)
    rm, rv = torch.randn(O, generator=g).to(dev), torch.rand(O, generator=g).to(dev) + 0.5
    inv_t = 1.0 / torch.sqrt(var_t + 1e-5)
    truth = dict(mean=mean_t, invstd=inv_t, scale=gamma.double() * inv_t, shift=beta.double() - mean_t * gamma.double() * inv_t,
                 rm=0.9 * rm.double() + 0.1 * mean_t, rv=0.9 * rv.double() + 0.1 * var_t * P / (P - 1),
                 beta=beta.double(), rm_old=rm.double())
    gram = _gram_stats(x, Wt, gamma, beta, rm, rv, dev)
    sep = _separate_stats(x, Wt, gamma, beta, rm, rv, dev)
    torch.cuda.synchronize()

    report = []
    for i, r in enumerate(targets.tolist()):
        sel = slice(i * (O // 4), (i + 1) * (O // 4))
        row = {"ratio": r, "measured_ratio": (float(ratio_t[sel].min()), float(ratio_t[sel].max()))}
        for k in ("invstd", "mean", "scale", "shift", "rm", "rv"):
            row[k] = (_stat_err(gram, truth, k, sel), _stat_err(sep, truth, k, sel))
        report.append(row)
        print(f"mean/std {r:>4}: measured {row['measured_ratio'][0]:.2f}..{row['measured_ratio'][1]:.2f}  " +
              "  ".join(f"{k} gram {row[k][0]:.2e} separate {row[k][1]:.2e}" for k in ("invstd", "mean", "scale", "shift", "rm", "rv")))
    return report


def _stat_err(out, truth, k, sel):
    """Largest relative error of statistic k over the channels sel. shift and the running mean are relative to the
    size of the terms they are made of (beta and mean * scale; the old running mean and the new mean), which may cancel."""
    err = (out[k].double() - truth[k]).abs()[sel]
    if k == "shift":
        den = truth["beta"].abs() + (truth["mean"] * truth["scale"]).abs()
    elif k == "rm":
        den = 0.9 * truth["rm_old"].abs() + 0.1 * truth["mean"].abs()
    else:
        den = truth[k].abs()
    return float((err / den[sel].clamp_min(1e-30)).max())


# Gram path, inputs offset by 7 std: relative errors measured on a B200 (1000 W) at mean / std 1, 3, 10, 30 were
# invstd 9.9e-5, 1.9e-4, 1.2e-3, 1.0e-2 and running_var 1.6e-5, 3.4e-5, 2.0e-4, 1.9e-3; the bounds leave a factor 2.
GRAM_BOUNDS = {1.0: (2e-4, 4e-5), 3.0: (4e-4, 7e-5), 10.0: (2.5e-3, 4e-4), 30.0: (2e-2, 4e-3)}


def test_gram_statistics_on_offset_inputs(gram_report):
    for row in gram_report:
        inv_b, rv_b = GRAM_BOUNDS[row["ratio"]]
        assert row["mean"][0] <= max(2 * row["mean"][1], 1e-6), row
        assert row["invstd"][0] <= inv_b and row["scale"][0] <= inv_b and row["shift"][0] <= inv_b, row
        assert row["rv"][0] <= rv_b, row
        assert row["rm"][0] <= 1e-6, row


@pytest.mark.xfail(strict=True, reason="G = x^T x is accumulated in fp32 before the inputs' common offset cancels in "
                   "W G W^T: with inputs offset by 7 std the Gram path's invstd error is 5-18x the separate pass's "
                   "(9.9e-5 vs 5.6e-6 at mean/std 1, B200); real activations stay out of this regime "
                   "(test_gram_statistics_on_real_activations)")
def test_gram_no_worse_than_separate_pass_on_offset_inputs(gram_report):
    for row in gram_report:
        if row["ratio"] <= 10:
            assert row["invstd"][0] <= max(2 * row["invstd"][1], 1e-6), row


from test_parity_gpu import probe, task, zero_init_checkpoint  # noqa: E402,F401  (fixtures)


def test_gram_statistics_on_real_activations(cuda_device, zero_init_checkpoint, task):
    """The inputs the fused block tail takes Gram matrices of -- act2 of every bottleneck of layers 1-3 and the block
    inputs of the first downsample branches -- from a train-mode forward of the zero-init checkpoint (test_parity_gpu.py),
    with the checkpoint's own weights: Gram-path statistics within 1e-4 of float64 batch norm and no worse than twice the
    separate-pass formula. Prints each input's common offset (channel mean / std) and the output mean / std ratios."""
    from argus_b200.models import NCameraCNN

    dev, sd = cuda_device, zero_init_checkpoint
    images = task[0][48:64]
    model = NCameraCNN().to(dev)
    model.load_state_dict(sd)
    model.train()
    with torch.no_grad():
        model(images)
    torch.cuda.synchronize()
    N = images.shape[0] * images.shape[1] // 3
    names = [(L, j) for L, n in ((1, 3), (2, 4), (3, 6)) for j in range(n)]
    inputs = []
    for i, (L, j) in enumerate(names):
        inputs.append((f"layer{L}.{j}.conv3", model.probe_activation(100 + i), f"resnet.layer{L}.{j}.conv3.weight",
                       f"resnet.layer{L}.{j}.bn3", 1))
    inputs.append(("layer1.0.downsample", model.probe_activation(-1), "resnet.layer1.0.downsample.0.weight",
                   "resnet.layer1.0.downsample.1", 1))
    inputs.append(("layer2.0.downsample", model.probe_activation(2), "resnet.layer2.0.downsample.0.weight",
                   "resnet.layer2.0.downsample.1", 2))
    failures = []
    for label, act, wname, bn, stride in inputs:
        rows, Cc = act.shape
        hw = int(round((rows // N) ** 0.5))
        x = act.view(N, hw, hw, Cc)[:, ::stride, ::stride, :].contiguous()
        Wt = sd[wname].reshape(sd[wname].shape[0], Cc).to(dev).to(torch.bfloat16).contiguous()
        gamma, beta = sd[bn + ".weight"].to(dev).float(), sd[bn + ".bias"].to(dev).float()
        rm, rv = sd[bn + ".running_mean"].to(dev).float(), sd[bn + ".running_var"].to(dev).float()
        xs = x.reshape(-1, Cc).double()
        P = xs.shape[0]
        m_x = xs.mean(0)
        G64 = xs.t() @ xs
        Wd = Wt.double()
        mean_t = Wd @ m_x
        var_t = (torch.einsum("oc,cd,od->o", Wd, G64 / P, Wd) - mean_t ** 2).clamp_min(0)
        inv_t = 1.0 / torch.sqrt(var_t + 1e-5)
        gram = _gram_stats(x, Wt, gamma, beta, rm, rv, dev)
        sep = _separate_stats(x, Wt, gamma, beta, rm, rv, dev)
        torch.cuda.synchronize()
        e_g = float(((gram["invstd"].double() - inv_t).abs() / inv_t).max())
        e_s = float(((sep["invstd"].double() - inv_t).abs() / inv_t).max())
        em_g = float(((gram["mean"].double() - mean_t).abs() / (Wd.abs() @ m_x.abs()).clamp_min(1e-30)).max())
        offset = float((m_x / xs.std(0).clamp_min(1e-30)).max())
        ratio = float((mean_t.abs() / var_t.sqrt().clamp_min(1e-30)).max())
        print(f"{label}: rows {P} input offset/std <= {offset:.2f}  output mean/std <= {ratio:.2f}  "
              f"invstd rel err gram {e_g:.2e} separate {e_s:.2e}  mean err gram {em_g:.2e}")
        if not (e_g <= 1e-4 and e_g <= max(2 * e_s, 1e-6) and em_g <= 1e-6):
            failures.append((label, e_g, e_s, em_g))
    assert not failures, failures


# ------------------------------------------------------------------------------------------------------------------
# Coverage: every instance the model launches is one a case above pins
# ------------------------------------------------------------------------------------------------------------------
def test_model_launches_only_pinned_instances(cuda_device, monkeypatch):
    from argus_b200.engine import TrainEngine
    from argus_b200.models import NCameraCNN
    from gpu_util import random_targets, structured_images

    table = {key_of(i) for c in CASES for i in case_info(c)}
    seen = {}

    def run(label, B, H, train):
        model = NCameraCNN().to(cuda_device)
        x = structured_images(B, 6, H, H, 1, cuda_device)
        _lib.call("argus_conv_instances_record", 1)
        try:
            if train:
                model.train()
                TrainEngine(model, lr=1e-4, max_grad_norm=1.0, distributed=False).forward_backward(
                    x, random_targets(B, 2, cuda_device))
            else:
                model.eval()
                with torch.no_grad():
                    model(x)
            torch.cuda.synchronize()
        finally:
            _lib.call("argus_conv_instances_record", 0)
        seen[label] = recorded_keys()
        del model, x
        torch.cuda.empty_cache()

    run("train B=256 256x256", 256, 256, True)
    run("train B=8 128x128", 8, 128, True)
    run("eval B=1", 1, 256, False)
    run("eval B=64", 64, 256, False)
    monkeypatch.setenv("ARGUS_BN_REDUCE_FUSED", "2")    # read when the next model binds
    run("train B=256 256x256, fused BN reduction", 256, 256, True)
    monkeypatch.delenv("ARGUS_BN_REDUCE_FUSED")
    missing = {k: sorted(v - table) for k, v in seen.items() if v - table}
    assert not missing, f"instances the model launches that no case pins (block_n, b_mn, opt, halo, b_resident): {missing}"
