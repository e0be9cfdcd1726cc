"""The algebraic batch-norm backward (csrc/bn_algebra.cu) against the float64 reference of tests/bnalg_ref.py, kernel
by kernel and end to end, through the geometries and data edges where it can go wrong.

Every case runs the primitive chain in the model's order: [H; G] = [g | act]^T act (argus_conv2d_wgrad_gram into a zero
buffer), s = colsum(act), argus_bn_alg_backward_small, then the K-concatenated dgrad (argus_conv2d_dgrad_ex with the
B-stack and the bias). Each stage is checked from the GPU's own inputs to it, then the whole chain against the float64
algebra. k1k0, the B-stack, the bias and the o-split partials are filled with NaN before each call; every output sits
between 4 KB sentinels. dgamma, dbeta and dW are added to: a run from a random start D must give fl32(D + run from 0)
bit for bit; the dW kernel run inline and on its own (the model's side stream) must agree bit for bit, and so must
repeats. Where a case has one statistics slot, argus_conv_bn_backward_algebraic must equal the chain bit for bit.
"""
import ctypes
import time
import zlib

import pytest
import torch

import bnalg_ref as br
from argus_b200 import _lib

pytestmark = pytest.mark.gpu


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def C(name, O, Cc, N, Hh, stride=1, slots=1, data=(), chunks=None):
    """chunks: 32-row chunks per o-split of bn_alg_matrix_kernel (O / 8 / 32); slots: 1, a count, or "dgrad" (the slots
    of an argus_conv2d_dgrad_ex statistics launch that produced g)."""
    return dict(name=name, O=O, C=Cc, N=N, H=Hh, stride=stride, slots=slots, data=set(data),
                chunks=chunks if chunks is not None else O // 256)


CASES = [
    # O: one 32-row chunk per o-split up to the prefetch loop over 8 chunks
    C("o256_c64", 256, 64, 2, 8, chunks=1),
    C("o512_c64", 512, 64, 2, 8, chunks=2),
    C("o1024_c64", 1024, 64, 2, 8, chunks=4),
    C("o2048_c64", 2048, 64, 2, 8, chunks=8),
    # C: the bias row is grid row y = C / 16 (3 for C = 32)
    C("o256_c32", 256, 32, 2, 8),
    C("o256_c128", 256, 128, 2, 8),
    C("o256_c256", 256, 256, 2, 8),
    # the model's shapes at batch 8 (N = 16 images of 256 x 256) and layer 1 at batch 256
    C("layer1_b8", 256, 64, 16, 64),
    C("layer2_b8", 512, 128, 16, 32),
    C("layer2_ds_b8", 512, 256, 16, 64, stride=2),
    C("layer3_b8", 1024, 256, 16, 16),
    C("layer1_b256", 256, 64, 512, 64),
    # pixel counts that are not a multiple of 128 (spatial sizes are powers of two), and a single pixel (var = 0,
    # invstd = eps^-1/2)
    C("ragged_320", 256, 64, 5, 8),
    C("ragged_48_s2", 512, 256, 3, 8, stride=2),
    C("single_pixel", 256, 64, 1, 1),
    # statistics slots: the lanes' round-robin, and the slots the model's dgrad writes
    C("slots33", 512, 128, 2, 8, slots=33),
    C("slots1000", 256, 64, 2, 8, slots=1000),
    C("slots1000_s2", 512, 256, 2, 16, stride=2, slots=1000),
    C("dgrad_slots", 256, 64, 4, 16, slots="dgrad"),
    C("dgrad_slots_c256", 1024, 256, 4, 8, slots="dgrad"),
    # data edges
    C("zero_g_column", 256, 64, 2, 16, data=("zero_g_column",)),
    C("zero_w_row", 256, 64, 2, 16, data=("zero_w_row",)),
    C("negative_gamma", 512, 128, 2, 16, data=("negative_gamma",)),
    C("offset4", 512, 128, 2, 16, data=("offset4",)),
    C("offset16", 512, 128, 2, 16, data=("offset16",)),
    C("offset16_s2", 512, 256, 2, 16, stride=2, data=("offset16",)),
]
BY_NAME = {c["name"]: c for c in CASES}


# ------------------------------------------------------------------------------------------------------------------
# guarded buffers
# ------------------------------------------------------------------------------------------------------------------
class Guarded:
    """[4 KB sentinel | n elements = init | 4 KB sentinel] of fp32 or bf16."""

    def __init__(self, n, dtype, init, dev):
        self.n, self.dtype = n, dtype
        if dtype == torch.float32:
            self.g = br.SENTINEL
            self.buf = torch.full((2 * self.g + n,), br.SENTINEL_F32, device=dev)
        else:
            self.g = 2 * br.SENTINEL
            self.buf = torch.full((2 * self.g + n,), br.SENTINEL_BF16, dtype=torch.int16, device=dev).view(torch.bfloat16)
        self.v = self.buf[self.g:self.g + n]
        if init is not None:
            if isinstance(init, torch.Tensor):
                self.v.copy_(init.reshape(-1))
            else:
                self.v.fill_(init)

    def check(self, what):
        word = torch.int32 if self.dtype == torch.float32 else torch.int16
        want = torch.tensor(br.SENTINEL_F32).view(torch.int32) if word == torch.int32 else \
            torch.tensor(br.SENTINEL_BF16, dtype=torch.int16)
        b = self.buf.view(word)
        pre = torch.nonzero(b[:self.g] != want.to(b.device)).flatten()
        post = torch.nonzero(b[self.g + self.n:] != want.to(b.device)).flatten()
        assert pre.numel() == 0, f"{what}: {pre.numel()} elements before the buffer written (first at -{self.g - int(pre[0])})"
        assert post.numel() == 0, f"{what}: {post.numel()} elements past the buffer written (first at +{int(post[0])})"


def bits_equal(a, b):
    w = torch.int32 if a.dtype == torch.float32 else torch.int16
    return torch.equal(a.contiguous().view(w), b.contiguous().view(w))


# ------------------------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------------------------
def stat_slots_of(N, Hh, Cn, O):
    n = ctypes.c_int()
    _lib.check(_lib.load().argus_conv2d_stat_slots(N, Hh, Hh, Cn, O, 1, 1, 0, ctypes.byref(n)))
    return n.value


def make_inputs(case, dev):
    O, Cc, N, Hh, s = case["O"], case["C"], case["N"], case["H"], case["stride"]
    gen = torch.Generator(device=dev).manual_seed(zlib.crc32(case["name"].encode()))
    Ho = Hh // s
    rows = N * Ho * Ho
    data = case["data"]
    off = 4.0 if "offset4" in data else 16.0 if "offset16" in data else None
    if off is None:
        act = (torch.randn(N, Hh, Hh, Cc, generator=gen, device=dev) * 1.3).relu().bfloat16()
    else:
        act = (torch.randn(N, Hh, Hh, Cc, generator=gen, device=dev) + off).bfloat16()
    W = torch.randn(O, Cc, generator=gen, device=dev) / Cc ** 0.5
    if "zero_w_row" in data:
        W[7] = 0
    W = W.bfloat16()
    gamma = torch.rand(O, generator=gen, device=dev) + 0.5
    if "negative_gamma" in data:
        gamma[::3] *= -1
    slots, stride_stat = case["slots"], O
    if slots == "dgrad":
        # g as the model produces it: the dgrad of the next convolution (Cn -> O channels), masked by ReLU bits, with
        # per-CTA statistics slots [slots][2][O]
        Cn = 64
        dy = torch.randn(rows, Cn, generator=gen, device=dev).bfloat16()
        wn = (torch.randn(Cn, O, generator=gen, device=dev) / Cn ** 0.5).bfloat16()
        keep = torch.rand(rows, O, generator=gen, device=dev) > 0.45
        bits = (keep.view(rows, O // 8, 8).to(torch.int32) << torch.arange(8, device=dev, dtype=torch.int32)).sum(-1)
        bits = bits.to(torch.uint8).contiguous()
        slots = stat_slots_of(N, Ho, Cn, O)
        stat = torch.zeros(slots, 2, O, device=dev)
        g = torch.empty(N, Ho, Ho, O, device=dev, dtype=torch.bfloat16)
        _lib.call("argus_conv2d_dgrad_ex", dy, wn, g, N, Ho, Ho, O, Cn, 1, None, 0, None, None, bits, stat, slots,
                  _lib.stream_ptr())
        torch.cuda.synchronize()
        used = int((stat[:, 0].abs().sum(1) > 0).sum())
        assert used > 1, f"{case['name']}: the dgrad wrote {used} statistics slots"
        stride_stat = 2 * O
    else:
        g = (torch.randn(N, Ho, Ho, O, generator=gen, device=dev) *
             (torch.rand(N, Ho, Ho, O, generator=gen, device=dev) > 0.5)).bfloat16()
        if "zero_g_column" in data:
            g[..., 11] = 0
        gs = g.reshape(rows, O).double()
        if slots == 1:
            stat = gs.sum(0).float()
        else:
            stride_stat = 2 * O
            cut = torch.randint(0, slots, (rows,), generator=gen, device=dev)
            part = torch.zeros(slots, O, dtype=torch.float64, device=dev).index_add_(0, cut, gs)
            stat = torch.full((slots, 2, O), float("nan"), device=dev)   # the second row must not be read
            stat[:, 0] = part.float()
    a = br.sample(act, s).double()
    raw = a @ W.double().t()
    mean = raw.mean(0)
    var = (raw - mean).pow(2).mean(0)
    invstd = (1.0 / torch.sqrt(var + br.EPS)).float()
    scale = gamma * invstd
    return dict(act=act, W=W, g=g, gamma=gamma, mean=mean.float(), invstd=invstd, scale=scale, stat=stat.contiguous(),
                slots=slots, stat_stride=stride_stat, rows=rows, O=O, C=Cc, N=N, H=Hh, stride=s)


# ------------------------------------------------------------------------------------------------------------------
# launches
# ------------------------------------------------------------------------------------------------------------------
def mpartial_elems(Cc):
    n = ctypes.c_int64()
    _lib.check(_lib.load().argus_bn_alg_matrix_scratch_elems(Cc, ctypes.byref(n)))
    return n.value


def h_gram_colsum(p, dev):
    O, Cc = p["O"], p["C"]
    if Cc % 64:
        # the GEMMs take multiples of 64 channels; the small kernels take C = 32: H, G, s in fp32 from float64
        gs, a = p["g"].reshape(-1, O).double(), br.sample(p["act"], p["stride"]).double()
        return (gs.t() @ a).float(), (a.t() @ a).float(), a.sum(0).float()
    HG = torch.zeros(O + Cc, Cc, device=dev)
    st = _lib.stream_ptr()
    _lib.call("argus_conv2d_wgrad_gram", p["g"], p["act"], HG, p["N"], p["H"], p["H"], Cc, O, p["stride"], st)
    s = torch.empty(Cc, device=dev)
    scratch = torch.empty(4 * sms() * Cc, device=dev)
    _lib.call("argus_colsum_pixels", p["act"], p["N"], p["H"], p["H"], Cc, p["stride"], scratch, s, st)
    return HG[:O].contiguous(), HG[O:].contiguous(), s


def small(p, H, G, s, dev, dw_mode="inline", start=None):
    """argus_bn_alg_backward_small (+ argus_bn_alg_backward_dw for dw_mode "aside") into guarded outputs.
    start: (dgamma, dbeta, dW) start values (zeros by default)."""
    O, Cc = p["O"], p["C"]
    z = start or (torch.zeros(O, device=dev), torch.zeros(O, device=dev), torch.zeros(O, Cc, device=dev))
    out = dict(dgamma=Guarded(O, torch.float32, z[0], dev), dbeta=Guarded(O, torch.float32, z[1], dev),
               dW=Guarded(O * Cc, torch.float32, z[2], dev), k1k0=Guarded(2 * O, torch.float32, float("nan"), dev),
               bstack=Guarded((O + Cc) * Cc, torch.bfloat16, float("nan"), dev),
               bias=Guarded(Cc, torch.float32, float("nan"), dev))
    mpart = torch.full((mpartial_elems(Cc),), float("nan"), device=dev)
    st = _lib.stream_ptr()
    _lib.call("argus_bn_alg_backward_small", p["W"], H, G, s, p["stat"], p["slots"], p["stat_stride"], p["scale"],
              p["mean"], p["invstd"], _lib.c_double(p["rows"]), out["dgamma"].v, out["dbeta"].v,
              out["dW"].v if dw_mode == "inline" else None, out["k1k0"].v, out["bstack"].v, out["bias"].v, mpart, O, Cc, st)
    if dw_mode == "aside":
        _lib.call("argus_bn_alg_backward_dw", p["W"], H, G, s, p["scale"], out["k1k0"].v, out["dW"].v, O, Cc, st)
    torch.cuda.synchronize()
    for k, b in out.items():
        b.check(f"{k} ({dw_mode})")
    return dict(dgamma=out["dgamma"].v.clone(), dbeta=out["dbeta"].v.clone(), dW=out["dW"].v.view(O, Cc).clone(),
                k1k0=out["k1k0"].v.clone(), bstack=out["bstack"].v.view(O + Cc, Cc).clone(), bias=out["bias"].v.clone())


def concat_dgrad(p, bstack, bias, dev):
    n = p["N"] * p["H"] * p["H"] * p["C"]
    out = Guarded(n, torch.bfloat16, None, dev)
    _lib.call("argus_conv2d_dgrad_ex", p["g"], bstack, out.v, p["N"], p["H"], p["H"], p["C"], p["O"], p["stride"],
              p["act"], p["C"], bias, None, None, None, 0, _lib.stream_ptr())
    torch.cuda.synchronize()
    out.check("dAct")
    return out.v.view(p["N"], p["H"], p["H"], p["C"]).clone()


# ------------------------------------------------------------------------------------------------------------------
# the case table
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(BY_NAME))
def test_bnalg_case(cuda_device, name):
    dev = cuda_device
    case = BY_NAME[name]
    t0 = time.perf_counter()
    p = make_inputs(case, dev)
    O, Cc = p["O"], p["C"]
    # the geometry the case claims
    assert O % 256 == 0 and Cc % 32 == 0
    assert O // 8 // 32 == case["chunks"], f"{name}: {O // 256} chunks per o-split"
    assert (p["slots"] > 1) == (case["slots"] != 1)
    if name == "o256_c32":
        assert Cc // 16 + 1 == 3
    what = f"{name} (O {O}, C {Cc}, stride {p['stride']}, rows {p['rows']}, slots {p['slots']})"
    H, G, s = h_gram_colsum(p, dev)
    A = small(p, H, G, s, dev)
    worst = {}
    worst.update(br.check_coeffs(p["W"], H, p["stat"], p["slots"], p["stat_stride"], p["scale"], p["mean"], p["invstd"],
                                 p["rows"], A["dgamma"], A["dbeta"], A["k1k0"], what))
    br.check_bstack_rows(p["W"], p["scale"], A["bstack"], what)
    worst.update(br.check_matrix(p["W"], A["k1k0"], A["bstack"], A["bias"], what))
    worst["dW"] = br.check_dw(p["W"], H, G, s, p["scale"], A["k1k0"], A["dW"], what)
    if "zero_g_column" in case["data"]:
        for k in ("dgamma", "dbeta"):
            assert float(A[k][11]) == 0.0, f"{what}: {k} of the all-zero g column"
        assert float(A["k1k0"][11]) == 0.0 and float(A["k1k0"][O + 11]) == 0.0
    # repeats, the side-stream dW, and the start values that are added to
    for mode in ("inline", "aside"):
        R = small(p, H, G, s, dev, mode)
        for k in A:
            assert bits_equal(R[k], A[k]), f"{what}: {k} differs between runs ({mode} dW)"
    gen = torch.Generator(device=dev).manual_seed(1)
    D = (torch.randn(O, generator=gen, device=dev), torch.randn(O, generator=gen, device=dev),
         torch.randn(O, Cc, generator=gen, device=dev))
    for mode in ("inline", "aside"):
        R = small(p, H, G, s, dev, mode, start=D)
        for k, d in zip(("dgamma", "dbeta", "dW"), D):
            br.check_accumulated(R[k], d, A[k], f"{what} {k} from D ({mode})")
    if Cc % 64:
        print(f"{what}: err/bound " + " ".join(f"{k} {v:.3f}" for k, v in worst.items()) + " (no GEMMs at C = 32)")
        assert all(v <= 1 for v in worst.values()), worst
        return
    # the concat dgrad
    dact = concat_dgrad(p, A["bstack"], A["bias"], dev)
    worst["dact stage"] = br.check_dact(p["g"], p["act"], A["bstack"], A["bias"], dact, p["stride"], what)
    assert bits_equal(concat_dgrad(p, A["bstack"], A["bias"], dev), dact), f"{what}: dAct differs between runs"
    # end to end
    got = dict(dgamma=A["dgamma"], dbeta=A["dbeta"], dW=A["dW"], dact=dact)
    e2e = br.check_end_to_end(p["g"], p["act"], p["W"], p["scale"], p["mean"], p["invstd"], p["stat"], p["slots"],
                              p["stat_stride"], p["stride"], got, sms(), what)
    worst.update({f"e2e {k}": v for k, v in e2e.items()})
    # the composite entry point is the same chain
    if p["slots"] == 1:
        dg, db, dw = torch.zeros(O, device=dev), torch.zeros(O, device=dev), torch.zeros(O, Cc, device=dev)
        dact2 = torch.full_like(dact, float("nan"))
        _lib.call("argus_conv_bn_backward_algebraic", p["g"], p["act"], p["W"], p["stat"], p["scale"], p["mean"],
                  p["invstd"], dg, db, dw, dact2, p["N"], p["H"], p["H"], Cc, O, p["stride"], _lib.stream_ptr())
        torch.cuda.synchronize()
        for k, v in (("dgamma", dg), ("dbeta", db), ("dW", dw)):
            assert bits_equal(v, A[k]), f"{what}: argus_conv_bn_backward_algebraic {k} differs from the chain"
        sd = br.sample(dact, p["stride"])
        assert bits_equal(br.sample(dact2, p["stride"]), sd), f"{what}: composite dAct differs from the chain"
        if p["stride"] == 2:
            br._dact_check(what + " composite", dact2, sd.double(), torch.zeros_like(sd, dtype=torch.float64),
                           2, A["bias"], sentinel=False)
    print(f"{what}: err/bound " + " ".join(f"{k} {v:.3f}" for k, v in worst.items())
          + f" ({time.perf_counter() - t0:.2f} s)")
    assert all(v <= 1 for v in worst.values()), worst
    del p, H, G, s, A, dact
    torch.cuda.empty_cache()


def test_bad_arguments_are_errors(cuda_device):
    dev = cuda_device
    f = torch.zeros(4096, device=dev)
    b = torch.zeros(4096, device=dev, dtype=torch.bfloat16)
    st = _lib.stream_ptr()
    args = lambda O, Cc, W=b, k1k0=f: (W, f, f, f, f, 1, O, f, f, f, _lib.c_double(8.0), f, f, f, k1k0, b, f, f, O, Cc, st)
    for bad, msg in ((args(128, 32), "O % 256"), (args(256, 48), "C % 32"), (args(256, 32, W=None), "null"),
                     (args(256, 32, k1k0=None), "null")):
        with pytest.raises(_lib.ArgusError, match=msg):
            _lib.call("argus_bn_alg_backward_small", *bad)
    with pytest.raises(_lib.ArgusError, match="O % 256"):
        _lib.call("argus_bn_alg_backward_dw", b, f, f, f, f, f, f, 16, 32, st)
    with pytest.raises(_lib.ArgusError, match="null"):
        _lib.call("argus_bn_alg_backward_dw", b, f, f, None, f, f, f, 256, 32, st)


# ------------------------------------------------------------------------------------------------------------------
# coverage: every call the model makes is one a case pins
# ------------------------------------------------------------------------------------------------------------------
def recorded_calls():
    n = ctypes.c_int()
    _lib.call("argus_bn_alg_calls_get", None, 0, ctypes.byref(n))
    buf = (ctypes.c_int * (5 * n.value))()
    _lib.call("argus_bn_alg_calls_get", buf, 5 * n.value, ctypes.byref(n))
    return {tuple(buf[5 * i:5 * i + 5]) for i in range(n.value)}


def test_model_calls_are_pinned(cuda_device, monkeypatch):
    """Training steps at batch 256 and 8, with the default and the all-layers fused BN reduction, with dW on the side
    stream and inline: every (O, C, stride) the model passes to the algebraic backward has a case, every case runs
    both dW placements, and the model's multi-slot statistics have cases."""
    from argus_b200.engine import TrainEngine
    from argus_b200.models import NCameraCNN
    from gpu_util import random_targets, structured_images

    seen = set()
    for B, Hh, fused, overlap in ((256, 256, False, True), (8, 128, False, False), (256, 256, True, True),
                                  (8, 128, True, False)):
        if fused:
            monkeypatch.setenv("ARGUS_BN_REDUCE_FUSED", "2")    # read when the model binds
        model = NCameraCNN().to(cuda_device)
        model.train()
        if not overlap:
            _lib.call("argus_model_set_wgrad_overlap", model._handle.ptr, 0)
        x = structured_images(B, 6, Hh, Hh, 1, cuda_device)
        _lib.call("argus_conv_instances_record", 1)
        try:
            TrainEngine(model, lr=1e-4, max_grad_norm=1.0, distributed=False).forward_backward(
                x, random_targets(B, 2, cuda_device))
            torch.cuda.synchronize()
        finally:
            _lib.call("argus_conv_instances_record", 0)
        keys = recorded_calls()
        print(f"B={B} fused={fused} overlap={overlap}: (O, C, stride, dW aside, slots > 1) {sorted(keys)}")
        assert keys and {k[3] for k in keys} == {int(overlap)}, keys
        seen |= keys
        del model, x
        torch.cuda.empty_cache()
        monkeypatch.delenv("ARGUS_BN_REDUCE_FUSED", raising=False)
    table = {(c["O"], c["C"], c["stride"]) for c in CASES}
    multi = {(c["O"], c["C"], c["stride"]) for c in CASES if c["slots"] != 1}
    assert {k[:3] for k in seen} == {(256, 64, 1), (512, 128, 1), (512, 256, 2), (1024, 256, 1)}, sorted(seen)
    assert {k[:3] for k in seen} <= table, sorted({k[:3] for k in seen} - table)
    assert {k[3] for k in seen} == {0, 1}
    assert any(k[4] for k in seen) and multi


# ------------------------------------------------------------------------------------------------------------------
# real activations: the algebraic path against the textbook GPU path
# ------------------------------------------------------------------------------------------------------------------
from test_parity_gpu import probe, task, zero_init_checkpoint  # noqa: E402,F401  (fixtures)


@pytest.fixture(scope="module")
def real_inputs(cuda_device, zero_init_checkpoint, task):
    """act2 of every fused-tail bottleneck of layers 1-3 and the inputs of the two algebraic downsample branches, from
    a train-mode forward of the zero-init checkpoint (test_parity_gpu.py), with the checkpoint's weights and gains."""
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
    out = []
    for i, (L, j) in enumerate(names):
        out.append((f"layer{L}.{j}.conv3", model.probe_activation(100 + i), f"resnet.layer{L}.{j}.conv3.weight",
                    f"resnet.layer{L}.{j}.bn3.weight", 1))
    out.append(("layer1.0.downsample", model.probe_activation(-1), "resnet.layer1.0.downsample.0.weight",
                "resnet.layer1.0.downsample.1.weight", 1))
    out.append(("layer2.0.downsample", model.probe_activation(2), "resnet.layer2.0.downsample.0.weight",
                "resnet.layer2.0.downsample.1.weight", 2))
    res = []
    for label, act, wname, gname, stride in out:
        rows, Cc = act.shape
        hw = int(round((rows // N) ** 0.5))
        W = sd[wname].reshape(sd[wname].shape[0], Cc).to(dev).bfloat16().contiguous()
        res.append((label, act.view(N, hw, hw, Cc).contiguous().clone(), W, sd[gname].to(dev).float(), stride))
    del model
    torch.cuda.empty_cache()
    return res


def test_algebraic_no_worse_than_textbook_on_real_activations(cuda_device, real_inputs):
    """Random masked g on each real input. Truth: float64 backward of BatchNorm2d(train) o conv1x1 on the unrounded
    raw = act W^T. The algebraic path (argus_conv_bn_backward_algebraic) must be no farther from it, in norm-relative
    error of dgamma, dW and dAct, than the textbook GPU path on the same inputs: the bf16 raw the forward would store,
    argus_bn_backward, then the dgrad and the weight gradient of dRaw. dgamma and dW of the algebraic path carry no bf16
    rounding (measured on a B200: 1e-7 ... 1e-6 against the textbook's 2e-3 ... 3e-3). dAct of both paths carries the
    same two bf16 roundings (of the B-stack or of dRaw, then of the stored output) and both measure 2.33e-3 ... 2.36e-3:
    the two are equal up to the noise of those roundings, which the 2 % allowance covers; test_bnalg_case pins dAct
    element by element."""
    dev = cuda_device
    st = _lib.stream_ptr()
    failures = []
    for label, act, W, gamma, stride in real_inputs:
        N, Hh, _, Cc = act.shape
        O = W.shape[0]
        gen = torch.Generator(device=dev).manual_seed(zlib.crc32(label.encode()))
        Ho = Hh // stride
        rows = N * Ho * Ho
        g = (torch.randn(N, Ho, Ho, O, generator=gen, device=dev) * 0.01 *
             (torch.rand(N, Ho, Ho, O, generator=gen, device=dev) > 0.5)).bfloat16()
        a = br.sample(act, stride).double()
        raw = a @ W.double().t()
        mean = raw.mean(0)
        invstd = (1.0 / torch.sqrt((raw - mean).pow(2).mean(0) + br.EPS)).float()
        scale = gamma * invstd
        mean = mean.float()
        truth = br.algebra(g, act, W, scale, mean, invstd, stride, mirror=False)
        # algebraic
        dg, db, dw = torch.zeros(O, device=dev), torch.zeros(O, device=dev), torch.zeros(O, Cc, device=dev)
        dact = torch.empty_like(act)
        colsum = g.reshape(rows, O).double().sum(0).float()
        _lib.call("argus_conv_bn_backward_algebraic", g, act, W, colsum, scale, mean, invstd, dg, db, dw, dact,
                  N, Hh, Hh, Cc, O, stride, st)
        # textbook
        raw16 = raw.bfloat16().contiguous()
        shift = torch.zeros(O, device=dev)
        tg, tb = torch.zeros(O, device=dev), torch.zeros(O, device=dev)
        draw = torch.empty_like(raw16)
        _lib.call("argus_bn_backward", g.reshape(rows, O).clone(), raw16, None, scale, shift, mean, invstd, tg, tb, draw,
                  _lib.c_int64(rows), O, 0, st)
        tdact = torch.zeros_like(act)
        _lib.call("argus_conv2d_dgrad", draw, W, tdact, N, Hh, Hh, Cc, O, 1, stride, None, st)
        tdw = torch.zeros(O, Cc, device=dev)
        _lib.call("argus_conv2d_wgrad", draw, act, tdw, N, Hh, Hh, Cc, O, 1, stride, 0, st)
        torch.cuda.synchronize()

        def rel(x, y):
            return float((x.double() - y).norm() / y.norm().clamp_min(1e-300))

        errs = {k: (rel(u, truth[t]), rel(v, truth[t])) for k, u, v, t in
                (("dgamma", dg, tg, "dgamma"), ("dW", dw, tdw, "dW"), ("dAct", dact, tdact, "dact"))}
        print(f"{label}: rows {rows} relative error algebraic / textbook " +
              "  ".join(f"{k} {e[0]:.3e} / {e[1]:.3e}" for k, e in errs.items()) +
              f"  (dAct ratio {errs['dAct'][0] / errs['dAct'][1]:.4f})")
        for k, (e_alg, e_txt) in errs.items():
            if not e_alg <= max(e_txt * (1.02 if k == "dAct" else 1.0), 1e-6):
                failures.append((label, k, e_alg, e_txt))
    assert not failures, failures
