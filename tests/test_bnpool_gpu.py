"""Batch-norm and pooling passes (csrc/elementwise.cu) against the float64 references of tests/bnpool_ref.py, element by
element, through every ring geometry. Every output is first filled with a sentinel (NaN for bf16, a pattern byte for
bit masks and arg-max bytes), so an element the kernel never writes fails.

The ring passes launch grid = min(nvec / 512, 2 x SMs) CTAs of 512-vector stages (nvec = rows x C / 8); the geometries
below are derived from the SM count of the device and the deepest ring (10 stages: apply without residual), so that
they mean the same on any part: a launch that is all tail, whole stages only, a short and a long ragged tail, fewer
stages than CTAs, and every CTA lapping its ring at least three times. The largest error / bound of every check is
collected and printed at the end of the module (pytest -s), or written as JSON to $ARGUS_BNPOOL_REPORT."""
import ctypes
import json
import os

import pytest
import torch

import bnpool_ref as R
from argus_b200 import _lib

pytestmark = pytest.mark.gpu
MAX_STAGES = 10
RATIOS = {}
GEOMETRY = []


def note(name, ratio):
    RATIOS[name] = max(RATIOS.get(name, 0.0), ratio)


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    text = json.dumps({"ratios": RATIOS, "geometry": GEOMETRY}, indent=1)
    print("\nlargest error / bound per check:\n" + text)
    path = os.environ.get("ARGUS_BNPOOL_REPORT")
    if path:
        with open(path, "w") as f:
            f.write(text)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def ring_rows(C, kind):
    """Rows of a (rows, C) tensor whose ring launch has the named geometry (None: unreachable at this C)."""
    cvec = C // 8
    v = R.RING_VEC
    short_tail = cvec if cvec < 256 else None                       # a tail in [1, 255] vectors
    long_tail = (511 // cvec) * cvec if (511 // cvec) * cvec > 256 else None   # a tail in [257, 511]
    nvec = {
        "tail_only": 511 // cvec * cvec,
        "whole_stages": 3 * v,
        "short_tail": None if short_tail is None else 2 * v + short_tail,
        "long_tail": None if long_tail is None else 2 * v + long_tail,
        "fewer_stages_than_ctas": (sms() + 3) * v + cvec,
        "three_laps": 3 * MAX_STAGES * 2 * sms() * v + 7 * v + cvec,
    }[kind]
    return None if nvec is None else nvec // cvec


KINDS = ["tail_only", "whole_stages", "short_tail", "long_tail", "fewer_stages_than_ctas", "three_laps"]
CHANNELS = [64, 128, 256, 512, 1024, 2048]
RING_CASES = [(C, k) for C in CHANNELS for k in KINDS if not (C == 2048 and k in ("short_tail", "long_tail"))]
# C = 2048 is 256 vectors per row: its tails can only be 0 or 256 vectors (both covered by the other kinds)


def record_geometry(rows, C, what):
    g = R.ring_geometry(rows, C, sms())
    g.update(rows=rows, C=C, what=what)
    GEOMETRY.append(g)
    return g


def nan_like(t):
    return torch.full_like(t, float("nan"))


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def rand(shape, g, dev, scale=1.0, offset=0.0):
    return (torch.randn(shape, generator=g, device=dev) * scale + offset)


# ---------------------------------------------------------------------------------------------------- apply
def run_apply(lib, x, sc, sh, res, rs, rb, relu, bits, colsum=False):
    rows, C = x.shape
    y = nan_like(x)
    b = torch.full((rows, C // 8), 0xA5, dtype=torch.uint8, device=x.device) if bits else None
    if colsum:
        n = ctypes.c_int()
        _lib.check(lib.argus_bn_apply_colsum(_lib.ptr(x), _lib.ptr(sc), _lib.ptr(sh), ctypes.c_int(relu), _lib.ptr(y),
                                             _lib.ptr(b), None, ctypes.c_int64(rows), ctypes.c_int(C), ctypes.byref(n),
                                             _lib.stream_ptr()))
        part = torch.full((n.value, C), float("nan"), device=x.device)
        _lib.check(lib.argus_bn_apply_colsum(_lib.ptr(x), _lib.ptr(sc), _lib.ptr(sh), ctypes.c_int(relu), _lib.ptr(y),
                                             _lib.ptr(b), _lib.ptr(part), ctypes.c_int64(rows), ctypes.c_int(C),
                                             ctypes.byref(n), _lib.stream_ptr()))
        return y, b, part
    fn = lib.argus_bn_apply_bits if bits else lib.argus_bn_apply
    args = [_lib.ptr(x), _lib.ptr(sc), _lib.ptr(sh), _lib.ptr(res), _lib.ptr(rs), _lib.ptr(rb), ctypes.c_int(relu),
            _lib.ptr(y)] + ([_lib.ptr(b)] if bits else []) + [ctypes.c_int64(rows), ctypes.c_int(C), _lib.stream_ptr()]
    _lib.check(fn(*args))
    return y, b, None


def check_apply_variants(lib, rows, C, seed, variants):
    dev = torch.device("cuda", 0)
    g = gen(seed)
    x = rand((rows, C), g, dev, 1.5, 0.3).bfloat16()
    res = rand((rows, C), g, dev).bfloat16()
    sc, sh = rand(C, g, dev), rand(C, g, dev, 0.5)          # mixed signs
    rs, rb = rand(C, g, dev), rand(C, g, dev, 0.5)
    for mode, relu, bits, colsum in variants:
        r = res if mode else None
        a, b_ = (rs, rb) if mode == 2 else (None, None)
        y, bm, part = run_apply(lib, x, sc, sh, r, a, b_, relu, bits, colsum)
        pre, ref, E = R.apply_ref(x, sc, sh, r, a, b_, bool(relu))
        tag = f"apply res{mode} relu{relu}{' bits' if bits else ''}{' colsum' if colsum else ''} C{C} rows{rows}"
        note("apply y", R.check_apply(y, pre, ref, E, tag))
        if bits:
            R.check_bits(bm, y, pre, E, tag + " bits")
        if colsum:
            note("apply column sums", R.check_colsum(part, y, what=tag))
            y2, _, part2 = run_apply(lib, x, sc, sh, None, None, None, relu, bits, True)
            assert torch.equal(part, part2) and torch.equal(y, y2), tag + ": second call differs"


APPLY_VARIANTS = [(m, relu, bits, False) for m in (0, 1, 2) for relu in (0, 1) for bits in (False, True)] + \
                 [(0, 1, False, True), (0, 1, True, True)]


@pytest.mark.parametrize("C,kind", RING_CASES)
def test_apply_geometry(cuda_device, C, kind):
    rows = ring_rows(C, kind)
    record_geometry(rows, C, f"apply {kind}")
    check_apply_variants(_lib.load(), rows, C, C + len(kind), APPLY_VARIANTS)


# ---------------------------------------------------------------------------------------------------- backward
def bn_inputs(rows, C, seed, mode, dev):
    g = gen(seed)
    x = rand((rows, C), g, dev, 1.5, 0.0).add_(rand(C, g, dev)).bfloat16()
    dy = rand((rows, C), g, dev).bfloat16()
    xd = x.double()
    mean = xd.mean(0).float()
    invstd = (1.0 / torch.sqrt(xd.var(0, unbiased=False) + 1e-5)).float()
    gamma = rand(C, g, dev)                                    # mixed signs
    beta = rand(C, g, dev, 0.5)
    sc = gamma * invstd
    sh = beta - mean * sc
    out = None
    if mode == 2:
        out = rand((rows, C), g, dev).bfloat16()
    elif mode == 3:
        out = torch.randint(0, 256, (rows, C // 8), generator=g, device=dev, dtype=torch.uint8)
    return x, dy, out, sc, sh, mean, invstd


def run_backward(lib, dy, x, out, sc, sh, mean, invstd, mode, dgamma=None, dbeta=None):
    rows, C = x.shape
    dgamma = torch.zeros(C, device=x.device) if dgamma is None else dgamma
    dbeta = torch.zeros(C, device=x.device) if dbeta is None else dbeta
    dx = nan_like(x)
    dy_io = dy.clone()
    _lib.check(lib.argus_bn_backward(_lib.ptr(dy_io), _lib.ptr(x), _lib.ptr(out), _lib.ptr(sc), _lib.ptr(sh),
                                     _lib.ptr(mean), _lib.ptr(invstd), _lib.ptr(dgamma), _lib.ptr(dbeta), _lib.ptr(dx),
                                     ctypes.c_int64(rows), ctypes.c_int(C), ctypes.c_int(mode), _lib.stream_ptr()))
    return dgamma, dbeta, dx, dy_io


def check_backward_modes(lib, rows, C, seed, modes):
    dev = torch.device("cuda", 0)
    for mode in modes:
        x, dy, out, sc, sh, mean, invstd = bn_inputs(rows, C, seed + mode, mode, dev)
        dgamma, dbeta, dx, dy_io = run_backward(lib, dy, x, out, sc, sh, mean, invstd, mode)
        gm = R.bn_mask(mode, dy, x, out, sc, sh)
        ref = R.bn_backward_ref(gm, x, sc, mean, invstd)
        tag = f"bn backward mode {mode} C{C} rows{rows}"
        for k, v in R.check_bn_backward(dgamma, dbeta, dx, ref, tag).items():
            note(f"bn backward {k}", v)
        if mode == 2:
            R.check_equal(dy_io, gm.bfloat16(), tag + ": dy masked in place")
        else:
            assert torch.equal(dy_io, dy), tag + ": dy changed"
        g2, b2, dx2, _ = run_backward(lib, dy, x, out, sc, sh, mean, invstd, mode)
        assert torch.equal(g2, dgamma) and torch.equal(b2, dbeta) and torch.equal(dx2, dx), tag + ": not deterministic"


@pytest.mark.parametrize("C,kind", RING_CASES)
def test_backward_geometry(cuda_device, C, kind):
    rows = ring_rows(C, kind)
    record_geometry(rows, C, f"backward {kind}")
    check_backward_modes(_lib.load(), rows, C, 3 * C + len(kind), (0, 1, 2, 3))


def test_model_shape(cuda_device):
    """layer1 of the flagship step (256 pairs of 256 x 256 images: 2 097 152 rows x 256 channels): the block-output
    apply with its ReLU bits, the act2 apply with column sums, and the backward modes the block runs there."""
    rows, C = 2097152, 256
    record_geometry(rows, C, "model shape")
    lib = _lib.load()
    check_apply_variants(lib, rows, C, 7, [(1, 1, True, False), (0, 1, False, True)])
    check_backward_modes(lib, rows, C, 8, (1, 3))


# ---------------------------------------------------------------------------------------------------- finalize
@pytest.mark.parametrize("C", [8, 64, 72, 2048])
@pytest.mark.parametrize("count_kind", ["one", "two", "large"])
def test_finalize(cuda_device, C, count_kind):
    """Partials of inputs whose mean is ~1000 x their spread: E[x^2] and mean^2 cancel to ~6 digits in the variance.
    The kernel's ordered float64 sum differs from the reference's only in order; the bound carries what that order can
    change through the cancellation (finalize_ref's var_err), and the report shows E[x^2] / var."""
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    for slots in (1, 2, 31, 32, 33, 255, 256, 257, 2 * sms(), 1184, 4000):
        g = gen(slots * 7 + C)
        mu = rand(C, g, dev, 50.0)
        sigma = torch.rand(C, generator=g, device=dev) * 0.1 + 0.01
        if count_kind == "large":
            per = 16
            x = mu + sigma * torch.randn(slots, per, C, generator=g, device=dev)
            partial = torch.stack([x.sum(1), (x * x).sum(1)], 1)
            count = slots * per
        else:
            count = 1 if count_kind == "one" else 2
            x = mu + sigma * torch.randn(count, C, generator=g, device=dev)
            partial = torch.zeros(slots, 2, C, device=dev)
            where = [0, slots - 1][:count]
            for i, s in enumerate(where):
                partial[s, 0] += x[i]
                partial[s, 1] += x[i] * x[i]
        gamma, beta = rand(C, g, dev), rand(C, g, dev)
        rm0, rv0 = rand(C, g, dev), torch.rand(C, generator=g, device=dev) + 0.5
        outs = []
        for _ in range(2):
            rm, rv = rm0.clone(), rv0.clone()
            sc, shf, mean, invstd = (torch.full((C,), float("nan"), device=dev) for _ in range(4))
            _lib.check(lib.argus_bn_finalize(_lib.ptr(partial), ctypes.c_int(slots), ctypes.c_double(count),
                                             _lib.ptr(gamma), _lib.ptr(beta), _lib.ptr(rm), _lib.ptr(rv),
                                             ctypes.c_float(0.1), ctypes.c_float(1e-5), _lib.ptr(sc), _lib.ptr(shf),
                                             _lib.ptr(mean), _lib.ptr(invstd), ctypes.c_int(C), _lib.stream_ptr()))
            outs.append(dict(mean=mean, invstd=invstd, scale=sc, shift=shf, running_mean=rm, running_var=rv))
        for k in outs[0]:
            assert torch.equal(outs[0][k], outs[1][k]), f"finalize {k} not deterministic (slots {slots})"
        ref = R.finalize_ref(partial, float(count), gamma, beta, 1e-5, 0.1, rm0, rv0)
        try:
            for k, v in R.check_finalize(outs[0], ref, 1e-5).items():
                note(f"finalize {k}", v)
        except AssertionError as e:
            raise AssertionError(f"slots {slots} count {count}: {e}") from None
        note("finalize E[x^2]/var (cancellation)", float(ref["cond"][ref["var"] > 0].max()) if (ref["var"] > 0).any() else 0.0)


# ---------------------------------------------------------------------------------------------------- max-pool
POOL_SHAPES = [(3, 2, 2), (2, 4, 4), (2, 6, 10), (1, 12, 20), (2, 16, 32), (1, 32, 8), (1, 128, 128)]


def shift_path(H, W, C):
    p2 = lambda v: v > 0 and (v & (v - 1)) == 0
    return "SHIFT" if p2(C // 8) and p2(W // 2) and p2(H // 2) else "division"


@pytest.mark.parametrize("N,H,W", POOL_SHAPES)
@pytest.mark.parametrize("C", [64, 128])
def test_maxpool(cuda_device, N, H, W, C):
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    GEOMETRY.append(dict(what="maxpool", N=N, H=H, W=W, C=C, path=shift_path(H, W, C)))
    g = gen(N * 1000 + H * 10 + W + C)
    for inputs in ("random", "tied", "dead"):
        if inputs == "tied":
            x = torch.randint(-2, 3, (N, H, W, C), generator=g, device=dev).bfloat16()
            x[:, : H // 2, : W // 2] = 1.0                      # whole windows of equal values
        else:
            x = rand((N, H, W, C), g, dev).bfloat16()
        for scales in ("positive", "negative", "mixed", "zero", "none"):
            sc = torch.rand(C, generator=g, device=dev) + 0.5
            if scales == "negative":
                sc = -sc
            elif scales == "mixed":
                sc[1::2] = -sc[1::2]                             # opposite signs within every channel pair
            elif scales == "zero":
                sc[::3] = 0.0
            sh = rand(C, g, dev) - (8.0 if inputs == "dead" else 0.0)   # dead: every window <= 0 after the ReLU
            sc_arg, sh_arg = (None, None) if scales == "none" else (sc, sh)
            y = torch.full((N, H // 2, W // 2, C), float("nan"), device=dev, dtype=torch.bfloat16)
            idx = torch.full((N, H // 2, W // 2, C), 0xEE, device=dev, dtype=torch.uint8)
            _lib.call("argus_maxpool_forward", x, sc_arg, sh_arg, y, idx, N, H, W, C, _lib.stream_ptr())
            tag = f"maxpool {N}x{H}x{W}x{C} {inputs} {scales}"
            note("maxpool y", R.check_maxpool_forward(x, sc_arg, sh_arg, y, idx, tag))
            dy = rand((N, H // 2, W // 2, C), g, dev).bfloat16()
            dx = torch.full((N, H, W, C), float("nan"), device=dev, dtype=torch.bfloat16)
            _lib.call("argus_maxpool_backward", dy, idx, dx, N, H, W, C, _lib.stream_ptr())
            note("maxpool backward dx", R.check_maxpool_backward(dx, dy, idx, tag + " backward"))


# ---------------------------------------------------------------------------------------------------- stem
def stem_inputs(N, H, W, seed, gamma_kind, dev):
    C = 64
    g = gen(seed)
    raw = rand((N, H, W, C), g, dev, 1.5).add_(rand(C, g, dev)).bfloat16()
    xd = raw.double().reshape(-1, C)
    mean = xd.mean(0).float()
    invstd = (1.0 / torch.sqrt(xd.var(0, unbiased=False) + 1e-5)).float()
    gamma = torch.rand(C, generator=g, device=dev) + 0.5
    if gamma_kind == "negative":
        gamma = -gamma
    elif gamma_kind == "mixed":
        gamma[1::2] = -gamma[1::2]
    beta = rand(C, g, dev, 0.5)
    sc = gamma * invstd
    sh = beta - mean * sc
    pooled = torch.empty(N, H // 2, W // 2, C, device=dev, dtype=torch.bfloat16)
    idx = torch.empty(N, H // 2, W // 2, C, device=dev, dtype=torch.uint8)
    _lib.call("argus_maxpool_forward", raw, sc, sh, pooled, idx, N, H, W, C, _lib.stream_ptr())
    dpool = rand((N, H // 2, W // 2, C), g, dev).bfloat16()
    return raw, sc, sh, mean, invstd, idx, dpool


def run_stem(lib, dpool, idx, raw, sc, sh, mean, invstd, dgamma=None, dbeta=None):
    N, H, W, C = raw.shape
    dgamma = torch.zeros(C, device=raw.device) if dgamma is None else dgamma
    dbeta = torch.zeros(C, device=raw.device) if dbeta is None else dbeta
    dx = nan_like(raw)
    _lib.check(lib.argus_stem_pool_bn_backward(_lib.ptr(dpool), _lib.ptr(idx), _lib.ptr(raw), _lib.ptr(sc), _lib.ptr(sh),
                                               _lib.ptr(mean), _lib.ptr(invstd), _lib.ptr(dgamma), _lib.ptr(dbeta),
                                               _lib.ptr(dx), ctypes.c_int(N), ctypes.c_int(H), ctypes.c_int(W),
                                               ctypes.c_int(C), _lib.stream_ptr()))
    return dgamma, dbeta, dx


def stem_shapes():
    # the model (512 stem images of 128 x 128), one window, the division path (Wo = 10), and enough 16 x 16 images
    # that the statistics pass (grid capped at 4 x SMs blocks of 32 patches) loops about three times
    return [(512, 128, 128), (1, 2, 2), (2, 12, 20), (6 * sms(), 16, 16)]


@pytest.mark.parametrize("shape_i", range(4))
@pytest.mark.parametrize("gamma_kind", ["positive", "negative", "mixed"])
def test_stem_pool_bn_backward(cuda_device, shape_i, gamma_kind):
    N, H, W = stem_shapes()[shape_i]
    if N == 512 and gamma_kind != "mixed":
        pytest.skip("the model shape runs once, with mixed gamma")
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    rows = N * H * W
    stat_grid = max(1, min((rows * 2 + 255) // 256, 4 * sms()))
    GEOMETRY.append(dict(what="stem", N=N, H=H, W=W, lg_wo=-1 if shift_path(H, W, 64) != "SHIFT" else "shift",
                         stat_blocks=stat_grid, patch_loops=rows // 4 / (stat_grid * 32)))
    raw, sc, sh, mean, invstd, idx, dpool = stem_inputs(N, H, W, N + H + W, gamma_kind, dev)
    dgamma, dbeta, dx = run_stem(lib, dpool, idx, raw, sc, sh, mean, invstd)
    g0, gabs = R.unpool_ref(dpool, idx, H, W)
    g0, gabs = g0.reshape(rows, 64), gabs.reshape(rows, 64)
    keep = raw.double().reshape(rows, 64) * sc.double() + sh.double() > 0
    gm = torch.where(keep, g0, torch.zeros_like(g0))
    ref = R.bn_backward_ref(gm, raw, sc, mean, invstd, g_abs=torch.where(keep, gabs, torch.zeros_like(gabs)))
    for k, v in R.check_bn_backward(dgamma, dbeta, dx, ref, f"stem {N}x{H}x{W} gamma {gamma_kind}").items():
        note(f"stem backward {k}", v)
    g2, b2, dx2 = run_stem(lib, dpool, idx, raw, sc, sh, mean, invstd)
    assert torch.equal(g2, dgamma) and torch.equal(b2, dbeta) and torch.equal(dx2, dx), "stem backward not deterministic"


# ---------------------------------------------------------------------------------------------------- avg-pool
@pytest.mark.parametrize("HW", [1, 4, 7, 8, 9, 16, 63, 64, 65])
@pytest.mark.parametrize("C", [64, 2048])
@pytest.mark.parametrize("N", [1, 512])
def test_avgpool(cuda_device, N, HW, C):
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    g = gen(N + HW + C)
    x = rand((N, HW, C), g, dev, 1.0, 0.5).bfloat16()
    y = torch.full((N, C), float("nan"), device=dev, dtype=torch.bfloat16)
    _lib.call("argus_avgpool_forward", x, y, N, HW, C, _lib.stream_ptr())
    note("avgpool y", R.check_avgpool_forward(y, x, f"avgpool {N}x{HW}x{C}"))
    dy = rand((N, C), g, dev).bfloat16()
    dx = torch.full((N * HW, C), float("nan"), device=dev, dtype=torch.bfloat16)
    _lib.call("argus_avgpool_backward", dy, dx, N, HW, C, _lib.stream_ptr())
    R.check_equal(dx.view(torch.int16), R.avgpool_backward_ref(dy, N, HW, C).view(torch.int16), "avgpool backward")
    bits = torch.randint(0, 256, (N * HW, C // 8), generator=g, device=dev, dtype=torch.uint8)
    dx.fill_(float("nan"))
    _lib.check(lib.argus_avgpool_backward_bits(_lib.ptr(dy), _lib.ptr(dx), _lib.ptr(bits), ctypes.c_int(N),
                                               ctypes.c_int(HW), ctypes.c_int(C), _lib.stream_ptr()))
    R.check_equal(dx.view(torch.int16), R.avgpool_backward_ref(dy, N, HW, C, bits).view(torch.int16),
                  "avgpool backward with bits")


# ---------------------------------------------------------------------------------------------------- accumulation
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_backward_accumulates(cuda_device, mode):
    """dgamma / dbeta that already hold gradients: dx is the same bits as with zeroed accumulators, and the accumulators
    end at prefill + this call's sums (one fp32 add each)."""
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    rows, C = ring_rows(256, "fewer_stages_than_ctas"), 256
    x, dy, out, sc, sh, mean, invstd = bn_inputs(rows, C, 40 + mode, mode, dev)
    g0, b0, dx0, dyo0 = run_backward(lib, dy, x, out, sc, sh, mean, invstd, mode)
    pg, pb = rand(C, gen(5), dev, 1e3), rand(C, gen(6), dev, 1e3)
    g1, b1, dx1, dyo1 = run_backward(lib, dy, x, out, sc, sh, mean, invstd, mode, pg.clone(), pb.clone())
    assert torch.equal(dx1, dx0) and torch.equal(dyo1, dyo0), "dx depends on what dgamma / dbeta held"
    assert torch.equal(g1, pg + g0) and torch.equal(b1, pb + b0)


def test_stem_backward_accumulates(cuda_device):
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    raw, sc, sh, mean, invstd, idx, dpool = stem_inputs(4, 32, 32, 77, "mixed", dev)
    g0, b0, dx0 = run_stem(lib, dpool, idx, raw, sc, sh, mean, invstd)
    pg, pb = rand(64, gen(7), dev, 1e3), rand(64, gen(8), dev, 1e3)
    g1, b1, dx1 = run_stem(lib, dpool, idx, raw, sc, sh, mean, invstd, pg.clone(), pb.clone())
    assert torch.equal(dx1, dx0), "dx depends on what dgamma / dbeta held"
    assert torch.equal(g1, pg + g0) and torch.equal(b1, pb + b0)


@pytest.mark.parametrize("variant", ["bf16", "fp32", "bf16-frozen"])
def test_model_backward_accumulates(cuda_device, variant):
    """argus_model_backward ADDS into the bound gradient arena: two backward passes of one forward without zeroing in
    between give twice the gradients of one. The frozen-statistics backward has no batch-norm pass (control)."""
    from argus_b200.models import NCameraCNN
    from gpu_util import structured_images

    model = NCameraCNN().to(cuda_device).set_precision("fp32" if variant == "fp32" else "bf16")
    x = structured_images(2, 6, 128, 128, 3, cuda_device)
    frozen = variant.endswith("frozen")
    if frozen:
        model.train()
        model._forward_impl(x, True)          # running statistics that are not the initial ones
        model.eval()
    else:
        model.train()
    out = model._forward_impl(x, not frozen, frozen=frozen)
    d_out = torch.randn(out.shape, generator=gen(11), device=cuda_device)
    h = model._handle.ptr
    grads = model.flat_grads
    _lib.call("argus_model_zero_grads", h, _lib.stream_ptr())
    _lib.call("argus_model_backward", h, d_out, 0, 4, _lib.stream_ptr())
    g1 = grads.clone()
    _lib.call("argus_model_backward", h, d_out, 0, 4, _lib.stream_ptr())
    torch.cuda.synchronize()
    worst = []
    for name, off, numel, _shape in model._param_infos:
        a, b = g1[off:off + numel].double(), grads[off:off + numel].double()
        err = (b - 2 * a).norm().item()
        bound = 1e-6 * a.norm().item()
        worst.append((err / bound if bound > 0 else (0.0 if err == 0 else float("inf")), name))
    worst.sort(reverse=True)
    assert worst[0][0] <= 1.0, f"{variant}: gradients of a second backward are not added: {worst[:5]}"
