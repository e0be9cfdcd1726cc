"""The float64 comparators of tests/bnpool_ref.py accept a faithful result and reject each kind of wrong kernel output
they exist to catch. No GPU: the "kernel outputs" are the references rounded as the kernels round them, then damaged."""
import pytest
import torch

import bnpool_ref as R

C = 64
ROWS = (3 * R.RING_VEC + 200) * 8 // C      # three full ring stages and a 200-vector ragged tail


def bf16_next(t, ulps):
    """t (bf16) moved by `ulps` bf16 ulps away from zero."""
    bits = t.view(torch.int16).to(torch.int32) + ulps
    return bits.to(torch.int16).view(torch.bfloat16)


def apply_case(seed=0, relu=True):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(ROWS, C, generator=g).bfloat16()
    sc = torch.randn(C, generator=g) + 0.2
    sh = torch.randn(C, generator=g)
    pre, ref, E = R.apply_ref(x, sc, sh, relu=relu)
    return x, pre, ref, E, ref.bfloat16()


def vectors(t):
    return t.reshape(-1, 8)


def test_apply_accepts_faithful_output():
    _, pre, ref, E, y = apply_case()
    assert R.check_apply(y, pre, ref, E) <= 1.0
    R.check_bits(R.bool_to_bits(pre > 0), y, pre, E)


def test_apply_rejects_two_ulps_in_one_element():
    _, pre, ref, E, y = apply_case(relu=False)
    bad = y.clone()
    i = int((ref.abs() > 0.5).flatten().nonzero()[0])
    bad.view(-1)[i] = bf16_next(bad.view(-1)[i:i + 1], 2)[0]
    with pytest.raises(AssertionError, match="ring stage"):
        R.check_apply(bad, pre, ref, E)


def test_apply_rejects_neighbouring_stage():
    _, pre, ref, E, y = apply_case(relu=False)
    bad = y.clone()
    v = vectors(bad)
    v[R.RING_VEC:2 * R.RING_VEC] = v[2 * R.RING_VEC:3 * R.RING_VEC].clone()
    with pytest.raises(AssertionError, match="ring stage 1"):
        R.check_apply(bad, pre, ref, E)


@pytest.mark.parametrize("how", ["dropped", "duplicated"])
def test_apply_rejects_wrong_tail(how):
    _, pre, ref, E, y = apply_case(relu=False)
    bad = y.clone()
    v = vectors(bad)
    nfull = v.shape[0] // R.RING_VEC * R.RING_VEC
    tail = v.shape[0] - nfull
    if how == "dropped":
        v[nfull:] = float("nan")                # the sentinel of an unwritten output
    else:
        v[nfull:] = v[nfull - tail:nfull].clone()
    with pytest.raises(AssertionError, match="tail position 0"):
        R.check_apply(bad, pre, ref, E)


def test_bits_reject_one_flip():
    _, pre, ref, E, y = apply_case()
    bits = R.bool_to_bits(pre > 0)
    bits.view(-1)[37] ^= 4
    with pytest.raises(AssertionError, match="bits"):
        R.check_bits(bits, y, pre, E)


def test_colsum_accepts_and_rejects():
    _, pre, ref, E, y = apply_case()
    yd = y.double().reshape(-1, C)
    partial = torch.stack([yd[i::5].sum(0) for i in range(5)]).float()
    assert R.check_colsum(partial, y) <= 1.0
    partial[3, 7] += yd[:, 7].abs().sum() * 2 ** -14
    with pytest.raises(AssertionError, match="ch 7"):
        R.check_colsum(partial, y)


def bn_case(mode, seed=1):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(ROWS, C, generator=g) * 1.5 + torch.randn(C, generator=g)).bfloat16()
    dy = torch.randn(ROWS, C, generator=g).bfloat16()
    xf = x.double()
    mean, var = xf.mean(0), xf.var(0, unbiased=False)
    invstd = (1 / torch.sqrt(var + 1e-5)).float()
    mean = mean.float()
    gamma = torch.rand(C, generator=g) + 0.5
    sc = gamma * invstd
    sh = -mean * sc
    out = None
    if mode == 2:
        out = torch.randn(ROWS, C, generator=g).bfloat16()
    elif mode == 3:
        out = R.bool_to_bits(torch.rand(ROWS, C, generator=g) > 0.5)
    gm = R.bn_mask(mode, dy, x, out, sc, sh)
    return x, gm, sc, mean, invstd, R.bn_backward_ref(gm, x, sc, mean, invstd)


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_bn_backward_accepts_faithful_output(mode):
    x, gm, sc, mean, invstd, ref = bn_case(mode)
    r = R.check_bn_backward(ref["dgamma"].float(), ref["dbeta"].float(), ref["dx"].bfloat16(), ref)
    assert max(r.values()) <= 1.0


def test_bn_backward_rejects_dgamma_off_by_one_partial():
    """dx formed with a dgamma that still holds one block's partial sum (what reading an accumulator that was not zero
    gives) fails, although dgamma / dbeta themselves are right."""
    x, gm, sc, mean, invstd, ref = bn_case(1)
    xd = x.double().reshape(-1, C)
    rows_per_stage = R.RING_VEC * 8 // C
    part = (gm[:rows_per_stage] * (xd[:rows_per_stage] - mean.double())).sum(0) * invstd.double()
    dg = ref["dgamma"] + part
    M = xd.shape[0]
    c2 = sc.double() * dg * invstd.double() / M
    dx = sc.double() * gm - c2 * xd + (c2 * mean.double() - sc.double() * ref["dbeta"] / M)
    with pytest.raises(AssertionError, match="dx"):
        R.check_bn_backward(ref["dgamma"].float(), ref["dbeta"].float(), dx.bfloat16(), ref)


def test_bn_backward_rejects_wrong_sums():
    x, gm, sc, mean, invstd, ref = bn_case(0)
    dbeta = ref["dbeta"].clone()
    dbeta[5] += gm[:, 5].abs().sum() * 2 ** -12
    with pytest.raises(AssertionError, match="dbeta"):
        R.check_bn_backward(ref["dgamma"].float(), dbeta.float(), ref["dx"].bfloat16(), ref)


def test_mode1_mask_is_the_fma_sign():
    """x sc + sh in float64 is the sign fmaf sees: an element exactly on the decision stays masked."""
    x = torch.tensor([[1.5] * 8], dtype=torch.bfloat16)
    sc = torch.full((8,), 2.0)
    sh = torch.full((8,), -3.0)
    g = R.bn_mask(1, torch.ones(1, 8).bfloat16(), x, None, sc, sh)
    assert torch.all(g == 0)


def pool_case(seed=3, N=2, H=6, W=10, Cp=16, scale_sign=1.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(-2, 3, (N, H, W, Cp), generator=g).bfloat16()   # heavily tied
    sc = scale_sign * (torch.rand(Cp, generator=g) + 0.5)
    sh = torch.randn(Cp, generator=g)
    sgn = torch.where(sc < 0, -1.0, 1.0).double()
    taps, ok = R.pool_windows(x.double(), 0.0)
    key = torch.where(ok, taps * sgn[:, None], torch.tensor(float("-inf"), dtype=torch.float64))
    best, first = key.max(-1)
    _, ref, _ = R.apply_ref(best * sgn, sc, sh)
    return x, sc, sh, ref.bfloat16(), first.to(torch.uint8), key


@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_maxpool_accepts_faithful_output(sign):
    x, sc, sh, y, idx, _ = pool_case(scale_sign=sign)
    assert R.check_maxpool_forward(x, sc, sh, y, idx) <= 1.0


def test_maxpool_rejects_non_maximal_tap():
    x, sc, sh, y, idx, key = pool_case()
    ok = torch.isfinite(key)
    best = key.max(-1).values
    smaller = ok & (key < best[..., None])
    n, a, b, c, t = (int(v) for v in smaller.nonzero()[0])
    bad = idx.clone()
    bad[n, a, b, c] = t
    with pytest.raises(AssertionError, match="non-maximal"):
        R.check_maxpool_forward(x, sc, sh, y, bad)


def test_maxpool_rejects_border_tap():
    x, sc, sh, y, idx, _ = pool_case()
    bad = idx.clone()
    bad[0, 0, 2, 0] = 1        # top row of the first window row: padding
    with pytest.raises(AssertionError, match="out-of-bounds"):
        R.check_maxpool_forward(x, sc, sh, y, bad)
    bad = idx.clone()
    bad[0, 1, 0, 0] = 9
    with pytest.raises(AssertionError, match="0..8"):
        R.check_maxpool_forward(x, sc, sh, y, bad)


def test_maxpool_backward_accepts_and_rejects():
    x, sc, sh, y, idx, _ = pool_case()
    g = torch.Generator().manual_seed(9)
    dy = torch.randn(*idx.shape, generator=g).bfloat16()
    ref, _ = R.unpool_ref(dy, idx, x.shape[1], x.shape[2])
    assert R.check_maxpool_backward(ref.bfloat16(), dy, idx) <= 1.0
    other = idx.clone()
    other[0, 1, 1, 3] = (int(other[0, 1, 1, 3]) + 1) % 9
    with pytest.raises(AssertionError):
        R.check_maxpool_backward(ref.bfloat16(), dy, other)


def test_finalize_accepts_and_rejects():
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(1000, C, generator=g, dtype=torch.float64) * 0.1 + 100).float()
    partial = torch.stack([torch.stack([x[i::7].double().sum(0), (x[i::7].double() ** 2).sum(0)]) for i in range(7)]).float()
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    rm, rv = torch.zeros(C), torch.ones(C)
    ref = R.finalize_ref(partial, 1000.0, gamma, beta, 1e-5, 0.1, rm, rv)
    out = {k: ref[k].float() for k in ("mean", "invstd", "running_mean", "running_var")}
    out["scale"] = gamma * out["invstd"]
    out["shift"] = beta - out["mean"] * out["scale"]
    assert max(R.check_finalize(out, ref, 1e-5).values()) <= 1.0
    out["invstd"] = out["invstd"].clone()
    out["invstd"][3] = torch.nextafter(torch.nextafter(out["invstd"][3:4], torch.tensor([1e9])),
                                       torch.tensor([1e9]))[0] * (1 + 2 ** -22)
    with pytest.raises(AssertionError, match="invstd"):
        R.check_finalize(out, ref, 1e-5)


def test_avgpool_backward_ref_is_exact_rounding():
    dy = torch.tensor([[1.0, 3.0, -7.0, 0.5, 1.0, 1.0, 1.0, 1.0]]).bfloat16()
    out = R.avgpool_backward_ref(dy, 1, 7, 8)
    want = (dy.float() * (torch.tensor(1.0) / 7)).bfloat16().expand(7, 8)
    assert torch.equal(out, want)
