"""The weight-gradient reference and comparators of tests/wgrad_ref.py, without a GPU: the reference against float64
autograd of the convolution it stands for, the planning mirror on known geometries, and each comparator rejecting the
faults the kernels could make, with a message that names the fault."""
import pytest
import torch
import torch.nn.functional as F

import wgrad_ref as wr
from test_conv_gpu import s2d_pack


def problem(mode, shape, exact=True, seed=0):
    dy, x = wr.make_operands(mode, shape, exact, torch.Generator().manual_seed(seed), "cpu")
    return wr.Problem(mode, shape, dy, x)


@pytest.mark.parametrize("shape", [(3, 8, 8, 64, 128, 3, 1), (2, 8, 8, 128, 64, 3, 2), (5, 4, 4, 64, 128, 1, 2),
                                   (2, 2, 2, 128, 64, 3, 1)])
def test_reference_is_the_convolution_gradient(shape):
    N, H, W, Cin, Cout, k, s = shape[:7]
    prob = problem("conv", shape + (0,), exact=False)
    ref, A = prob.reference()
    x = prob.x.double().permute(0, 3, 1, 2)
    w = torch.zeros(Cout, Cin, k, k, dtype=torch.float64, requires_grad=True)
    F.conv2d(x, w, stride=s, padding=k // 2).backward(prob.dy.double().permute(0, 3, 1, 2))
    want = w.grad.permute(0, 2, 3, 1).reshape(Cout, -1)
    assert torch.allclose(ref, want, rtol=1e-12, atol=1e-12)
    assert bool((A >= ref.abs()).all())


def test_stem_reference_is_the_7x7_gradient():
    N, H, W = 2, 32, 32
    g = torch.Generator().manual_seed(1)
    img = torch.rand(N, 3, H, W, generator=g).to(torch.bfloat16).double()
    xs = s2d_pack(img.float())
    dy = torch.randn(N, H // 2, W // 2, 64, generator=g).to(torch.bfloat16)
    ref, _ = wr.Problem("conv", (N, H, W, 3, 64, 7, 2, 1), dy, xs).reference()
    w = torch.zeros(64, 3, 7, 7, dtype=torch.float64, requires_grad=True)
    F.conv2d(img, w, stride=2, padding=3).backward(dy.double().permute(0, 3, 1, 2))
    want = torch.zeros(64, 4, 4, 16, dtype=torch.float64)
    for p in range(4):
        for q in range(4):
            for a in range(2):
                for b in range(2):
                    kh, kw = 2 * p + a - 1, 2 * q + b - 1
                    if 0 <= kh < 7 and 0 <= kw < 7:
                        want[:, p, q, (a * 2 + b) * 3:(a * 2 + b) * 3 + 3] = w.grad[:, :, kh, kw]
    want = want.reshape(64, 256)
    mask = wr.stem_mask()
    assert int(mask[0].sum()) == 147
    assert torch.allclose(ref[mask], want[mask], rtol=1e-12, atol=1e-12)
    # slots outside the mask (kh = -1, kw = -1, the spare channels) still multiply image pixels the packed window holds:
    # the kernel computes them like any other column, and the weight update ignores them
    assert bool((ref[~mask] != 0).any())


def test_stacked_and_gram_references():
    shape = (3, 8, 8, 64, 128, 1, 2, 0)
    prob = problem("stacked", shape, exact=False)
    ref, _ = prob.reference()
    xs = prob.x[:, ::2, ::2, :].reshape(-1, 64).double()
    assert torch.allclose(ref[:128], prob.dy.reshape(-1, 128).double().t() @ xs, rtol=1e-12, atol=1e-12)
    assert torch.allclose(ref[128:], xs.t() @ xs, rtol=1e-12, atol=1e-12)
    gram, _ = wr.Problem("gram", shape, None, prob.x).reference()
    assert torch.equal(gram, ref[128:])


def test_split_sums_add_up():
    shape = (37, 4, 4, 128, 128, 1, 1, 0)
    prob = problem("conv", shape)
    p = wr.plan("conv", shape, 148)
    assert (p["splits"], p["per"], p["kblocks"]) == (2, 5, 10)
    assert torch.equal(sum(prob.split_sums(p)), prob.reference()[0])


def test_plan_mirror():
    # the model's layer1 3x3 at batch 256 on 148 SMs: transposed kernel, 148 splits of 111 k-blocks, last one 67
    p = wr.plan("conv", (256, 64, 64, 64, 64, 3, 1, 0), 148)
    assert (p["xpose"], p["n"], p["splits"], p["per"], p["kblocks"]) == (1, 10, 148, 111, 16384)
    assert (p["xpose"], p["n"]) == (1, 10)
    p = wr.plan("conv", (2, 64, 64, 3, 64, 7, 2, 1), 148)
    assert (p["xpose"], p["n"], p["num_taps"], p["ktot"]) == (1, 4, 4, 256)
    p = wr.plan("conv", (300, 1, 1, 2048, 1024, 1, 1, 0), 148)            # the fc at batch 300: one split
    assert (p["xpose"], p["n"], p["splits"], p["scratch"]) == (0, 256, 1, 0)
    p = wr.plan("conv", (40, 4, 4, 256, 256, 1, 1, 0), 148)               # 10 k-blocks: 74 splits capped to 2
    assert (p["uncapped"], p["capped"], p["splits"]) == (74, 2, 2)
    # 13 k-blocks asked for 3 splits of 5: the shrink keeps 3 (5 + 5 + 3); 9 k-blocks in 8 splits would leave the last
    # ones empty: per = 2, so 4 splits cover them
    assert wr._shrink(3, 13) == 3 and wr._shrink(8, 9) == 5 and wr._shrink(148, 150) == 75
    p = wr.plan("stacked", (4, 16, 16, 64, 256, 1, 1, 0), 148)
    assert (p["rows"], p["co_split"], p["stacked"], p["co_tiles"], p["n"]) == (320, 256, 1, 3, 64)
    p = wr.plan("gram", (4, 16, 16, 256, 512, 1, 2, 0), 148)
    assert (p["rows"], p["co_split"], p["stacked"], p["ktot"]) == (256, 0, 1, 256)


# ------------------------------------------------------------------------------------------------------------------
# mutations: every fault is rejected, and the message names it
# ------------------------------------------------------------------------------------------------------------------
RAGGED_1X1 = (37, 4, 4, 128, 128, 1, 1, 0)   # 592 pixels: 10 k-blocks in 2 splits of 5, the last k-block holds 16
TAPS_3X3 = (13, 4, 4, 128, 128, 3, 1, 0)


def setup(shape, exact=True, mode="conv"):
    prob = problem(mode, shape, exact)
    p = wr.plan(mode, shape, 148)
    ref, A = prob.reference()
    return prob, p, ref, A


def rejects(fn, *needles):
    with pytest.raises(wr.WgradMismatch) as e:
        fn()
    msg = str(e.value)
    for n in needles:
        assert n in msg, msg
    return msg


def test_exact_accepts_the_reference():
    prob, p, ref, A = setup(RAGGED_1X1)
    wr.check_exact(prob, ref.float(), ref, A, p)
    assert float(A.max()) < wr.EXACT_LIMIT and bool((ref != 0).any())


def test_exact_rejects_one_element_off_by_one():
    prob, p, ref, A = setup(RAGGED_1X1)
    got = ref.float().clone()
    got[70, 33] += 1
    rejects(lambda: wr.check_exact(prob, got, ref, A, p), "1 of", "co 70, tap 0, ci 33", "co tile 0, ci tile 0")


def test_bound_rejects_four_times_the_bound():
    prob, p, ref, A = setup(RAGGED_1X1, exact=False)
    got = ref.float()
    worst = wr.check_bound(prob, got, ref, A, p)
    assert worst <= 1.0
    b = wr.bound(ref, A, p)
    got = got.clone()
    got[5, 100] = float(ref[5, 100] + 4 * b[5, 100])
    rejects(lambda: wr.check_bound(prob, got, ref, A, p), "co 5, tap 0, ci 100", "err/bound 3.99")


def test_rejects_a_dropped_kblock():
    prob, p, ref, A = setup(RAGGED_1X1)
    kb = 3
    block = prob.reference(kb, kb + 1)[0]
    got = ref.clone()
    got[:128, :128] -= block[:128, :128]     # one (co tile, ci tile, tap) item of split 0 skipped k-block 3
    rejects(lambda: wr.check_exact(prob, got.float(), ref, A, p), "k-block 3 (split 0) missing")


def test_rejects_a_split_added_twice():
    prob, p, ref, A = setup(RAGGED_1X1)
    got = ref + prob.split_sums(p)[1]
    msg = rejects(lambda: wr.check_exact(prob, got.float(), ref, A, p), "split 1 (k-blocks 5..9) added twice")
    assert "k-block" in msg


def test_rejects_the_ragged_kblock_counted_twice():
    prob, p, ref, A = setup(RAGGED_1X1)
    last = p["kblocks"] - 1
    got = ref + prob.reference(last, last + 1)[0]
    rejects(lambda: wr.check_exact(prob, got.float(), ref, A, p),
            "k-block 9 (split 1) (the ragged last k-block) counted twice")


def test_rejects_a_tap_written_into_the_next_taps_columns():
    prob, p, ref, A = setup(TAPS_3X3)
    got = ref.clone()
    got[:, 4 * 128:5 * 128] = ref[:, 3 * 128:4 * 128]
    rejects(lambda: wr.check_exact(prob, got.float(), ref, A, p), "tap 4",
            "a tap's block was written into the next tap's columns")


def test_rejects_two_rows_swapped():
    prob, p, ref, A = setup(TAPS_3X3)
    got = ref.clone()
    got[[17, 90]] = ref[[90, 17]]
    rejects(lambda: wr.check_exact(prob, got.float(), ref, A, p), "co 17", "reference of row 90: rows swapped")


def test_rejects_a_write_past_cout():
    shape = (3, 4, 4, 128, 64, 1, 1, 0)    # Cout = 64: rows 64..127 of the only co tile must be skipped
    p = wr.plan("conv", shape, 148)
    n = 64 * 128
    buf = torch.full((wr.SENTINEL * 2 + n,), wr.SENTINEL_VALUE)
    wr.check_sentinels(buf, n, p)
    buf[wr.SENTINEL + n + 130] = 2.0
    rejects(lambda: wr.check_sentinels(buf, n, p), "row 65 (>= 64 rows), column 2")
    buf = torch.full((wr.SENTINEL * 2 + n,), wr.SENTINEL_VALUE)
    buf[3] = 0.0
    rejects(lambda: wr.check_sentinels(buf, n, p), "before dW")


def test_rejects_the_stem_mask_on_a_real_tap():
    shape = (2, 32, 32, 3, 64, 7, 2, 1)
    prob, p, ref, A = setup(shape)
    wr.check_exact(prob, ref.float(), ref, A, p)
    mask = wr.stem_mask().clone()
    mask[:, 64 + 16 + 4] = False              # tap 1, column block 1, channel 4: a real filter tap (kh 1 or 2, kw 1)
    assert bool(wr.stem_mask()[:, 64 + 16 + 4].all())
    got = (ref * (mask | ~wr.stem_mask())).float()
    rejects(lambda: wr.check_exact(prob, got, ref, A, p), "tap 1 (s2d row offset -1), slot 20", "zero: never written")


def test_nan_is_named_stale_scratch():
    prob, p, ref, A = setup(RAGGED_1X1)
    got = ref.float().clone()
    got[1, 2] = float("nan")
    rejects(lambda: wr.check_exact(prob, got, ref, A, p), "stale split-K scratch")
    rejects(lambda: wr.check_bound(prob, got, ref, A, p), "stale split-K scratch")


def test_accumulation_check():
    prob, p, ref, A = setup(RAGGED_1X1, exact=False)
    r0 = ref.float()
    D = torch.randn(r0.shape, generator=torch.Generator().manual_seed(3))
    wr.check_accumulated(D + r0, D, r0, p)
    got = D + r0
    got[7, 8] = r0[7, 8]        # the start value was overwritten instead of added to
    rejects(lambda: wr.check_accumulated(got, D, r0, p), "fl(D + result from 0)", "co 7, tap 0, ci 8")


def test_exact_operands_must_be_exact():
    prob, p, ref, A = setup(RAGGED_1X1, exact=False)
    A = A + wr.EXACT_LIMIT
    with pytest.raises(ValueError):
        wr.check_exact(prob, ref.float(), ref, A, p)
