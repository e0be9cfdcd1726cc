"""CPU: the element-wise epilogue comparator (tests/epilogue_ref.py) accepts a correctly computed output and rejects
outputs that a norm-based check would pass: one element off by two ulps, one 128-row block shifted by a row, one
channel with its neighbour's shift, one flipped bit of the ReLU mask."""
import pytest
import torch

import epilogue_ref as er


def _case():
    g = torch.Generator().manual_seed(0)
    N, H, W, Cin, Cout = 2, 16, 16, 64, 64          # 512 rows: four M tiles
    x = torch.randn(N, H, W, Cin, generator=g).to(torch.bfloat16)
    w = (torch.randn(Cout, 1, 1, Cin, generator=g) / Cin ** 0.5).to(torch.bfloat16)
    scale = torch.randn(Cout, generator=g)          # negative scales included
    shift = torch.randn(Cout, generator=g)
    res = torch.randn(N * H * W, Cout, generator=g).to(torch.bfloat16)
    acc, absacc = er.conv_nhwc_f64(x, w, 1, 1)
    # what a correct kernel stores: fp32 accumulation and epilogue, bf16 result, bits of the fp32 pre-activation
    acc32 = x.float().reshape(-1, Cin) @ w.float().reshape(Cout, Cin).t()
    pre32 = acc32 * scale + shift + res.float()
    y = pre32.clamp_min(0).to(torch.bfloat16)
    bits = er.bool_to_bits(pre32 > 0)
    pre, ref, E = er.epilogue_ref(acc, absacc, scale, shift, res, relu=True)
    return dict(y=y, bits=bits, pre=pre, ref=ref, E=E, acc32=acc32, scale=scale, shift=shift, res=res)


def test_bit_mask_layout_round_trips():
    m = torch.rand(300, 128, generator=torch.Generator().manual_seed(1)) > 0.5
    assert torch.equal(er.bits_to_bool(er.bool_to_bits(m), 128), m)
    one = torch.zeros(1, 64, dtype=torch.bool)
    one[0, 9] = True
    assert er.bool_to_bits(one).tolist() == [[0, 2, 0, 0, 0, 0, 0, 0]]   # channel c = byte c // 8, bit c % 8


def test_accepts_correct_output():
    c = _case()
    worst = er.check_values(c["y"], c["ref"], c["E"])
    assert worst <= 1.0
    er.check_bits(c["bits"], c["y"], c["pre"], c["E"])


def test_rejects_two_ulp_error():
    c = _case()
    y = c["y"].clone()
    r, ch = divmod(int(c["ref"].abs().argmax()), c["ref"].shape[1])
    y.view(torch.int16)[r, ch] += 2
    with pytest.raises(AssertionError, match="1 of"):
        er.check_values(y, c["ref"], c["E"])


def test_rejects_row_shift_in_one_tile():
    c = _case()
    y = c["y"].clone()
    y[256:384] = c["y"][255:383]
    with pytest.raises(AssertionError, match="M tile 2"):
        er.check_values(y, c["ref"], c["E"])


def test_rejects_neighbour_shift():
    c = _case()
    shift = c["shift"].clone()
    shift[37] = shift[38]
    y = (c["acc32"] * c["scale"] + shift + c["res"].float()).clamp_min(0).to(torch.bfloat16)
    with pytest.raises(AssertionError, match="ch 37"):
        er.check_values(y, c["ref"], c["E"])


def test_rejects_flipped_mask_bit():
    c = _case()
    bits = c["bits"].clone()
    bits[511, 7] ^= 0x10     # last row of the last M tile, channel 60
    with pytest.raises(AssertionError, match="M tile 3"):
        er.check_bits(bits, c["y"], c["pre"], c["E"])


def test_statistics_check_rejects_a_lost_row():
    c = _case()
    y = c["y"].float()
    partial = torch.stack([y.sum(0), (y * y).sum(0)]).unsqueeze(0)
    er.check_stat_slots(partial, c["y"], 64)
    partial_short = torch.stack([y[:-1].sum(0), (y[:-1] * y[:-1]).sum(0)]).unsqueeze(0)
    with pytest.raises(AssertionError):
        er.check_stat_slots(partial_short, c["y"], 64)
