"""GPU parity of the tcgen05 convolution primitives (through the C ABI) against torch fp32 convolutions.

Inputs are rounded to bf16 first, so the only differences are fp32 accumulation order and the final bf16 rounding.
"""
import pytest
import torch
import torch.nn.functional as F

from argus_b200 import _lib

pytestmark = pytest.mark.gpu


def nhwc(x):  # NCHW fp32 -> NHWC bf16 contiguous
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def from_nhwc(y):
    return y.float().permute(0, 3, 1, 2).contiguous()


def pack_w(w):  # [Cout,Cin,kh,kw] -> [Cout,kh,kw,Cin] bf16
    return w.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def rel_err(a, b):
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


CASES = [
    # N, H, W, Cin, Cout, k, stride
    (4, 64, 64, 64, 256, 1, 1),
    (4, 64, 64, 64, 64, 3, 1),
    (2, 64, 64, 128, 128, 3, 2),
    (2, 64, 64, 256, 512, 1, 2),
    (2, 16, 16, 1024, 256, 1, 1),
    (2, 8, 8, 512, 512, 3, 1),
    (4, 8, 8, 512, 2048, 1, 1),
    (2, 4, 4, 512, 512, 3, 1),      # tile spans several images, M tail
    (6, 16, 16, 256, 256, 3, 2),
    (300, 1, 1, 2048, 1024, 1, 1),  # fully connected layer, ragged M
    (2, 64, 64, 256, 64, 1, 1),     # Cout = 64: transposed all-taps weight-gradient kernel (4 channel boxes)
    (3, 32, 32, 64, 64, 1, 1),      # ... single box, padded pair
    (20, 32, 32, 128, 128, 3, 1),   # halo mode with BLOCK_N = 128 and two channel blocks (layer2 shape)
    (3, 16, 16, 64, 128, 3, 1),     # halo mode, eight image rows per tile
    (2, 8, 16, 128, 64, 3, 1),      # halo mode, tile = one whole (8 x 16) image
    (8, 64, 64, 64, 256, 1, 1),     # >= 148 tiles of 256 columns in the forward
    (8, 64, 64, 256, 64, 1, 1),     # ... and in the dgrad (output = the 256 input channels)
    (16, 32, 32, 128, 512, 1, 1),   # 256-column tiles, two N tiles
]


@pytest.mark.parametrize("case", CASES)
def test_conv_forward(cuda_device, case):
    N, H, W, Cin, Cout, k, s = case
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.randn(N, Cin, H, W, generator=g).to(cuda_device)
    w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5).to(cuda_device)
    xb, wb = nhwc(x), pack_w(w)
    Ho, Wo = H // s, W // s
    y = torch.full((N, Ho, Wo, Cout), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    import ctypes
    slots = ctypes.c_int()
    _lib.check(_lib.load().argus_conv2d_stat_slots(N, H, W, Cin, Cout, k, s, 0, ctypes.byref(slots)))
    partial = torch.zeros(slots.value, 2, Cout, device=cuda_device)
    _lib.call("argus_conv2d_forward", xb, wb, y, N, H, W, Cin, Cout, k, s, 0, None, None, None, 0, partial,
              slots.value, _lib.stream_ptr())
    torch.cuda.synchronize()
    ref = F.conv2d(xb.float().permute(0, 3, 1, 2), wb.float().permute(0, 3, 1, 2), stride=s, padding=k // 2)
    got = from_nhwc(y)
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) < 5e-3
    assert (got - ref).abs().max().item() < 0.06
    yf = y.float().reshape(-1, Cout)
    ssum, ssq = partial.double().sum(0)
    assert torch.allclose(ssum, yf.double().sum(0), rtol=1e-4, atol=1e-2)
    assert torch.allclose(ssq, (yf.double() ** 2).sum(0), rtol=1e-4, atol=1e-2)
    # deterministic reduction: a second launch reproduces every partial sum bit for bit
    partial2 = torch.zeros_like(partial)
    _lib.call("argus_conv2d_forward", xb, wb, y, N, H, W, Cin, Cout, k, s, 0, None, None, None, 0, partial2,
              slots.value, _lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(partial, partial2)


def test_conv_forward_fused_epilogue(cuda_device):
    N, H, W, Cin, Cout, k, s = 2, 32, 32, 128, 512, 1, 1
    g = torch.Generator(device="cpu").manual_seed(2)
    x = torch.randn(N, Cin, H, W, generator=g).to(cuda_device)
    w = (torch.randn(Cout, Cin, k, k, generator=g) / Cin ** 0.5).to(cuda_device)
    scale = (torch.rand(Cout, generator=g) + 0.5).to(cuda_device)
    shift = torch.randn(Cout, generator=g).to(cuda_device)
    res = nhwc(torch.randn(N, Cout, H, W, generator=g).to(cuda_device))
    xb, wb = nhwc(x), pack_w(w)
    y = torch.empty((N, H, W, Cout), device=cuda_device, dtype=torch.bfloat16)
    _lib.call("argus_conv2d_forward", xb, wb, y, N, H, W, Cin, Cout, k, s, 0, scale, shift, res, 1, None, 0,
              _lib.stream_ptr())
    torch.cuda.synchronize()
    ref = F.conv2d(xb.float().permute(0, 3, 1, 2), wb.float().permute(0, 3, 1, 2))
    ref = torch.relu(ref * scale[None, :, None, None] + shift[None, :, None, None] + from_nhwc(res))
    assert rel_err(from_nhwc(y), ref) < 5e-3


@pytest.mark.parametrize("case", CASES[:9] + CASES[10:])
def test_conv_dgrad(cuda_device, case):
    N, H, W, Cin, Cout, k, s = case
    g = torch.Generator(device="cpu").manual_seed(3)
    Ho, Wo = H // s, W // s
    dy = torch.randn(N, Cout, Ho, Wo, generator=g).to(cuda_device)
    w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cout * k * k) ** 0.5).to(cuda_device)
    dyb, wb = nhwc(dy), pack_w(w)
    dx = torch.zeros((N, H, W, Cin), device=cuda_device, dtype=torch.bfloat16)
    res = None
    if s == 1:
        res = nhwc(torch.randn(N, Cin, H, W, generator=g).to(cuda_device))
    _lib.call("argus_conv2d_dgrad", dyb, wb, dx, N, H, W, Cin, Cout, k, s, res, _lib.stream_ptr())
    torch.cuda.synchronize()
    ref = F.conv_transpose2d(dyb.float().permute(0, 3, 1, 2), wb.float().permute(0, 3, 1, 2), stride=s,
                             padding=k // 2, output_padding=s - 1)
    if res is not None:
        ref = ref + from_nhwc(res)
    assert ref.shape == (N, Cin, H, W)
    assert rel_err(from_nhwc(dx), ref) < 5e-3


@pytest.mark.parametrize("case", CASES)
def test_conv_wgrad(cuda_device, case):
    N, H, W, Cin, Cout, k, s = case
    g = torch.Generator(device="cpu").manual_seed(4)
    Ho, Wo = H // s, W // s
    x = torch.randn(N, Cin, H, W, generator=g).to(cuda_device)
    dy = torch.randn(N, Cout, Ho, Wo, generator=g).to(cuda_device)
    xb, dyb = nhwc(x), nhwc(dy)
    dw = torch.zeros((Cout, k, k, Cin), device=cuda_device, dtype=torch.float32)
    _lib.call("argus_conv2d_wgrad", dyb, xb, dw, N, H, W, Cin, Cout, k, s, 0, _lib.stream_ptr())
    torch.cuda.synchronize()
    xr = xb.float().permute(0, 3, 1, 2).requires_grad_(True)
    wr = torch.zeros(Cout, Cin, k, k, device=cuda_device, requires_grad=True)
    out = F.conv2d(xr, wr, stride=s, padding=k // 2)
    out.backward(dyb.float().permute(0, 3, 1, 2))
    ref = wr.grad.permute(0, 2, 3, 1)
    assert rel_err(dw, ref) < 2e-3
    dw2 = torch.zeros_like(dw)
    _lib.call("argus_conv2d_wgrad", dyb, xb, dw2, N, H, W, Cin, Cout, k, s, 0, _lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(dw, dw2)  # split-K partials are reduced in a fixed order


def s2d_pack(img):
    """Test-side restatement of the stem input layout: [N,3,H,W] fp32 -> [N,H/2,W/2+4,16] bf16."""
    N, C, H, W = img.shape
    v = img.reshape(N, C, H // 2, 2, W // 2, 2).permute(0, 2, 4, 3, 5, 1)  # N, i, j, a, b, c
    v = v.reshape(N, H // 2, W // 2, 12)
    out = torch.zeros(N, H // 2, W // 2 + 4, 16, device=img.device)
    out[:, :, 2:2 + W // 2, :12] = v
    return out.to(torch.bfloat16).contiguous()


def stem_pack_w(w):
    """[64,3,7,7] -> [64][p 4][q 4][16] bf16 with kh = 2p + a - 1, kw = 2q + b - 1."""
    out = torch.zeros(64, 4, 4, 16, device=w.device)
    for p in range(4):
        for a in range(2):
            kh = 2 * p + a - 1
            if not 0 <= kh < 7:
                continue
            for q in range(4):
                for b in range(2):
                    kw = 2 * q + b - 1
                    if not 0 <= kw < 7:
                        continue
                    out[:, p, q, (a * 2 + b) * 3:(a * 2 + b) * 3 + 3] = w[:, :, kh, kw]
    return out.reshape(64, 256).to(torch.bfloat16).contiguous()


@pytest.mark.parametrize("N,H,W", [(2, 64, 64), (3, 256, 256)])
def test_stem(cuda_device, N, H, W):
    g = torch.Generator(device="cpu").manual_seed(5)
    img = torch.rand(N, 3, H, W, generator=g).to(cuda_device)
    w = (torch.randn(64, 3, 7, 7, generator=g) / 147 ** 0.5).to(cuda_device)
    xs, ws = s2d_pack(img), stem_pack_w(w)
    y = torch.empty((N, H // 2, W // 2, 64), device=cuda_device, dtype=torch.bfloat16)
    _lib.call("argus_conv2d_forward", xs, ws, y, N, H, W, 3, 64, 7, 2, 1, None, None, None, 0, None, 0,
              _lib.stream_ptr())
    torch.cuda.synchronize()
    ref = F.conv2d(img.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), stride=2, padding=3)
    assert rel_err(from_nhwc(y), ref) < 5e-3
    # weight gradient of the stem, in the repacked [64][256] layout
    dy = torch.randn(N, 64, H // 2, W // 2, generator=g).to(cuda_device)
    dyb = nhwc(dy)
    dw = torch.zeros((64, 256), device=cuda_device)
    _lib.call("argus_conv2d_wgrad", dyb, xs, dw, N, H, W, 3, 64, 7, 2, 1, _lib.stream_ptr())
    torch.cuda.synchronize()
    wr = torch.zeros(64, 3, 7, 7, device=cuda_device, requires_grad=True)
    F.conv2d(img.to(torch.bfloat16).float(), wr, stride=2, padding=3).backward(dyb.float().permute(0, 3, 1, 2))
    ref_packed = stem_pack_w_f32(wr.grad)
    mask = stem_pack_w_f32(torch.ones_like(wr.grad))  # slots that alias no real filter tap hold don't-care values
    assert rel_err(dw * mask, ref_packed) < 2e-3


def stem_pack_w_f32(w):
    out = torch.zeros(64, 4, 4, 16, device=w.device)
    for p in range(4):
        for a in range(2):
            kh = 2 * p + a - 1
            if not 0 <= kh < 7:
                continue
            for q in range(4):
                for b in range(2):
                    kw = 2 * q + b - 1
                    if not 0 <= kw < 7:
                        continue
                    out[:, p, q, (a * 2 + b) * 3:(a * 2 + b) * 3 + 3] = w[:, :, kh, kw]
    return out.reshape(64, 256)
