"""Per-op parity (through the C ABI) of the masked, statistics-producing dgrad that feeds the algebraic batch-norm
backward (csrc/bn_algebra.cu). The small kernels of that backward and the whole conv(1x1) + BN backward are checked
element by element in test_bnalg_gpu.py, the stacked weight-gradient + Gram launch in test_wgrad_gpu.py."""
import ctypes

import pytest
import torch

from argus_b200 import _lib

pytestmark = pytest.mark.gpu


def bf(t):
    return t.bfloat16()


@pytest.mark.parametrize("N,H,W,Cin,Cout", [(4, 16, 16, 256, 64), (20, 32, 32, 512, 128), (3, 8, 8, 1024, 256)])
def test_dgrad_out_bits_and_statistics(cuda_device, N, H, W, Cin, Cout):
    """conv1-dgrad as the model launches it: + identity-branch gradient, masked by the ReLU bits of the tensor whose
    gradient it produces, with per-CTA channel sums of the stored (masked) result."""
    g = torch.Generator().manual_seed(N + Cin)
    rows = N * H * W
    dy = bf(torch.randn(rows, Cout, generator=g)).to(cuda_device)
    w = bf(torch.randn(Cout, Cin, generator=g) / Cout ** 0.5).to(cuda_device)
    res = bf(torch.randn(rows, Cin, generator=g)).to(cuda_device)
    keep = (torch.rand(rows, Cin, generator=g) > 0.45).to(cuda_device)
    bits = (keep.view(rows, Cin // 8, 8).to(torch.int32) << torch.arange(8, device=cuda_device, dtype=torch.int32)).sum(-1).to(torch.uint8).contiguous()
    plain = torch.empty(rows, Cin, device=cuda_device, dtype=torch.bfloat16)
    _lib.call("argus_conv2d_dgrad", dy, w, plain, N, H, W, Cin, Cout, 1, 1, res, _lib.stream_ptr())
    slots = ctypes.c_int()
    _lib.check(_lib.load().argus_conv2d_stat_slots(N, H, W, Cout, Cin, 1, 1, 0, ctypes.byref(slots)))
    stats = torch.zeros(slots.value, 2, Cin, device=cuda_device)
    out = torch.empty_like(plain)
    _lib.call("argus_conv2d_dgrad_ex", dy, w, out, N, H, W, Cin, Cout, 1, None, 0, None, res, bits, stats, slots.value,
              _lib.stream_ptr())
    torch.cuda.synchronize()
    want = torch.where(keep, plain, torch.zeros_like(plain))
    assert torch.equal(out, want)
    assert torch.allclose(stats[:, 0].sum(0), out.float().sum(0), rtol=1e-4, atol=1e-2)
    assert torch.allclose(stats[:, 1].sum(0), (out.float() ** 2).sum(0), rtol=1e-4, atol=1e-2)
