"""Per-op parity (through the C ABI) of the primitives behind the algebraic batch-norm backward (csrc/bn_algebra.cu):
the K-concatenated / masked / statistics-producing dgrad and the whole conv(1x1) + BN backward against float64 autograd
of the textbook formulation on the same bf16 inputs. The stacked weight-gradient + Gram launch is checked element by
element in test_wgrad_gpu.py."""
import ctypes

import pytest
import torch

from argus_b200 import _lib
from gpu_util import rel

pytestmark = pytest.mark.gpu


def bf(t):
    return t.bfloat16()


@pytest.mark.parametrize("N,H,W,C,O,stride", [(4, 16, 16, 64, 256, 1), (2, 16, 16, 128, 512, 1), (2, 16, 16, 256, 512, 2),
                                              (3, 8, 8, 256, 1024, 1), (20, 32, 32, 64, 256, 1)])
def test_conv_bn_backward_algebraic(cuda_device, N, H, W, C, O, stride):
    g = torch.Generator().manual_seed(N * H + C + O + stride)
    act = bf((torch.randn(N, H, W, C, generator=g) * 1.3).relu()).to(cuda_device)
    w = bf(torch.randn(O, C, generator=g) / C ** 0.5).to(cuda_device)
    gamma = (torch.rand(O, generator=g) + 0.5).to(cuda_device)
    Ho, Wo = H // stride, W // stride
    rows = N * Ho * Wo
    act_s = act[:, ::stride, ::stride, :].reshape(rows, C)
    raw = bf(act_s.float() @ w.float().t())                      # what the forward stored (bf16)
    mean = raw.float().mean(0)
    var = raw.float().var(0, unbiased=False)
    invstd = (var + 1e-5).rsqrt()
    scale = gamma * invstd
    up = bf(torch.randn(rows, O, generator=g).to(cuda_device) * 0.01 * (torch.rand(rows, O, generator=g).to(cuda_device) > 0.5) + 0.003)
    # float64 truth of the textbook BN backward on the stored raw, then the two conv gradients
    r64, u64, a64, w64 = raw.double(), up.double(), act_s.double(), w.double()
    xh = (r64 - mean.double()) * invstd.double()
    dbeta = u64.sum(0)
    dgamma = (u64 * xh).sum(0)
    q = scale.double() * (u64 - dbeta / rows - xh * dgamma / rows)
    dact_s = q @ w64
    dw_true = q.t() @ a64
    dact_true = torch.zeros(N, H, W, C, dtype=torch.float64, device=cuda_device)
    dact_true[:, ::stride, ::stride, :] = dact_s.view(N, Ho, Wo, C)

    dg, db = torch.zeros(O, device=cuda_device), torch.zeros(O, device=cuda_device)
    dw = torch.zeros(O, C, device=cuda_device)
    dact = torch.full((N, H, W, C), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    colsum = up.float().sum(0).contiguous()

    def run(dg, db, dw, dact):
        _lib.call("argus_conv_bn_backward_algebraic", up, act, w, colsum, scale.contiguous(), mean.contiguous(),
                  invstd.contiguous(), dg, db, dw, dact, N, H, W, C, O, stride, _lib.stream_ptr())

    run(dg, db, dw, dact)
    torch.cuda.synchronize()
    print(f"\n[{N}x{H}x{W} C={C} O={O} s={stride}] dact {rel(dact, dact_true):.2e} dw {rel(dw, dw_true):.2e} "
          f"dgamma {rel(dg, dgamma):.2e} dbeta {rel(db, dbeta):.2e}")
    assert rel(db, dbeta) < 1e-5
    assert rel(dg, dgamma) < 1e-2           # sum g*raw is rebuilt from the unrounded raw = act W^T
    assert rel(dw, dw_true) < 3e-3
    assert rel(dact, dact_true) < 6e-3      # bf16 output + bf16 stacked operand
    # deterministic
    dg2, db2, dw2 = torch.zeros_like(dg), torch.zeros_like(db), torch.zeros_like(dw)
    dact2 = torch.empty_like(dact)
    run(dg2, db2, dw2, dact2)
    torch.cuda.synchronize()
    assert torch.equal(dg, dg2) and torch.equal(dw, dw2) and torch.equal(dact, dact2)


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
