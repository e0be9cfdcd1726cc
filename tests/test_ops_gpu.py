"""Strict per-op GPU parity (through the C ABI) of the batch-norm / pooling kernels against torch fp32 autograd on
the same bf16-rounded inputs. Outputs are bf16, so the tolerance is one bf16 rounding (2^-8 relative)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from argus_b200 import _lib

pytestmark = pytest.mark.gpu
BF16_EPS = 2.0 ** -8


def close_bf16(got, want, extra=0.0):
    got, want = got.float(), want.float()
    tol = BF16_EPS * want.abs() + 1e-6 + extra
    bad = (got - want).abs() > tol * 1.01
    assert bad.float().mean().item() < 1e-4, (bad.float().mean().item(), (got - want).abs().max().item())


def bn_train_forward(x, gamma, beta, eps=1e-5):
    mean = x.mean(0)
    var = x.var(0, unbiased=False)
    invstd = (var + eps).rsqrt()
    return (x - mean) * invstd * gamma + beta, mean, var, invstd


@pytest.mark.parametrize("rows,C", [(4096, 64), (1000, 256), (513, 2048)])
def test_bn_finalize_and_apply(cuda_device, rows, C):
    g = torch.Generator().manual_seed(rows + C)
    x = (torch.randn(rows, C, generator=g) * 2 + torch.randn(C, generator=g)).to(cuda_device).bfloat16()
    gamma = (torch.rand(C, generator=g) + 0.5).to(cuda_device)
    beta = torch.randn(C, generator=g).to(cuda_device)
    res = torch.randn(rows, C, generator=g).to(cuda_device).bfloat16()
    xf = x.float()
    partial = torch.zeros(3, 2, C, device=cuda_device)           # three "CTA slots", as the conv epilogue writes them
    bounds = [0, rows // 3, rows // 2, rows]
    for k in range(3):
        partial[k, 0] = xf[bounds[k]:bounds[k + 1]].sum(0)
        partial[k, 1] = (xf[bounds[k]:bounds[k + 1]] ** 2).sum(0)
    rm, rv = torch.zeros(C, device=cuda_device), torch.ones(C, device=cuda_device)
    scale, shift, mean, invstd = (torch.empty(C, device=cuda_device) for _ in range(4))
    lib = _lib.load()
    _lib.check(lib.argus_bn_finalize(_lib.ptr(partial), ctypes.c_int(3), ctypes.c_double(rows), _lib.ptr(gamma), _lib.ptr(beta),
                                     _lib.ptr(rm), _lib.ptr(rv), ctypes.c_float(0.1), ctypes.c_float(1e-5),
                                     _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(mean), _lib.ptr(invstd), ctypes.c_int(C),
                                     _lib.stream_ptr()))
    y_ref, m_ref, v_ref, is_ref = bn_train_forward(xf, gamma, beta)
    assert torch.allclose(mean, m_ref, rtol=1e-4, atol=1e-5)
    assert torch.allclose(invstd, is_ref, rtol=1e-4, atol=1e-5)
    assert torch.allclose(rm, 0.1 * m_ref, rtol=1e-4, atol=1e-5)
    assert torch.allclose(rv, 0.9 + 0.1 * xf.var(0, unbiased=True), rtol=1e-4, atol=1e-5)
    for use_res, relu in ((False, True), (True, True), (False, False)):
        y = torch.empty_like(x)
        _lib.check(lib.argus_bn_apply(_lib.ptr(x), _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(res if use_res else None),
                                      None, None, ctypes.c_int(int(relu)), _lib.ptr(y), ctypes.c_int64(rows),
                                      ctypes.c_int(C), _lib.stream_ptr()))
        want = y_ref + (res.float() if use_res else 0)
        if relu:
            want = want.relu()
        close_bf16(y, want, extra=2e-3 * (1 + xf.abs().max().item()) * 0)
    # residual with its own scale/shift (downsample branch)
    y = torch.empty_like(x)
    _lib.check(lib.argus_bn_apply(_lib.ptr(x), _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(res), _lib.ptr(gamma), _lib.ptr(beta),
                                  ctypes.c_int(1), _lib.ptr(y), ctypes.c_int64(rows), ctypes.c_int(C), _lib.stream_ptr()))
    close_bf16(y, (y_ref + res.float() * gamma + beta).relu())


@pytest.mark.parametrize("rows,C,mask", [(4096, 64, 1), (2048, 256, 0), (777, 512, 2), (4096, 2048, 1), (300, 128, 2)])
def test_bn_backward(cuda_device, rows, C, mask):
    g = torch.Generator().manual_seed(rows * 3 + C + mask)
    x = (torch.randn(rows, C, generator=g) * 1.5 + torch.randn(C, generator=g)).to(cuda_device).bfloat16()
    dy = torch.randn(rows, C, generator=g).to(cuda_device).bfloat16()
    ident = torch.randn(rows, C, generator=g).to(cuda_device).bfloat16()
    gamma = (torch.rand(C, generator=g) + 0.5).to(cuda_device)
    beta = (torch.randn(C, generator=g) * 0.5).to(cuda_device)
    xr = x.float().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    y, mean, var, invstd = bn_train_forward(xr, gr, br)
    scale = (gamma * invstd).detach()
    shift = (beta - mean * gamma * invstd).detach()
    if mask == 0:
        out_t = y
    elif mask == 1:
        # the kernel recomputes the mask as fma(x, scale, shift) > 0: build the reference the same way so that
        # elements within rounding of zero do not flip
        pre = torch.addcmul(shift, x.float(), scale)
        out_t = y * (pre > 0)
    else:
        out_bf16 = (y.detach() + ident.float()).relu().bfloat16()
        out_t = (y + ident.float()) * (out_bf16.float() > 0)
    out_t.backward(dy.float())
    dgamma, dbeta = torch.zeros(C, device=cuda_device), torch.zeros(C, device=cuda_device)
    dx = torch.empty_like(x)
    dy_io = dy.clone()
    out_arg = out_bf16 if mask == 2 else None
    _lib.check(_lib.load().argus_bn_backward(_lib.ptr(dy_io), _lib.ptr(x), _lib.ptr(out_arg), _lib.ptr(scale), _lib.ptr(shift),
                                             _lib.ptr(mean.detach()), _lib.ptr(invstd.detach()), _lib.ptr(dgamma),
                                             _lib.ptr(dbeta), _lib.ptr(dx), ctypes.c_int64(rows), ctypes.c_int(C),
                                             ctypes.c_int(mask), _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.allclose(dbeta, br.grad, rtol=2e-3, atol=2e-3 * rows ** 0.5)
    assert torch.allclose(dgamma, gr.grad, rtol=2e-3, atol=2e-3 * rows ** 0.5)
    rel = ((dx.float() - xr.grad).norm() / xr.grad.norm()).item()
    assert rel < 4e-3, rel
    if mask == 2:
        assert torch.equal(dy_io, (dy.float() * (out_bf16.float() > 0)).bfloat16())
    # deterministic: a second call reproduces the reductions bit for bit
    dgamma2, dbeta2 = torch.zeros_like(dgamma), torch.zeros_like(dbeta)
    dx2 = torch.empty_like(dx)
    dy_io2 = dy.clone()
    _lib.check(_lib.load().argus_bn_backward(_lib.ptr(dy_io2), _lib.ptr(x), _lib.ptr(out_arg), _lib.ptr(scale), _lib.ptr(shift),
                                             _lib.ptr(mean.detach()), _lib.ptr(invstd.detach()), _lib.ptr(dgamma2),
                                             _lib.ptr(dbeta2), _lib.ptr(dx2), ctypes.c_int64(rows), ctypes.c_int(C),
                                             ctypes.c_int(mask), _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(dgamma, dgamma2) and torch.equal(dbeta, dbeta2) and torch.equal(dx, dx2)


def unpack_bits(bits, rows, C):
    """[rows][C/8] bytes -> bool (rows, C): bit k of byte j = channel 8j+k."""
    b = bits.view(rows, C // 8, 1).to(torch.int32)
    return ((b >> torch.arange(8, device=bits.device, dtype=torch.int32)) & 1).bool().view(rows, C)


@pytest.mark.parametrize("rows,C,ds", [(777, 512, False), (300, 128, True), (4096, 256, False)])
def test_bn_relu_bits_forward_backward(cuda_device, rows, C, ds):
    """Residual-block tail with the ReLU mask kept as a bit mask: bn_apply_bits writes it, bn_backward mode 3 reads it
    (and leaves dy alone). Must reproduce mask mode 2 (mask = bf16 output > 0) exactly."""
    g = torch.Generator().manual_seed(rows + C)
    x = (torch.randn(rows, C, generator=g) * 1.5 + torch.randn(C, generator=g)).to(cuda_device).bfloat16()
    ident = torch.randn(rows, C, generator=g).to(cuda_device).bfloat16()
    dy = torch.randn(rows, C, generator=g).to(cuda_device).bfloat16()
    gamma = (torch.rand(C, generator=g) + 0.5).to(cuda_device)
    beta = (torch.randn(C, generator=g) * 0.5).to(cuda_device)
    _, mean, var, invstd = bn_train_forward(x.float(), gamma, beta)
    scale, shift = gamma * invstd, beta - mean * gamma * invstd
    rs = (torch.rand(C, generator=g) + 0.5).to(cuda_device) if ds else None
    rb = torch.randn(C, generator=g).to(cuda_device) if ds else None
    lib = _lib.load()
    y = torch.empty_like(x)
    y_plain = torch.empty_like(x)
    bits = torch.zeros(rows, C // 8, device=cuda_device, dtype=torch.uint8)
    _lib.check(lib.argus_bn_apply_bits(_lib.ptr(x), _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(ident), _lib.ptr(rs), _lib.ptr(rb),
                                       ctypes.c_int(1), _lib.ptr(y), _lib.ptr(bits), ctypes.c_int64(rows), ctypes.c_int(C),
                                       _lib.stream_ptr()))
    _lib.check(lib.argus_bn_apply(_lib.ptr(x), _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(ident), _lib.ptr(rs), _lib.ptr(rb),
                                  ctypes.c_int(1), _lib.ptr(y_plain), ctypes.c_int64(rows), ctypes.c_int(C), _lib.stream_ptr()))
    assert torch.equal(y, y_plain)
    assert torch.equal(unpack_bits(bits, rows, C), y.float() > 0)

    def backward(mask_mode, out_arg):
        dgamma, dbeta = torch.zeros(C, device=cuda_device), torch.zeros(C, device=cuda_device)
        dx = torch.empty_like(x)
        dy_io = dy.clone()
        _lib.check(lib.argus_bn_backward(_lib.ptr(dy_io), _lib.ptr(x), _lib.ptr(out_arg), _lib.ptr(scale), _lib.ptr(shift),
                                         _lib.ptr(mean), _lib.ptr(invstd), _lib.ptr(dgamma), _lib.ptr(dbeta), _lib.ptr(dx),
                                         ctypes.c_int64(rows), ctypes.c_int(C), ctypes.c_int(mask_mode), _lib.stream_ptr()))
        return dgamma, dbeta, dx, dy_io

    g2, b2, dx2, dy2 = backward(2, y)
    g3, b3, dx3, dy3 = backward(3, bits)
    assert torch.equal(g2, g3) and torch.equal(b2, b3) and torch.equal(dx2, dx3)
    assert torch.equal(dy3, dy)                                              # mode 3 does not touch dy
    assert torch.equal(dy2, (dy.float() * (y.float() > 0)).bfloat16())       # mode 2 masks it in place


def misaligned_copy(t):
    """t's contents in a larger allocation, one element (2 bytes of bf16, 1 byte of a bit mask) past a 16-byte boundary:
    valid device memory that is not 16-byte aligned."""
    big = torch.empty(t.numel() + 16, dtype=t.dtype, device=t.device)
    v = big[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0
    return v


@pytest.mark.parametrize("op", ["apply", "apply_bits", "backward0", "backward1", "backward2", "backward3"])
def test_bn_passes_reject_misaligned_tensors(cuda_device, op):
    """The batch-norm passes stream every tensor with 16-byte vectors and bulk copies. A tensor that is not 16-byte
    aligned is rejected on the host before anything runs: the call fails, and the outputs and the dgamma / dbeta
    accumulators keep their sentinel values. For the backward this includes dx, which only its second pass uses."""
    rows, C = 1000, 64
    g = torch.Generator().manual_seed(11)
    x, dy, res, blk_out = (torch.randn(rows, C, generator=g).to(cuda_device).bfloat16() for _ in range(4))
    bits = torch.randint(0, 256, (rows, C // 8), generator=g, dtype=torch.uint8).to(cuda_device)
    scale, invstd = ((torch.rand(C, generator=g) + 0.5).to(cuda_device) for _ in range(2))
    shift, mean = (torch.randn(C, generator=g).to(cuda_device) for _ in range(2))
    dgamma, dbeta = torch.full((C,), 7.0, device=cuda_device), torch.full((C,), 7.0, device=cuda_device)
    lib = _lib.load()
    P = _lib.ptr
    if op.startswith("apply"):
        with_bits = op == "apply_bits"
        tensors = {"x": x, "res": res, "y": torch.full_like(x, 3.0)}
        if with_bits:
            tensors["bits"] = torch.full((rows, C // 8), 0xA5, dtype=torch.uint8, device=cuda_device)

        def run(t):
            if with_bits:
                return lib.argus_bn_apply_bits(P(t["x"]), P(scale), P(shift), P(t["res"]), None, None, ctypes.c_int(1),
                                               P(t["y"]), P(t["bits"]), ctypes.c_int64(rows), ctypes.c_int(C),
                                               _lib.stream_ptr())
            return lib.argus_bn_apply(P(t["x"]), P(scale), P(shift), P(t["res"]), None, None, ctypes.c_int(1), P(t["y"]),
                                      ctypes.c_int64(rows), ctypes.c_int(C), _lib.stream_ptr())
    else:
        mask = int(op[-1])
        tensors = {"dy": dy, "x": x, "dx": torch.full_like(x, 3.0)}
        if mask in (2, 3):
            tensors["out"] = blk_out if mask == 2 else bits

        def run(t):
            return lib.argus_bn_backward(P(t["dy"]), P(t["x"]), P(t.get("out")), P(scale), P(shift), P(mean), P(invstd),
                                         P(dgamma), P(dbeta), P(t["dx"]), ctypes.c_int64(rows), ctypes.c_int(C),
                                         ctypes.c_int(mask), _lib.stream_ptr())

    for name in tensors:
        t = dict(tensors, **{name: misaligned_copy(tensors[name])})
        before = {k: v.clone() for k, v in t.items()}
        status = run(t)
        assert status != 0, name
        assert "16-byte aligned" in lib.argus_last_error_string().decode(), name
        torch.cuda.synchronize()
        for k, v in t.items():
            assert torch.equal(v, before[k]), (name, k)
        assert torch.all(dgamma == 7.0) and torch.all(dbeta == 7.0), name
    # the same call with every tensor aligned runs
    assert run(tensors) == 0, lib.argus_last_error_string()
    torch.cuda.synchronize()
    if op.startswith("apply"):
        assert not torch.all(tensors["y"] == 3.0)
    else:
        assert not torch.all(dbeta == 7.0)


@pytest.mark.parametrize("N,H,W,Cin,Cout", [(2, 16, 16, 256, 64), (1, 8, 8, 512, 128), (3, 8, 16, 64, 64)])
def test_dgrad_residual_bits(cuda_device, N, H, W, Cin, Cout):
    """1x1 dgrad whose residual is gated by the bit mask == dgrad with the pre-masked residual, bit for bit."""
    g = torch.Generator().manual_seed(N * H + Cin)
    rows = N * H * W
    dyt = torch.randn(rows, Cout, generator=g).to(cuda_device).bfloat16()
    w = (torch.randn(Cout, Cin, generator=g) / Cout ** 0.5).to(cuda_device).bfloat16()
    res = torch.randn(rows, Cin, generator=g).to(cuda_device).bfloat16()
    keep = torch.rand(rows, Cin, generator=g).to(cuda_device) > 0.4
    k8 = keep.view(rows, Cin // 8, 8).to(torch.int32)
    bits = (k8 << torch.arange(8, device=cuda_device, dtype=torch.int32)).sum(-1).to(torch.uint8).contiguous()
    masked = (res.float() * keep).bfloat16()
    dx_a = torch.empty(rows, Cin, device=cuda_device, dtype=torch.bfloat16)
    dx_b = torch.empty_like(dx_a)
    _lib.call("argus_conv2d_dgrad", dyt, w, dx_a, N, H, W, Cin, Cout, 1, 1, masked, _lib.stream_ptr())
    _lib.call("argus_conv2d_dgrad_bits", dyt, w, dx_b, N, H, W, Cin, Cout, 1, res, bits, _lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(dx_a, dx_b)
    want = dyt.float() @ w.float() + masked.float()
    close_bf16(dx_b, want, extra=2e-2)


@pytest.mark.parametrize("N,H,W,C", [(2, 16, 16, 64), (3, 64, 32, 64), (1, 8, 8, 128)])
def test_maxpool(cuda_device, N, H, W, C):
    g = torch.Generator().manual_seed(N + H)
    x = torch.randn(N, H, W, C, generator=g).to(cuda_device).bfloat16()
    scale = (torch.rand(C, generator=g) + 0.5).to(cuda_device)
    shift = torch.randn(C, generator=g).to(cuda_device)
    y = torch.empty(N, H // 2, W // 2, C, device=cuda_device, dtype=torch.bfloat16)
    idx = torch.empty(N, H // 2, W // 2, C, device=cuda_device, dtype=torch.uint8)
    _lib.call("argus_maxpool_forward", x, scale, shift, y, idx, N, H, W, C, _lib.stream_ptr())
    act = torch.addcmul(shift, x.float(), scale).relu().permute(0, 3, 1, 2).requires_grad_(True)
    ref = F.max_pool2d(act, 3, 2, 1)
    close_bf16(y, ref.permute(0, 2, 3, 1))
    dy = torch.randn(N, H // 2, W // 2, C, generator=g).to(cuda_device).bfloat16()
    dx = torch.empty(N, H, W, C, device=cuda_device, dtype=torch.bfloat16)
    _lib.call("argus_maxpool_backward", dy, idx, dx, N, H, W, C, _lib.stream_ptr())
    ref.backward(dy.float().permute(0, 3, 1, 2))
    # Ties among equal maxima may route the gradient to a different (equally valid) tap. The kernel takes the arg-max on
    # the raw values (relu(bn(x)) is monotone in x), so a window that is entirely <= 0 after the ReLU -- every tap ties at
    # 0 -- may pick another tap than torch's "first maximum"; the ReLU backward that always follows zeroes both. Where the
    # activation is positive the routing must agree (up to exact ties between positive bf16 values).
    want = act.grad.permute(0, 2, 3, 1)
    live = (act.detach() > 0).permute(0, 2, 3, 1).float()
    mism = (((dx.float() - want) * live).abs() > BF16_EPS * want.abs() * 2 + 1e-6).float().mean().item()
    assert mism < 0.004, mism
    assert torch.allclose(dx.float().sum((1, 2)), want.sum((1, 2)), rtol=2e-2, atol=0.5)
    # already-activated input (inference path)
    y2 = torch.empty_like(y)
    _lib.call("argus_maxpool_forward", act.detach().permute(0, 2, 3, 1).contiguous().bfloat16(), None, None, y2, None, N,
              H, W, C, _lib.stream_ptr())
    close_bf16(y2, F.max_pool2d(act.detach().bfloat16().float(), 3, 2, 1).permute(0, 2, 3, 1))


@pytest.mark.parametrize("N,H,W", [(2, 16, 16), (3, 64, 32), (1, 8, 128)])
def test_stem_pool_bn_backward_fused(cuda_device, N, H, W):
    """max-pool backward + ReLU mask + BN backward in two fused passes == the unfused composition (which rounds the
    un-pooled gradient to bf16 in between) within one bf16 rounding, and == torch autograd."""
    C = 64
    g = torch.Generator().manual_seed(N + H + W)
    raw = (torch.randn(N, H, W, C, generator=g) * 1.5 + torch.randn(C, generator=g)).to(cuda_device).bfloat16()
    gamma = (torch.rand(C, generator=g) + 0.5).to(cuda_device)
    beta = (torch.randn(C, generator=g) * 0.5).to(cuda_device)
    rows = N * H * W
    xr = raw.float().view(rows, C).requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    y, mean, var, invstd = bn_train_forward(xr, gr, br)
    scale, shift = (gamma * invstd).detach(), (beta - mean * gamma * invstd).detach()
    pooled = torch.empty(N, H // 2, W // 2, C, device=cuda_device, dtype=torch.bfloat16)
    idx = torch.empty(N, H // 2, W // 2, C, device=cuda_device, dtype=torch.uint8)
    _lib.call("argus_maxpool_forward", raw, scale, shift, pooled, idx, N, H, W, C, _lib.stream_ptr())
    dpool = torch.randn(N, H // 2, W // 2, C, generator=g).to(cuda_device).bfloat16()
    # unfused composition
    dact = torch.empty_like(raw)
    _lib.call("argus_maxpool_backward", dpool, idx, dact, N, H, W, C, _lib.stream_ptr())
    dg_a, db_a = torch.zeros(C, device=cuda_device), torch.zeros(C, device=cuda_device)
    dx_a = torch.empty_like(raw)
    lib = _lib.load()
    _lib.check(lib.argus_bn_backward(_lib.ptr(dact), _lib.ptr(raw), None, _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(mean.detach()),
                                     _lib.ptr(invstd.detach()), _lib.ptr(dg_a), _lib.ptr(db_a), _lib.ptr(dx_a),
                                     ctypes.c_int64(rows), ctypes.c_int(C), ctypes.c_int(1), _lib.stream_ptr()))
    # fused
    dg_b, db_b = torch.zeros(C, device=cuda_device), torch.zeros(C, device=cuda_device)
    dx_b = torch.empty_like(raw)
    _lib.check(lib.argus_stem_pool_bn_backward(_lib.ptr(dpool), _lib.ptr(idx), _lib.ptr(raw), _lib.ptr(scale), _lib.ptr(shift),
                                               _lib.ptr(mean.detach()), _lib.ptr(invstd.detach()), _lib.ptr(dg_b), _lib.ptr(db_b),
                                               _lib.ptr(dx_b), ctypes.c_int(N), ctypes.c_int(H), ctypes.c_int(W), ctypes.c_int(C),
                                               _lib.stream_ptr()))
    torch.cuda.synchronize()
    # torch reference: the un-pooled gradient routed by OUR arg-max bytes (ties are equally valid), then autograd
    ii = idx.long()
    dact_ref = torch.zeros(N, H, W, C, device=cuda_device)
    ph, pw = torch.meshgrid(torch.arange(H // 2, device=cuda_device), torch.arange(W // 2, device=cuda_device), indexing="ij")
    hh = (2 * ph - 1)[None, :, :, None] + ii // 3
    ww = (2 * pw - 1)[None, :, :, None] + ii % 3
    nn_ = torch.arange(N, device=cuda_device)[:, None, None, None].expand_as(ii)
    cc = torch.arange(C, device=cuda_device)[None, None, None, :].expand_as(ii)
    dact_ref.index_put_((nn_, hh, ww, cc), dpool.float(), accumulate=True)
    pre = torch.addcmul(shift, raw.float().view(rows, C), scale)
    (y * (pre > 0)).backward(dact_ref.view(rows, C))
    assert torch.allclose(db_b, br.grad, rtol=2e-3, atol=2e-3 * rows ** 0.5)
    assert torch.allclose(dg_b, gr.grad, rtol=2e-3, atol=2e-3 * rows ** 0.5)
    assert rel_err(dx_b.float().view(rows, C), xr.grad) < 4e-3
    assert rel_err(dx_b.float(), dx_a.float()) < 6e-3      # the unfused path rounds the un-pooled gradient to bf16
    # deterministic
    dg_c, db_c, dx_c = torch.zeros_like(dg_b), torch.zeros_like(db_b), torch.empty_like(dx_b)
    _lib.check(lib.argus_stem_pool_bn_backward(_lib.ptr(dpool), _lib.ptr(idx), _lib.ptr(raw), _lib.ptr(scale), _lib.ptr(shift),
                                               _lib.ptr(mean.detach()), _lib.ptr(invstd.detach()), _lib.ptr(dg_c), _lib.ptr(db_c),
                                               _lib.ptr(dx_c), ctypes.c_int(N), ctypes.c_int(H), ctypes.c_int(W), ctypes.c_int(C),
                                               _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(dg_b, dg_c) and torch.equal(db_b, db_c) and torch.equal(dx_b, dx_c)


def rel_err(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


def test_avgpool(cuda_device):
    N, HW, C = 6, 64, 2048
    x = torch.randn(N, HW, C, device=cuda_device).bfloat16()
    y = torch.empty(N, C, device=cuda_device, dtype=torch.bfloat16)
    _lib.call("argus_avgpool_forward", x, y, N, HW, C, _lib.stream_ptr())
    close_bf16(y, x.float().mean(1))
    dy = torch.randn(N, C, device=cuda_device).bfloat16()
    dx = torch.empty_like(x)
    _lib.call("argus_avgpool_backward", dy, dx, N, HW, C, _lib.stream_ptr())
    close_bf16(dx, (dy.float() / HW)[:, None, :].expand(N, HW, C))
