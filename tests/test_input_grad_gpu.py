"""Gradients with respect to the input images: the stem's transposed convolution (argus_stem_dgrad, tcgen05) against
float64 torch, and x.grad of the whole network in both precisions against the fp32 / float64 reference."""
import pytest
import torch
import torch.nn.functional as F

from argus_b200 import _lib
from gpu_util import random_targets, rel, structured_images

pytestmark = pytest.mark.gpu


def stem_pack_w(w):
    """[64,3,7,7] -> [64][p 4][q 4][16] bf16 with kh = 2p + a - 1, kw = 2q + b - 1 (the forward's kind-1 layout)."""
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


def stem_dgrad(dy_nhwc, w_packed, N, H, W):
    dx = torch.full((N, 3, H, W), float("nan"), device=dy_nhwc.device)
    _lib.call("argus_stem_dgrad", dy_nhwc, w_packed, dx, N, H, W, _lib.stream_ptr())
    torch.cuda.synchronize()
    return dx


@pytest.mark.parametrize("N,H,W", [(1, 32, 32), (2, 64, 64), (2, 64, 128), (5, 128, 64), (3, 256, 256), (64, 128, 128)])
def test_stem_dgrad_primitive(cuda_device, N, H, W):
    g = torch.Generator().manual_seed(7)
    w = (torch.randn(64, 3, 7, 7, generator=g) / 147 ** 0.5).to(cuda_device).to(torch.bfloat16)
    dy = torch.randn(N, H // 2, W // 2, 64, generator=g).to(cuda_device).to(torch.bfloat16)
    wp = stem_pack_w(w.float())

    def truth(dyb):
        return F.conv_transpose2d(dyb.double().permute(0, 3, 1, 2), w.double(), stride=2, padding=3, output_padding=1)

    dx = stem_dgrad(dy, wp, N, H, W)
    want = truth(dy)
    r = rel(dx, want)
    print(f"stem dgrad N={N} {H}x{W}: rel err {r:.2e}")
    assert torch.isfinite(dx).all()
    assert r < 1e-4
    # bitwise reproducible
    assert torch.equal(dx, stem_dgrad(dy, wp, N, H, W))
    # borders: dy only near the edges of the dY grid, compared on the outer 4-pixel frame of dx
    keep = torch.zeros(H // 2, W // 2, dtype=torch.bool, device=cuda_device)
    keep[:3], keep[-3:], keep[:, :3], keep[:, -3:] = True, True, True, True
    dyb = dy * keep[None, :, :, None]
    frame = torch.ones(H, W, dtype=torch.bool, device=cuda_device)
    frame[4:-4, 4:-4] = False
    dx_b, want_b = stem_dgrad(dyb, wp, N, H, W), truth(dyb)
    r_b = rel(dx_b[..., frame], want_b[..., frame])
    print(f"   border frame rel err {r_b:.2e}")
    assert r_b < 1e-4


def build_pair(device, residual_gain=None, n_cams=2, precision="bf16", seed=42):
    from argus_b200.models import NCameraCNN, NCameraCNNConfig
    from oracle.ref_model import make_reference_model

    ref = make_reference_model(seed, n_cams=n_cams).to(device)
    if residual_gain is not None:
        # conditioned residual branches, as in test_model_gpu.py::build_pair
        with torch.no_grad():
            for m in ref.modules():
                if hasattr(m, "bn3"):
                    m.bn3.weight.fill_(residual_gain)
    ours = NCameraCNN(NCameraCNNConfig(n_cams=n_cams)).to(device).set_precision(precision)
    ours.load_state_dict(ref.state_dict(), strict=True)
    ref.train(); ours.train()
    return ref, ours


def ours_input_grad(model, x, target):
    from argus_b200.loss import geometric_loss_fn

    xg = x.clone().requires_grad_(True)
    loss = geometric_loss_fn(model(xg), target).mean()
    loss.backward()
    torch.cuda.synchronize()
    return xg.grad, loss.detach()


def ref_input_grad(ref, x, target, autocast=False):
    from oracle.ref_model import torch_loss

    xg = x.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        y = ref(xg)
    torch_loss(y.float() if autocast else y, target).mean().backward()
    return xg.grad


@pytest.mark.parametrize("B,H,W,gain,n_cams", [(8, 128, 128, 0.1, 2), (4, 256, 256, 0.2, 2), (8, 128, 128, None, 2),
                                               (8, 128, 128, 0.2, 1), (8, 128, 128, 0.2, 3), (8, 128, 256, 0.2, 2)])
def test_model_input_grad_bf16(cuda_device, B, H, W, gain, n_cams):
    """x.grad of the mean pose loss against the fp32 reference, with torch's bf16 autocast of the same reference as the
    yardstick for what bf16 storage costs (overall and per view)."""
    ref, ours = build_pair(cuda_device, gain, n_cams)
    x = structured_images(B, 3 * n_cams, H, W, 3, cuda_device)
    target = random_targets(B, 4, cuda_device)
    g_ref = ref_input_grad(ref, x, target)
    g_ac = ref_input_grad(ref, x, target, autocast=True)
    g, _ = ours_input_grad(ours, x, target)
    assert g.shape == x.shape and g.dtype == torch.float32
    cos = F.cosine_similarity(g.flatten().double(), g_ref.flatten().double(), dim=0).item()
    r, r_ac = rel(g, g_ref), rel(g_ac, g_ref)
    print(f"\n[B={B} {H}x{W} gain={gain} n_cams={n_cams}] x.grad rel err: ours {r:.3e} autocast {r_ac:.3e}; cosine {cos:.6f}")
    assert r < max(1.25 * r_ac, 2e-2)
    for v in range(n_cams):
        sl = slice(3 * v, 3 * v + 3)
        rv, rv_ac = rel(g[:, sl], g_ref[:, sl]), rel(g_ac[:, sl], g_ref[:, sl])
        print(f"   view {v}: ours {rv:.3e} autocast {rv_ac:.3e}")
        assert rv < max(1.25 * rv_ac, 2e-2)


@pytest.fixture
def no_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("B,H,W,gain", [(8, 256, 256, 0.2), (8, 256, 256, None), (4, 128, 128, 0.2), (2, 64, 64, None)])
def test_model_input_grad_fp32(cuda_device, no_tf32, B, H, W, gain):
    """fp32 parity mode: x.grad against the float64 truth, as close as the reference's own fp32 x.grad (the cases of
    test_fp32_mode_gpu.py::test_fp32_train_forward_backward)."""
    ref, ours = build_pair(cuda_device, gain, precision="fp32")
    x = structured_images(B, 6, H, W, 3, cuda_device)
    target = random_targets(B, 4, cuda_device)
    state0 = {k: v.clone() for k, v in ref.state_dict().items()}
    g_ref32 = ref_input_grad(ref, x, target)
    ref.load_state_dict(state0)
    g64 = ref_input_grad(ref.double(), x.double(), target)
    g, _ = ours_input_grad(ours, x, target)
    r, r_ref = rel(g, g64), rel(g_ref32, g64)
    print(f"\n[fp32 B={B} {H}x{W} gain={gain}] x.grad vs fp64 truth: ours {r:.3e} reference-fp32 {r_ref:.3e}")
    assert r <= max(2.0 * r_ref, 1e-4)


def test_input_grad_surface(cuda_device):
    from argus_b200.loss import geometric_loss_fn

    B, H, W = 4, 64, 64
    x = structured_images(B, 6, H, W, 3, cuda_device)
    target = random_targets(B, 4, cuda_device)

    # torch.autograd.grad with respect to the input
    _, ours = build_pair(cuda_device, 0.2)
    xg = x.clone().requires_grad_(True)
    (gx,) = torch.autograd.grad(geometric_loss_fn(ours(xg), target).mean(), xg)
    assert gx.shape == x.shape and torch.isfinite(gx).all() and gx.abs().sum() > 0

    # parameter gradients and loss do not depend on whether x requires grad
    _, a = build_pair(cuda_device, 0.2)
    loss_a = geometric_loss_fn(a(x), target).mean()
    loss_a.backward()
    _, b = build_pair(cuda_device, 0.2)
    g_b, loss_b = ours_input_grad(b, x, target)
    assert torch.equal(loss_a.detach(), loss_b)
    for (n, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        assert torch.equal(pa.grad, pb.grad), n

    # two fresh models: bitwise equal x.grad
    _, c = build_pair(cuda_device, 0.2)
    g_c, _ = ours_input_grad(c, x, target)
    assert torch.equal(g_b, g_c)

    # frozen weights: the node still runs, x.grad has the same bits, no parameter receives a gradient
    _, d = build_pair(cuda_device, 0.2)
    d.requires_grad_(False)
    g_d, _ = ours_input_grad(d, x, target)
    assert torch.equal(g_d, g_b)
    assert all(p.grad is None for p in d.parameters())

    # float64 / bf16 inputs get gradients of their own dtype
    for dt in (torch.float64, torch.bfloat16):
        xd = x.to(dt).requires_grad_(True)
        geometric_loss_fn(b(xd), target).mean().backward()
        assert xd.grad is not None and xd.grad.dtype == dt and torch.isfinite(xd.grad.float()).all()


def test_input_grad_fp32_mode_deterministic(cuda_device):
    B, H, W = 2, 64, 64
    x = structured_images(B, 6, H, W, 3, cuda_device)
    target = random_targets(B, 4, cuda_device)
    g1, _ = ours_input_grad(build_pair(cuda_device, 0.2, precision="fp32")[1], x, target)
    g2, _ = ours_input_grad(build_pair(cuda_device, 0.2, precision="fp32")[1], x, target)
    assert torch.equal(g1, g2)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_input_grad_errors(cuda_device, precision):
    from argus_b200.models import NCameraCNN

    B, H, W = 2, 64, 64
    m = NCameraCNN().to(cuda_device).set_precision(precision).train()
    dx = torch.empty(B, 6, H, W, device=cuda_device)
    with pytest.raises(_lib.ArgusError, match="training forward"):
        _lib.call("argus_model_input_grad", m._handle.ptr, dx, _lib.stream_ptr())
    x = structured_images(B, 6, H, W, 3, cuda_device)
    with torch.no_grad():
        out = m(x)
    with pytest.raises(_lib.ArgusError, match="stage 3"):
        _lib.call("argus_model_input_grad", m._handle.ptr, dx, _lib.stream_ptr())
    # a training step on uint8 images (B, n_cams, H, W, 3): no input gradient exists
    u8 = (x * 255).to(torch.uint8).reshape(B, 2, 3, H, W).permute(0, 1, 3, 4, 2).contiguous()
    out = m._forward_impl(u8, True)
    m._backward_impl(torch.ones_like(out))
    with pytest.raises(_lib.ArgusError, match="uint8"):
        _lib.call("argus_model_input_grad", m._handle.ptr, dx, _lib.stream_ptr())
    # the same step on the fp32 images does have one
    out = m._forward_impl(x, True)
    m._backward_impl(torch.ones_like(out))
    _lib.call("argus_model_input_grad", m._handle.ptr, dx, _lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.isfinite(dx).all()
