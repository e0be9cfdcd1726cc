"""Fine-tuning with frozen batch-norm statistics in the fused engine: TrainEngine(frozen_bn=True) runs the
frozen-statistics forward (argus_model_forward_frozen) and its backward inside the training step -- float, uint8 with
the fused augmentation, and batches staged ahead with prefetch() (argus_model_stage_input_frozen_u8) -- under the
same loss, bucketed all-reduce and optimizer as a training step. Checked bitwise against the autograd path of an
eval-mode module, against itself with and without look-ahead and loss scaling, and under two-rank NCCL."""
import os

import pytest
import torch

from argus_b200 import _lib
from gpu_util import random_targets, rel, structured_images
from test_frozen_bn_gpu import build_frozen_pair

pytestmark = pytest.mark.gpu


def clone_model(m):
    from argus_b200.models import NCameraCNN, NCameraCNNConfig

    c = NCameraCNN(NCameraCNNConfig(n_cams=m.n_cams)).to(m.flat_params.device).set_precision(m.precision)
    c.load_state_dict(m.state_dict(), strict=True)
    return c.eval()


def bn_state(m):
    return {k: v.clone() for k, v in m.state_dict().items() if "running" in k or "num_batches" in k}


def assert_bn_state_equal(m, want):
    got = bn_state(m)
    assert got.keys() == want.keys()
    for k in want:
        assert torch.equal(got[k], want[k]), k


def autograd_flat_grads(m, x, t):
    """geometric_loss_fn(model.eval()(x), t).mean().backward(), gathered into the flat arena's layout."""
    from argus_b200.loss import geometric_loss_fn

    m.eval()
    m.zero_grad(set_to_none=True)
    loss = geometric_loss_fn(m(x), t).mean()
    loss.backward()
    g = torch.zeros_like(m.flat_params)
    for p, (_n, off, numel, _shape) in zip(m.parameters(), m._param_infos):
        g[off:off + numel] = p.grad.reshape(-1)
    return loss.detach(), g


def engine(m, **kw):
    from argus_b200.engine import TrainEngine

    kw.setdefault("lr", 1e-4)
    return TrainEngine(m, max_grad_norm=1.0, distributed=False, frozen_bn=True, **kw)


# ------------------------------------------------------------------------------------------------------------------
# 1. gradients: the autograd path of the eval-mode module, and bitwise repeats
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_gradients_equal_autograd_path(cuda_device, precision):
    _, a = build_frozen_pair(cuda_device, precision=precision)
    b = clone_model(a)
    x = structured_images(8, 6, 128, 128, 9, cuda_device)
    t = random_targets(8, 10, cuda_device)
    bn0 = bn_state(a)
    eng = engine(a)
    loss_a = eng.forward_backward(x, t)
    ga = a.flat_grads.clone()
    loss_a2 = eng.forward_backward(x, t)
    ga2 = a.flat_grads.clone()
    assert torch.equal(ga, ga2) and loss_a.item() == loss_a2.item()
    assert not a.training                                   # the engine leaves the module's mode alone
    assert_bn_state_equal(a, bn0)
    loss_b, gb = autograd_flat_grads(b, x, t)
    r = rel(ga, gb)
    print(f"[{precision}] frozen engine vs autograd path: {r:.3e}")
    assert abs(loss_a.item() - loss_b.item()) <= 1e-5 * abs(loss_b.item())
    assert r < 1e-6, r


# ------------------------------------------------------------------------------------------------------------------
# 2. trajectory: optimizer, fold and scaled-pack refresh; 5. loss scaling
# ------------------------------------------------------------------------------------------------------------------
def batches_f32(n, B, H, seed, device):
    return [(structured_images(B, 6, H, H, seed + i, device), random_targets(B, seed + 50 + i, device)) for i in range(n)]


def test_trajectory_equals_autograd_oracle(cuda_device):
    _, a = build_frozen_pair(cuda_device)
    b = clone_model(a)
    bn0 = bn_state(a)
    data = batches_f32(4, 8, 128, 60, cuda_device)
    eng_a, eng_b = engine(a), engine(b)
    for i in range(3):
        x, t = data[i]
        eng_a.step(x, t)
        # oracle: autograd gradients of the eval-mode module, then the same optimizer step
        _, g = autograd_flat_grads(b, x, t)
        b.flat_grads.copy_(g)
        eng_b.optimizer_step()
        torch.cuda.synchronize()
        assert torch.equal(a.flat_params, b.flat_params), i
        assert_bn_state_equal(a, bn0)
        # the next frozen forward sees the updated weights: bitwise a no-grad eval forward, of this model and of a fresh
        # one built from its state (whose eval fold and packed weights were never stale)
        xn = data[i + 1][0]
        y_frozen = a._forward_impl(xn, False, frozen=True)
        with torch.no_grad():
            y_eval = a(xn)
            y_fresh = clone_model(a)(xn)
        assert torch.equal(y_frozen.view(torch.int32), y_eval.view(torch.int32)), i
        assert torch.equal(y_frozen.view(torch.int32), y_fresh.view(torch.int32)), i
    # the backward runs against diag(scale) W packed from the updated weights: the same gradients as a fresh model's
    x, t = data[3]
    eng_a.forward_backward(x, t)
    ga = a.flat_grads.clone()
    c = clone_model(a)
    engine(c).forward_backward(x, t)
    assert torch.equal(ga, c.flat_grads)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_loss_scaling_is_exact(cuda_device, precision):
    from argus_b200.engine import GradScaler

    _, a = build_frozen_pair(cuda_device, precision=precision)
    b = clone_model(a)
    data = batches_f32(3, 8, 128, 70, cuda_device)
    eng_a, eng_b = engine(a), engine(b, scaler=GradScaler())
    la = [eng_a.step(x, t).clone() for x, t in data]
    lb = [eng_b.step(x, t).clone() for x, t in data]
    torch.cuda.synchronize()
    assert eng_b.scaler.get_scale() == 2.0 ** 16 and eng_b.scaler.skipped_steps == 0
    assert torch.equal(torch.stack(la), torch.stack(lb))
    assert torch.equal(a.flat_params, b.flat_params)


# ------------------------------------------------------------------------------------------------------------------
# 3. look-ahead staging
# ------------------------------------------------------------------------------------------------------------------
def u8_batches(sizes, H, seed, device):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randint(0, 256, (b, 2, H, H, 3), dtype=torch.uint8, generator=g).to(device),
             random_targets(b, seed + i, device)) for i, b in enumerate(sizes)]


def test_prefetch_is_bitwise_equivalent(cuda_device):
    from argus_b200.data import Augmentation, AugmentationConfig

    _, base = build_frozen_pair(cuda_device)
    bn0 = bn_state(base)
    batches = u8_batches([16, 16, 5, 16, 3], 64, 11, cuda_device)

    def run(prefetch):
        m = clone_model(base)
        eng = engine(m, lr=1e-3, augmentation=Augmentation(AugmentationConfig(), train=True, seed=9, gpu_spaghetti=True))
        assert eng.augmentation.gpu_spaghetti
        losses = []
        for i in range(len(batches)):
            losses.append(eng.step(*batches[i]).clone())
            if prefetch and i + 1 < len(batches):
                eng.prefetch(batches[i + 1][0])
        torch.cuda.synchronize()
        assert_bn_state_equal(m, bn0)
        return torch.stack(losses), m.flat_params.clone()

    l0, p0 = run(False)
    l1, p1 = run(True)
    assert torch.isfinite(l0).all()
    assert torch.equal(l0, l1), (l0, l1)
    assert torch.equal(p0, p1)
    assert not torch.equal(p0, base.flat_params)


def test_staged_batch_is_dropped_by_another_forward(cuda_device):
    _, m = build_frozen_pair(cuda_device)
    (u8, _t), = u8_batches([4], 64, 12, cuda_device)
    x = structured_images(4, 6, 64, 64, 1, cuda_device)
    out = torch.empty(4, 6, device=cuda_device)
    m.sync_weights()
    _lib.call("argus_model_stage_input_frozen_u8", m._handle.ptr, u8, None, None, None, 4, 64, 64, 0, _lib.stream_ptr())
    m._forward_impl(x, False, frozen=True)
    with pytest.raises(_lib.ArgusError, match="stage_input_u8"):
        _lib.call("argus_model_forward_frozen", m._handle.ptr, None, 0, 4, 64, 64, out, _lib.stream_ptr())
    # staged for the frozen forward: a training forward does not consume it, and a staged input has no input gradient
    _lib.call("argus_model_stage_input_frozen_u8", m._handle.ptr, u8, None, None, None, 4, 64, 64, 0, _lib.stream_ptr())
    with pytest.raises(_lib.ArgusError, match="stage_input_u8"):
        _lib.call("argus_model_forward", m._handle.ptr, None, 0, 4, 64, 64, 1, out, _lib.stream_ptr())
    _lib.call("argus_model_stage_input_frozen_u8", m._handle.ptr, u8, None, None, None, 4, 64, 64, 0, _lib.stream_ptr())
    _lib.call("argus_model_forward_frozen", m._handle.ptr, None, 0, 4, 64, 64, out, _lib.stream_ptr())
    # (the staged input is the unaugmented uint8 batch: the same output as the uint8 forward)
    want = m._forward_impl(u8, False, frozen=True)
    assert torch.equal(out.view(torch.int32), want.view(torch.int32))
    _lib.call("argus_model_stage_input_frozen_u8", m._handle.ptr, u8, None, None, None, 4, 64, 64, 0, _lib.stream_ptr())
    _lib.call("argus_model_forward_frozen", m._handle.ptr, None, 0, 4, 64, 64, out, _lib.stream_ptr())
    m._backward_impl(torch.ones_like(out))
    dx = torch.empty(4, 6, 64, 64, device=cuda_device)
    with pytest.raises(_lib.ArgusError, match="staged"):
        _lib.call("argus_model_input_grad", m._handle.ptr, dx, _lib.stream_ptr())


# ------------------------------------------------------------------------------------------------------------------
# 4. batch size 1
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_batch_size_one(cuda_device, precision):
    from argus_b200.engine import TrainEngine

    # one image of 32 x 32: one value per channel after layer4, which train-mode batch norm cannot normalise
    _, m = build_frozen_pair(cuda_device, n_cams=1, precision=precision)
    bn0 = bn_state(m)
    x = structured_images(1, 3, 32, 32, 4, cuda_device)
    t = random_targets(1, 4, cuda_device)
    p0 = m.flat_params.clone()
    loss = engine(m).step(x, t)
    torch.cuda.synchronize()
    assert torch.isfinite(loss) and torch.isfinite(m.flat_params).all()
    assert not torch.equal(p0, m.flat_params)
    assert_bn_state_equal(m, bn0)
    with pytest.raises(_lib.ArgusError, match="more than one value per channel"):
        TrainEngine(m, distributed=False).step(x, t)
    # and the bench resolution
    _, m2 = build_frozen_pair(cuda_device, precision=precision)
    p0 = m2.flat_params.clone()
    loss = engine(m2).step(structured_images(1, 6, 256, 256, 5, cuda_device), random_targets(1, 5, cuda_device))
    torch.cuda.synchronize()
    assert torch.isfinite(loss) and not torch.equal(p0, m2.flat_params)


# ------------------------------------------------------------------------------------------------------------------
# 6. no interference with training through the shared stem buffers
# ------------------------------------------------------------------------------------------------------------------
def test_training_trajectory_unchanged(cuda_device):
    from argus_b200.data import Augmentation, AugmentationConfig
    from argus_b200.engine import TrainEngine

    _, base = build_frozen_pair(cuda_device)
    batches = u8_batches([16, 16, 5, 16], 64, 21, cuda_device)
    frozen_data = batches_f32(4, 8, 64, 80, cuda_device)

    def run(interleave):
        m = clone_model(base)
        m.train()
        eng = TrainEngine(m, lr=1e-3, distributed=False,
                          augmentation=Augmentation(AugmentationConfig(), train=True, seed=9, gpu_spaghetti=True))
        # lr = 0: the frozen steps run in full (optimizer and weight refresh included) and leave the weights as they are
        frz = engine(m, lr=0.0)
        losses = []
        for i in range(len(batches)):
            losses.append(eng.step(*batches[i]).clone())
            if interleave:
                frz.step(*frozen_data[i])
                m.eval()
                autograd_flat_grads(m, *frozen_data[(i + 1) % 4])
                m.train()
            if i + 1 < len(batches):
                eng.prefetch(batches[i + 1][0])
        torch.cuda.synchronize()
        return torch.stack(losses), m.flat_params.clone(), {k: v.clone() for k, v in m.state_dict().items()}

    l0, p0, s0 = run(False)
    l1, p1, s1 = run(True)
    assert torch.equal(l0, l1), (l0, l1)
    assert torch.equal(p0, p1)
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k


# ------------------------------------------------------------------------------------------------------------------
# 7. every convolution instance a frozen engine step launches is pinned by the element-wise epilogue cases
# ------------------------------------------------------------------------------------------------------------------
def test_frozen_engine_launches_only_pinned_instances(cuda_device):
    from argus_b200.models import NCameraCNN
    from test_conv_epilogue_gpu import CASES, case_info, key_of, recorded_keys
    from test_frozen_bn_gpu import extra_cases

    table = {key_of(i) for c in CASES + extra_cases() for i in case_info(c)}
    seen = {}
    for B, H in ((256, 256), (8, 128), (1, 256)):
        model = NCameraCNN().to(cuda_device).eval()
        eng = engine(model)
        x = structured_images(B, 6, H, H, 1, cuda_device)
        t = random_targets(B, 1, cuda_device)
        _lib.call("argus_conv_instances_record", 1)
        try:
            eng.step(x, t)
            torch.cuda.synchronize()
        finally:
            _lib.call("argus_conv_instances_record", 0)
        seen[f"frozen engine B={B} {H}x{H}"] = recorded_keys()
        del model, eng, x
        torch.cuda.empty_cache()
    missing = {k: sorted(v - table) for k, v in seen.items() if v - table}
    assert not missing, f"instances the frozen engine launches that no case pins: {missing}"


# ------------------------------------------------------------------------------------------------------------------
# 8. data parallel
# ------------------------------------------------------------------------------------------------------------------
def _set_running_stats(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, buf in model.named_buffers():
            if name.endswith("running_mean"):
                buf.copy_(0.1 * torch.randn(buf.shape, generator=g))
            elif name.endswith("running_var"):
                buf.copy_(0.5 + torch.rand(buf.shape, generator=g))
            elif name.endswith("num_batches_tracked"):
                buf.fill_(7)


def _dp_model(device, seed):
    from argus_b200.models import NCameraCNN
    from test_dp_gpu import _condition

    torch.manual_seed(1234 + seed)
    model = NCameraCNN().to(device)
    _condition(model)
    _set_running_stats(model, seed)
    return model.eval()


def _dp_worker(rank: int, world: int, port: int, out_dir: str) -> None:
    import sys
    from pathlib import Path

    import torch.distributed as dist

    root = Path(__file__).resolve().parent.parent
    sys.path.insert(0, str(root))
    sys.path.insert(0, str(root / "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from argus_b200.engine import TrainEngine
    from test_dp_gpu import B_PER_RANK, _global_batches

    # different weights and running statistics per rank: the constructor must broadcast rank 0's
    model = _dp_model(dev, rank)
    engine = TrainEngine(model, lr=1e-4, max_grad_norm=1.0, frozen_bn=True)
    assert engine.world == world
    sl = slice(rank * B_PER_RANK, (rank + 1) * B_PER_RANK)
    losses = [engine.step(x[sl], t[sl]).clone() for x, t in _global_batches(dev)]
    torch.cuda.synchronize()
    torch.save({"params": model.flat_params.detach().cpu(), "buffers": model._flat_buffers.detach().cpu(),
                "nbt": model._flat_nbt.detach().cpu(), "losses": torch.stack(losses).cpu()},
               os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_nccl_equals_single_process_oracle(tmp_path):
    import torch.multiprocessing as mp

    from test_dp_gpu import B_PER_RANK, _free_port, _global_batches

    mp.spawn(_dp_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "rank0.pt"), torch.load(tmp_path / "rank1.pt")
    dev = torch.device("cuda", 0)
    model = _dp_model(dev, 0)
    buffers0, nbt0 = model._flat_buffers.detach().cpu().clone(), model._flat_nbt.detach().cpu().clone()
    eng = engine(model, lr=1e-4)
    eng.grad_divisor = 2.0
    losses = []
    for x, t in _global_batches(dev):
        losses.append(eng.forward_backward(x[:B_PER_RANK], t[:B_PER_RANK]).clone())
        g0 = model.flat_grads.clone()
        eng.forward_backward(x[B_PER_RANK:], t[B_PER_RANK:])
        model.flat_grads.add_(g0)
        eng.optimizer_step()
    torch.cuda.synchronize()
    assert torch.equal(r0["params"], r1["params"])
    assert torch.equal(r0["losses"], torch.stack(losses).cpu()), (r0["losses"], losses)
    assert torch.equal(r0["params"], model.flat_params.detach().cpu())
    for r in (r0, r1):
        assert torch.equal(r["buffers"], buffers0) and torch.equal(r["nbt"], nbt0)


# ------------------------------------------------------------------------------------------------------------------
# 9. command line: fine-tune a checkpoint with frozen statistics
# ------------------------------------------------------------------------------------------------------------------
def test_train_cli_fine_tunes_with_frozen_statistics(cuda_device, tmp_path):
    import numpy as np

    from argus_b200.dataset import CameraCubePoseDatasetConfig, write_dataset
    from argus_b200.train import TrainConfig, state_dict_for_save, train

    rng = np.random.default_rng(0)

    def poses(n):
        q = rng.normal(size=(n, 4))
        q /= np.linalg.norm(q, axis=-1, keepdims=True)
        return np.concatenate([rng.normal(size=(n, 3)), q], -1)

    imgs = rng.integers(0, 256, (24, 2, 128, 128, 3), dtype=np.uint8)
    data = tmp_path / "data"
    write_dataset(str(data), imgs[:16], poses(16), imgs[16:], poses(8))
    _, m = build_frozen_pair(cuda_device)
    init = tmp_path / "init.pth"
    sd0 = state_dict_for_save(m, multigpu=True)       # with DDP's `module.` prefix
    torch.save(sd0, init)
    save_dir = tmp_path / "out"
    cfg = TrainConfig(dataset_config=CameraCubePoseDatasetConfig(dataset_path=str(data), center_crop=(128, 128)),
                      batch_size=8, n_epochs=1, device="cuda", wandb_log=False, save_dir=str(save_dir), num_workers=0,
                      num_gpus=1, freeze_bn=True, init_model_path=str(init))
    run_id = train(cfg)
    sd = torch.load(save_dir / f"{run_id}.pth", map_location="cpu", weights_only=True)
    assert len(sd) == 326 and [("module." + k) for k in sd] == list(sd0)
    changed = 0
    for k, v in sd.items():
        v0 = sd0["module." + k].cpu()
        if "running" in k or "num_batches" in k:
            assert torch.equal(v, v0), k
        elif not torch.equal(v, v0):
            changed += 1
    assert changed > 0
