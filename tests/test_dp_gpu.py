"""GPU multi-rank parity (needs >= 2 GPUs; skipped otherwise): the data-parallel path of the reference
(/root/reference/argus/train.py:137-140,154-166,199: NCCL process group, DistributedSampler shards, DDP gradient averaging,
per-rank batch-norm statistics, rank 0's buffers) against the DP oracle of SURVEY.md §8(c):

  * a 2-rank NCCL run of TrainEngine must equal, BIT FOR BIT, a single process that runs the two shards one after the
    other (per-shard BN statistics), sums their gradient arenas and applies the optimizer with the 1/world scale -- this
    catches a wrong scale, a stale or missing bucket and a missing parameter / buffer broadcast;
  * the same 2-rank run in fp32 parity mode must track torch's own DistributedDataParallel on the reference model
    (same shards, same weights) on the per-step losses (first step to fp32 round-off, then within 1e-3 while Adam's
    sign-like first updates amplify round-off).
"""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu

N_STEPS = 3
B_PER_RANK = 4
SIZE = 64


def _free_port() -> int:
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _condition(model) -> None:
    """Scale the last BN of every residual branch (what tests/test_fp32_mode_gpu.py does): a randomly initialised
    train-mode ResNet-50 amplifies fp32 round-off by orders of magnitude, which would hide what this test is about."""
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("bn3.weight"):
                p.fill_(0.2)


def _global_batches(device):
    from gpu_util import random_targets, structured_images

    return [(structured_images(2 * B_PER_RANK, 6, SIZE, SIZE, 100 + i, device), random_targets(2 * B_PER_RANK, 200 + i, device))
            for i in range(N_STEPS)]


def _worker(rank: int, world: int, port: int, out_dir: str, precision: str) -> None:
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
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    from argus_b200.engine import TrainEngine
    from argus_b200.models import NCameraCNN
    from oracle.ref_model import make_reference_model, torch_loss

    # deliberately DIFFERENT initial weights per rank: the engine's constructor must broadcast rank 0's (DDP does)
    torch.manual_seed(1234 + rank)
    model = NCameraCNN().to(dev).set_precision(precision)
    _condition(model)
    engine = TrainEngine(model, lr=1e-4, max_grad_norm=1.0)
    assert engine.world == world
    batches = _global_batches(dev)
    sl = slice(rank * B_PER_RANK, (rank + 1) * B_PER_RANK)
    losses = [engine.step(x[sl], t[sl]).clone() for x, t in batches]
    torch.cuda.synchronize()
    result = {"params": model.flat_params.detach().cpu(), "buffers": model._flat_buffers.detach().cpu(),
              "losses": torch.stack(losses).cpu()}
    if precision == "fp32":
        # torch's own DDP on the reference model, same shards (train.py:199: all DDP defaults)
        torch.manual_seed(1234)   # rank 0's initial weights == what the engine broadcast
        ours0 = NCameraCNN()
        _condition(ours0)
        ref = make_reference_model(0)
        ref.load_state_dict(ours0.state_dict())
        ddp = torch.nn.parallel.DistributedDataParallel(ref.to(dev), device_ids=[rank])
        opt = torch.optim.Adam(ddp.parameters(), lr=1e-4)
        ref_losses = []
        for x, t in batches:
            opt.zero_grad()
            loss = torch_loss(ddp(x[sl]).float(), t[sl]).mean().float()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(ddp.parameters(), 1.0)
            opt.step()
            ref_losses.append(loss.detach())
        result["ref_losses"] = torch.stack(ref_losses).cpu()
    torch.save(result, os.path.join(out_dir, f"rank{rank}_{precision}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def _single_process_oracle(device, precision: str):
    """The two shards one after the other on ONE GPU: per-shard BN statistics, summed gradients, 1/world in the
    optimizer; rank 0's running statistics are those of shard 0 only."""
    from argus_b200.engine import TrainEngine
    from argus_b200.models import NCameraCNN

    torch.manual_seed(1234)
    model = NCameraCNN().to(device).set_precision(precision)
    _condition(model)
    engine = TrainEngine(model, lr=1e-4, max_grad_norm=1.0, distributed=False)
    engine.grad_divisor = 2.0   # gradient scale 1/world, exactly what the 2-rank engine applies
    losses0 = []
    for x, t in _global_batches(device):
        l0 = engine.forward_backward(x[:B_PER_RANK], t[:B_PER_RANK]).clone()
        g0 = model.flat_grads.clone()
        buffers0 = model._flat_buffers.clone()
        nbt0 = model._flat_nbt.clone()
        engine.forward_backward(x[B_PER_RANK:], t[B_PER_RANK:])
        model.flat_grads.add_(g0)                       # what the NCCL SUM all-reduce leaves on every rank
        model._flat_buffers.copy_(buffers0)             # rank 0 never sees shard 1's statistics
        model._flat_nbt.copy_(nbt0)
        engine.optimizer_step()
        losses0.append(l0)
    torch.cuda.synchronize()
    return model.flat_params.detach().cpu(), model._flat_buffers.detach().cpu(), torch.stack(losses0).cpu()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_two_rank_nccl_equals_single_process_oracle(tmp_path, precision):
    import torch.multiprocessing as mp

    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path), precision), nprocs=2, join=True)
    r0 = torch.load(tmp_path / f"rank0_{precision}.pt")
    r1 = torch.load(tmp_path / f"rank1_{precision}.pt")
    # every rank holds the same parameters after every step (averaged gradients, identical optimizer)
    assert torch.equal(r0["params"], r1["params"])
    params, buffers, losses0 = _single_process_oracle(torch.device("cuda", 0), precision)
    assert torch.equal(r0["losses"], losses0), (r0["losses"], losses0)
    assert torch.equal(r0["params"], params), float((r0["params"] - params).abs().max())
    assert torch.equal(r0["buffers"], buffers)                     # rank 0's running statistics: its own shard only
    assert not torch.equal(r0["buffers"], r1["buffers"])           # per-rank statistics (no SyncBN in the reference)
    if precision == "fp32":
        rel = ((r0["losses"] - r0["ref_losses"]).abs() / r0["ref_losses"].abs()).max().item()
        # torch DDP on the reference model. Adam's first steps are sign-like (m / sqrt(v) = +-1), so round-off in
        # near-zero gradients moves single weights by 2 lr: the single-GPU fp32-mode test sees up to 1.5e-4 after eight
        # steps and asserts 1e-3 (tests/test_fp32_mode_gpu.py); same bound here
        assert rel < 1e-3, (r0["losses"], r0["ref_losses"])
