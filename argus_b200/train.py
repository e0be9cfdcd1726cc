"""Training entry point (reference: /root/reference/argus/train.py). Same TrainConfig fields, same
`train(cfg, rank)` / `geometric_loss_fn` / `initialize_training` names, same `.pth` output (`model.state_dict()`,
with DDP's `module.` key prefix under `multigpu`, train.py:357-358,199) — the step body (train.py:298-320) is the fused
engine of argus_b200.engine.

    python -m argus_b200.train --dataset-config.dataset-path <dir> [--multigpu] ...
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field
from pathlib import Path
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from torch.utils.data import DataLoader
from torch.utils.data.distributed import DistributedSampler

from . import ROOT
from .data import Augmentation, AugmentationConfig
from .dataset import CameraCubePoseDataset, CameraCubePoseDatasetConfig
from .engine import GradScaler, TrainEngine
from .loss import geometric_loss_fn
from .models import NCameraCNN, NCameraCNNConfig

__all__ = ["TrainConfig", "geometric_loss_fn", "initialize_training", "train", "ReduceLROnPlateau"]


@dataclass(frozen=True)
class TrainConfig:
    """Configuration for training (fields and defaults of the reference, train.py:29-103)."""

    # model and dataset parameters
    dataset_config: CameraCubePoseDatasetConfig
    model_config: NCameraCNNConfig = NCameraCNNConfig()
    compile_model: bool = False  # accepted for CLI parity; the CUDA path is already a static launch schedule

    # training parameters
    batch_size: int = 32
    learning_rate: float = 1e-4
    n_epochs: int = 100
    device: str = "cuda" if torch.cuda.is_available() else "cpu"
    max_grad_norm: float = 1.0
    num_gpus: int = torch.cuda.device_count()
    random_seed: int = 42

    # speed optimizations
    multigpu: bool = False
    # mixed precision under the reference's GradScaler protocol (train.py:74,234,298-300,316-320): loss scaling, unscale
    # before clipping, non-finite steps skipped. The reduced-precision arithmetic is the bf16 tensor-core path rather than
    # fp16 autocast (engine.GradScaler); amp=True therefore requires precision="bf16"
    amp: bool = False
    # not in the reference: "bf16" = tcgen05 tensor-core path (default), "fp32" = the fp32 parity mode (what the
    # reference computes with amp=False), see argus_model_set_precision in include/argus_b200.h
    precision: str = "bf16"
    # not in the reference: fine-tuning with frozen batch norm -- every training forward uses the running statistics as
    # constants and leaves them unchanged (TrainEngine(frozen_bn=True), argus_model_forward_frozen)
    freeze_bn: bool = False
    # not in the reference: a .pth (model.state_dict(), with or without DDP's `module.` prefix) loaded with strict=True
    # before training starts; what freeze_bn fine-tunes from, since the running statistics of a fresh network are 0 / 1
    init_model_path: Optional[str] = None

    # validation, printing, and saving
    val_epochs: int = 1
    print_epochs: int = 1
    save_epochs: int = 5
    save_dir: str = ROOT + "/outputs/models"

    # data augmentation
    augmentation_config: AugmentationConfig = AugmentationConfig()
    use_augmentation: bool = True

    # wandb
    wandb_project: str = "argus-estimator"
    wandb_log: bool = True

    # loader (not in the reference: worker count was hard-coded, train.py:147-149)
    num_workers: int = 8
    # draw_spaghetti on the device (one kernel per batch) instead of PIL in the loader workers (data.py:212-215)
    gpu_spaghetti: bool = True

    def __post_init__(self) -> None:
        assert isinstance(self.save_dir, str)
        if not os.path.exists(self.save_dir):
            if os.path.exists(ROOT + "/" + self.save_dir):
                object.__setattr__(self, "save_dir", ROOT + "/" + self.save_dir)
            else:
                os.makedirs(self.save_dir, exist_ok=True)
        assert self.num_gpus > 0, "The number of GPUs must be greater than 0!"
        assert self.num_gpus <= torch.cuda.device_count(), \
            "The number of GPUs must be less than or equal to the number of GPUs on the system!"
        assert not (self.amp and self.precision != "bf16"), \
            "amp=True is mixed precision: it cannot be combined with precision='fp32'"


class ReduceLROnPlateau:
    """torch.optim.lr_scheduler.ReduceLROnPlateau('min', patience, factor) (train.py:233) acting on engine.lr."""

    def __init__(self, engine: TrainEngine, patience: int = 5, factor: float = 0.5, threshold: float = 1e-4) -> None:
        self.engine, self.patience, self.factor, self.threshold = engine, patience, factor, threshold
        self.best = float("inf")
        self.num_bad_epochs = 0

    def step(self, metric: float) -> None:
        if metric < self.best * (1.0 - self.threshold):
            self.best = metric
            self.num_bad_epochs = 0
        else:
            self.num_bad_epochs += 1
        if self.num_bad_epochs > self.patience:
            self.engine.lr *= self.factor
            self.num_bad_epochs = 0


def _collate_u8(samples: list[dict]) -> dict:
    return {"images": torch.stack([s["images"] for s in samples]),
            "cube_pose": torch.stack([s["cube_pose"] for s in samples])}


def load_state_dict_for_init(path: str) -> dict:
    """A saved `.pth` as `model.load_state_dict` takes it: the `module.` prefix of a checkpoint saved under multigpu
    (state_dict_for_save) is removed."""
    sd = torch.load(path, map_location="cpu", weights_only=True)
    if sd and all(k.startswith("module.") for k in sd):
        sd = {k[len("module."):]: v for k, v in sd.items()}
    return sd


def initialize_training(cfg: TrainConfig, rank: int = 0):
    """Sets up the training (reference: train.py:122-255). Returns the reference's 10-tuple
    `(train_dataloader, val_dataloader, model, optimizer, scheduler, loss_fn, wandb_id, train_sampler, val_sampler,
    scaler)`; the `optimizer` slot holds the fused TrainEngine (Adam state + step; `param_groups`, `zero_grad`,
    `state_dict` as torch.optim.Adam), `scaler` an engine.GradScaler(enabled=cfg.amp)."""
    torch.cuda.manual_seed_all(cfg.random_seed)
    torch.manual_seed(cfg.random_seed)
    np.random.seed(cfg.random_seed)
    device = torch.device("cuda", rank) if cfg.multigpu else torch.device(cfg.device)
    if device.type != "cuda":
        raise RuntimeError("argus_b200 trains on sm_100a GPUs only (no CPU fallback)")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    torch.cuda.set_device(device)
    if cfg.multigpu:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "12355")
        dist.init_process_group("nccl", rank=rank, world_size=cfg.num_gpus)

    aug_cfg = cfg.augmentation_config if cfg.use_augmentation else None
    pil = not cfg.gpu_spaghetti
    train_dataset = CameraCubePoseDataset(cfg.dataset_config, cfg_aug=aug_cfg, train=True, as_uint8=True, pil_spaghetti=pil)
    val_dataset = CameraCubePoseDataset(cfg.dataset_config, cfg_aug=aug_cfg, train=False, as_uint8=True, pil_spaghetti=pil)
    if cfg.multigpu:
        train_sampler = DistributedSampler(train_dataset, num_replicas=cfg.num_gpus, rank=rank, shuffle=True)
        val_sampler = DistributedSampler(val_dataset, num_replicas=cfg.num_gpus, rank=rank, shuffle=False)
        train_shuffle = None
    else:
        train_sampler = val_sampler = None
        train_shuffle = True
    workers = cfg.num_workers
    common = dict(batch_size=cfg.batch_size, num_workers=workers, pin_memory=True, collate_fn=_collate_u8,
                  multiprocessing_context="fork" if workers > 0 else None, persistent_workers=workers > 0)
    train_dataloader = DataLoader(train_dataset, shuffle=train_shuffle, sampler=train_sampler, **common)
    val_dataloader = DataLoader(val_dataset, shuffle=False, sampler=val_sampler, **common)

    model = NCameraCNN(cfg.model_config).to(device).set_precision(cfg.precision)
    if cfg.init_model_path is not None:
        model.load_state_dict(load_state_dict_for_init(cfg.init_model_path), strict=True)
    augmentation = Augmentation(cfg.augmentation_config, train=True, seed=cfg.random_seed + 7919 * rank,
                                gpu_spaghetti=cfg.gpu_spaghetti) if cfg.use_augmentation else None
    scaler = GradScaler(enabled=cfg.amp)
    engine = TrainEngine(model, lr=cfg.learning_rate, max_grad_norm=cfg.max_grad_norm, augmentation=augmentation,
                         scaler=scaler, frozen_bn=cfg.freeze_bn)
    scheduler = ReduceLROnPlateau(engine, patience=5, factor=0.5)
    loss_fn = geometric_loss_fn

    wandb_id = None
    if cfg.wandb_log and rank == 0:
        import wandb
        from wandb.util import generate_id

        wandb_id = generate_id()
        wandb.init(project=cfg.wandb_project, config=cfg, id=wandb_id, resume="allow")
    if wandb_id is None:
        wandb_id = f"argus_b200_{os.getpid()}"
    return (train_dataloader, val_dataloader, model, engine, scheduler, loss_fn, wandb_id, train_sampler, val_sampler,
            scaler)


def rank_print(msg: str, rank: int = 0) -> None:
    if rank == 0:
        print(msg)


def state_dict_for_save(model: NCameraCNN, multigpu: bool) -> dict:
    """`model.state_dict()` as the reference writes it: contiguous CPU-loadable tensors; under multigpu the reference
    saves the DDP wrapper's state dict, so every key carries the `module.` prefix (train.py:199,357-358)."""
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return {("module." + k): v for k, v in sd.items()} if multigpu else sd


def train(cfg: TrainConfig, rank: int = 0) -> None:
    """Main training loop (reference: train.py:264-361)."""
    (train_dataloader, val_dataloader, model, engine, scheduler, loss_fn, wandb_id, train_sampler,
     val_sampler, _scaler) = initialize_training(cfg, rank=rank)
    device = model.flat_params.device
    log = cfg.wandb_log and rank == 0
    if log:
        import wandb
    for epoch in range(cfg.n_epochs):
        if cfg.multigpu:
            dist.barrier()
            train_sampler.set_epoch(epoch)
        model.train()
        epoch_losses = []
        pending = None  # loss of the previous step, read one step late so that no step ever synchronises

        def to_device(example):
            if example is None:
                return None
            return (example["images"].to(device, non_blocking=True),        # (B, n_cams, H, W, 3) uint8
                    example["cube_pose"].to(device, non_blocking=True))     # (B, 7) [t, q_xyzw]

        # one batch of look-ahead: while step k trains, batch k+1 is copied to the device and augmented + staged on the
        # engine's side stream (the reference augments on CPU workers, data.py:213-225)
        batches = iter(train_dataloader)
        current = to_device(next(batches, None))
        while current is not None:
            upcoming = to_device(next(batches, None))
            loss = engine.step(*current)
            if upcoming is not None:
                engine.prefetch(upcoming[0])
            epoch_losses.append(loss.detach().clone())
            if log and pending is not None:
                wandb.log({"loss": float(pending)})
            pending = epoch_losses[-1]
            current = upcoming
        if log and pending is not None:
            wandb.log({"loss": float(pending)})
        if epoch % cfg.print_epochs == 0 and epoch_losses:
            rank_print(f"    Avg. Loss in Epoch: {torch.stack(epoch_losses).mean().item()}", rank=rank)

        if epoch % cfg.val_epochs == 0:
            model.eval()
            with torch.no_grad():
                val_losses = []
                for example in val_dataloader:
                    images = example["images"].to(device, non_blocking=True)
                    cube_pose = example["cube_pose"].to(device, non_blocking=True)
                    aug = engine.augmentation
                    if aug is not None and aug.gpu_spaghetti:
                        images = aug.spaghetti_batch(images)   # the reference draws arcs on validation images too
                    pred = model(images)
                    val_losses.append(loss_fn(pred, cube_pose))
                if val_losses:
                    val_loss_t = torch.mean(torch.cat(val_losses))
                    if cfg.multigpu:
                        # the reference steps ReduceLROnPlateau on each rank's own shard (train.py:340-348), which lets
                        # the learning rates -- and then the weights -- of the ranks drift apart; every rank uses the
                        # mean over ranks here so that engine.lr stays identical everywhere
                        dist.all_reduce(val_loss_t, op=dist.ReduceOp.SUM)
                        val_loss_t = val_loss_t / cfg.num_gpus
                    val_loss = val_loss_t.item()
                    if log:
                        wandb.log({"val_loss": val_loss})
                    rank_print(f"    Validation loss: {val_loss}", rank=rank)
                    scheduler.step(val_loss)

        if epoch % cfg.save_epochs == 0:
            save_dir = Path(cfg.save_dir) if cfg.save_dir is not None else Path(ROOT + "/outputs/models")
            os.makedirs(save_dir, exist_ok=True)
            if rank == 0:
                torch.save(state_dict_for_save(model, cfg.multigpu), save_dir / f"{wandb_id}.pth")
    if cfg.multigpu:
        dist.destroy_process_group()
    return wandb_id


def _train_multigpu(rank: int, cfg: TrainConfig) -> None:
    train(cfg, rank=rank)


if __name__ == "__main__":
    import tyro

    cfg = tyro.cli(TrainConfig)
    if cfg.multigpu:
        mp.spawn(_train_multigpu, args=(cfg,), nprocs=cfg.num_gpus, join=True)
    else:
        train(cfg, rank=0)
