"""Fused training step for the hot path of /root/reference/argus/train.py:298-320:

    images.to(device) -> [augmentation] -> model(images) -> geometric_loss_fn -> mean -> backward
    -> clip_grad_norm_(max_grad_norm) -> Adam step

executed as a handful of C-ABI calls on one stream, with no host synchronisation inside the step (the reference
synchronises every step through `loss.item()`, train.py:312). Under data parallelism (train.py:137-166,199) the
gradient arena is all-reduced in four reverse-order buckets over NCCL while the rest of the backward pass runs.
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional

import torch
import torch.distributed as dist

from . import _lib
from .models import NCameraCNN


def gradient_buckets(flat: torch.Tensor, stage_ranges: list[tuple[int, int]]) -> list[torch.Tensor]:
    """Views of the flat gradient arena, one per backward stage, in the order they become final
    (stage 0 = layer4 + fc + head ... stage 3 = stem + layer1). Together they tile the arena exactly once."""
    return [flat[b:e] for (b, e) in stage_ranges]


def all_reduce_bucket(bucket: torch.Tensor, group=None, async_op: bool = True):
    """SUM all-reduce of one bucket (the 1/world average is folded into the optimizer's gradient scale).
    DDP in the reference averages 25 MiB buckets the same way (train.py:199)."""
    return dist.all_reduce(bucket, op=dist.ReduceOp.SUM, group=group, async_op=async_op)


class GradScaler:
    """The reference's `torch.cuda.amp.GradScaler(enabled=cfg.amp)` (argus/train.py:234,316-320) for the fused engine:
    same constructor defaults and the same protocol -- the loss gradient is multiplied by `get_scale()`, gradients are
    unscaled before `clip_grad_norm_`, a step whose unscaled gradient norm is not finite is skipped as a whole, and
    `update()` backs the scale off by `backoff_factor` after a skipped step or grows it by `growth_factor` after
    `growth_interval` clean ones. What differs (DESIGN.md §5): the reduced-precision arithmetic under `amp=True` is
    the bf16 tensor-core path (fp32 exponent range), not fp16 autocast, so skips are rare; like `scaler.step` in the
    reference, an enabled scaler costs one host synchronisation per step (it reads the gradient norm)."""

    def __init__(self, init_scale: float = 2.0 ** 16, growth_factor: float = 2.0, backoff_factor: float = 0.5,
                 growth_interval: int = 2000, enabled: bool = True) -> None:
        self._enabled = bool(enabled)
        self._scale = float(init_scale)
        self.growth_factor, self.backoff_factor = float(growth_factor), float(backoff_factor)
        self.growth_interval = int(growth_interval)
        self._growth_tracker = 0
        self.skipped_steps = 0

    def is_enabled(self) -> bool:
        return self._enabled

    def get_scale(self) -> float:
        return self._scale if self._enabled else 1.0

    def scale(self, outputs: torch.Tensor) -> torch.Tensor:
        return outputs * self._scale if self._enabled else outputs

    def update(self, found_inf: bool = False) -> None:
        if not self._enabled:
            return
        if found_inf:
            self._scale *= self.backoff_factor
            self._growth_tracker = 0
            self.skipped_steps += 1
        else:
            self._growth_tracker += 1
            if self._growth_tracker == self.growth_interval:
                self._scale *= self.growth_factor
                self._growth_tracker = 0

    def state_dict(self) -> dict:
        return {"scale": self._scale, "growth_factor": self.growth_factor, "backoff_factor": self.backoff_factor,
                "growth_interval": self.growth_interval, "_growth_tracker": self._growth_tracker} if self._enabled else {}

    def load_state_dict(self, state: dict) -> None:
        if self._enabled and state:
            self._scale = float(state["scale"])
            self._growth_tracker = int(state["_growth_tracker"])


class TrainEngine:
    """Owns the optimizer state (flat Adam moments) and runs fused training steps on an NCameraCNN.

    Args:
        model: an argus_b200 NCameraCNN already on a CUDA device.
        lr, betas, eps: torch.optim.Adam defaults as used by the reference (train.py:232).
        max_grad_norm: clip_grad_norm_ threshold (train.py:318); <= 0 disables clipping.
        process_group: torch.distributed group for data parallelism (None = single process).
        augmentation: optional argus_b200.data.Augmentation applied on device to uint8 image batches.
        scaler: optional GradScaler (the reference's amp mode, train.py:234,298-300,316-320).
        frozen_bn: not in the reference -- fine-tuning with frozen batch norm. Every forward is the frozen-statistics
            forward (argus_model_forward_frozen): batch norm uses the running statistics as constants, and neither the
            running statistics nor num_batches_tracked change. `model.training` is left as it is. Loss, backward,
            all-reduce buckets and the optimizer are those of a training step.

    It also stands in the reference's `optimizer` slot of `initialize_training` (train.py:245-255): `param_groups`,
    `zero_grad()`, `state_dict()` / `load_state_dict()` follow torch.optim.Adam's surface.
    """

    def __init__(self, model: NCameraCNN, lr: float = 1e-4, max_grad_norm: float = 1.0,
                 betas: tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                 process_group: Optional["dist.ProcessGroup"] = None, distributed: Optional[bool] = None,
                 augmentation=None, scaler: Optional[GradScaler] = None, frozen_bn: bool = False) -> None:
        if not model.flat_params.is_cuda:
            raise _lib.ArgusError("TrainEngine needs the model on a CUDA device (no CPU fallback)")
        self.model = model
        self.lr = float(lr)
        self.max_grad_norm = float(max_grad_norm)
        self.betas = (float(betas[0]), float(betas[1]))
        self.eps = float(eps)
        self.augmentation = augmentation
        self.scaler = scaler
        self.frozen_bn = bool(frozen_bn)
        self.step_count = 0
        self.device = model.flat_params.device
        if distributed is None:
            distributed = dist.is_available() and dist.is_initialized()
        self.distributed = bool(distributed)
        self.group = process_group
        self.world = dist.get_world_size(process_group) if self.distributed else 1
        # the all-reduce SUMS the ranks' gradients; DDP's averaging (train.py:199) is this divisor, folded into the
        # optimizer's gradient scale. (A test sets it by hand to emulate two ranks in one process.)
        self.grad_divisor = float(self.world)
        n = model.flat_params.numel()
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=self.device)
        self._scratch = torch.zeros(1024, dtype=torch.float32, device=self.device)
        self._grad_norm = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._loss_mean = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._stage_ranges = model.stage_ranges()
        self.last_grad_norm = self._grad_norm
        # look-ahead staging (prefetch): side stream + event, see prefetch()
        self._side = torch.cuda.Stream(device=self.device)
        self._staged_event = torch.cuda.Event()
        self._staged = None            # (data_ptr, shape) of the uint8 batch already augmented into the model
        if self.distributed:
            # DDP's constructor broadcasts rank 0's parameters and buffers (train.py:199); with frozen_bn the running
            # statistics never change afterwards, so the ranks keep identical buffers
            dist.broadcast(model.flat_params, src=0, group=process_group)
            dist.broadcast(model._flat_buffers, src=0, group=process_group)
            model.sync_weights(force=True)

    # ------------------------------------------------------------------------------------------------------------
    def prefetch(self, images: torch.Tensor, after: Optional["torch.cuda.Event"] = None) -> None:
        """Augment + stage the NEXT uint8 batch on a side stream while the step enqueued just before keeps the GPU
        busy (the augmentation kernel is ALU-bound, the training step HBM-bound: they overlap well). The model keeps
        two stem-input buffers, so the batch in flight is not disturbed. Call it right after step(); the following
        step() / forward_backward() must be given the same tensor. `after`: an event the staging must wait for (e.g. the
        host-to-device copy of `images` on a copy stream); work already enqueued on the current stream before the
        preceding step() is waited for automatically. A no-op for inputs the fused staging path does not cover (float
        images, fp32 mode)."""
        model = self.model
        if images.dtype != torch.uint8 or model.precision != "bf16":
            return
        aug = self.augmentation
        apply = aug is not None and aug.train and aug.enabled
        key = (images.data_ptr(), tuple(images.shape))
        # the buffer being written was last read by the forward BEFORE the one in flight (this engine's previous step, or
        # whatever training / frozen forward ran in between): wait for that one only
        if model._stem_free is not None:
            self._side.wait_event(model._stem_free)
        if after is not None:
            self._side.wait_event(after)
        with torch.cuda.stream(self._side):
            B, n_cams, H, W, _ = images.shape
            images = images.contiguous()
            # (workspaces of their own: the step in flight on the main stream may still be using the default ones)
            arc_mask = (aug.arc_mask(B * n_cams, H, W, self.device, tag="arcs_side")
                        if (aug is not None and aug.gpu_spaghetti) else None)
            params = aug.sample_params(B, n_cams, self.device, H=H, W=W) if apply else None
            ws = aug.workspace(B * n_cams, H, W, self.device, tag="plasma_side") if apply else None
            model._ensure_bound()
            with torch.cuda.device(self.device):
                if self.frozen_bn:
                    _lib.call("argus_model_stage_input_frozen_u8", model._handle.ptr, images, params, arc_mask, ws,
                              int(B), int(H), int(W), int(apply), _lib.stream_ptr())
                else:
                    _lib.call("argus_model_stage_input_u8", model._handle.ptr, images, params, arc_mask, ws, int(B),
                              int(H), int(W), 1, int(apply), _lib.stream_ptr())
            self._staged_event.record(self._side)
        # the next forward into the stem buffers, whichever it is, waits for this write
        model._staging = self._staged_event
        images.record_stream(self._side)
        if params is not None:
            params.record_stream(self._side)
        self._staged = key

    # ------------------------------------------------------------------------------------------------------------
    # torch.optim.Optimizer-like surface (the engine sits in the `optimizer` slot of initialize_training's tuple)
    @property
    def param_groups(self) -> list[dict]:
        return [{"params": list(self.model.parameters()), "lr": self.lr, "betas": self.betas, "eps": self.eps,
                 "weight_decay": 0.0}]

    def zero_grad(self, set_to_none: bool = False) -> None:
        """Gradients live in the model's flat arena and are zeroed at the start of every backward pass."""
        model = self.model
        with torch.cuda.device(self.device):
            _lib.call("argus_model_zero_grads", model._handle.ptr, _lib.stream_ptr())

    def forward_backward(self, images: torch.Tensor, targets: torch.Tensor, loss_scale: float = 1.0) -> torch.Tensor:
        """Forward, loss, backward (+ bucketed gradient all-reduce). Returns the mean loss as a device scalar.

        images: (B, 3*n_cams, H, W) float32 in [0,1]  or  (B, n_cams, H, W, 3) uint8; targets: (B, 7) [t, q_xyzw].
        loss_scale: GradScaler factor on d(loss)/d(pred) (`scaler.scale(loss).backward()`, train.py:316).
        """
        model = self.model
        lib_stream = _lib.stream_ptr()
        frozen = self.frozen_bn
        training = not frozen
        if training:
            model.train()
        # The model orders its stem buffers (NCameraCNN._stem_input_turn): the forward below waits for a staged batch
        # (also when it is not the one given now: its write into the alternate buffer must be over before anything else
        # is written there) and marks when everything enqueued before it, the previous step included, is done. A
        # prefetch() issued after this call may overwrite the stem buffer of the previous step from then on.
        staged, self._staged = self._staged, None
        if staged is not None and images.dtype == torch.uint8 and staged == (images.data_ptr(), tuple(images.shape)):
            out = model._forward_staged(images.shape[0], images.shape[2], images.shape[3], frozen=frozen)
        elif images.dtype == torch.uint8 and model.precision == "fp32":
            # fp32 parity mode: the same augmentation kernel with fp32 NCHW output, then the fp32 network
            aug = self.augmentation
            B_, n_cams, H, W, _ = images.shape
            if aug is not None and aug.train and aug.enabled:
                arc_mask = aug.arc_mask(B_ * n_cams, H, W, self.device) if aug.gpu_spaghetti else None
                out = model._forward_impl(aug.augment_batch(images, arc_mask=arc_mask), training, frozen=frozen)
            elif aug is not None and aug.gpu_spaghetti:
                out = model._forward_impl(aug.spaghetti_batch(images), training, frozen=frozen)
            else:
                out = model._forward_impl(images, training, frozen=frozen)
        elif images.dtype == torch.uint8:
            # fused augmentation + staging: uint8 pairs -> augmented bf16 stem input inside the model's staging buffer
            aug = self.augmentation
            B_, n_cams, H, W, _ = images.shape
            arc_mask = aug.arc_mask(B_ * n_cams, H, W, self.device) if (aug is not None and aug.gpu_spaghetti) else None
            apply = aug is not None and aug.train and aug.enabled
            params = aug.sample_params(B_, n_cams, self.device, H=H, W=W) if apply else None
            ws = aug.workspace(B_ * n_cams, H, W, self.device) if apply else None
            out = model._forward_impl(images, training, aug_params=params, augment=apply, arc_mask=arc_mask, plasma_ws=ws,
                                      frozen=frozen)
        else:
            out = model._forward_impl(images, training, frozen=frozen)
        B = out.shape[0]
        targets = targets.to(device=self.device, dtype=torch.float32).contiguous()
        grad = torch.empty_like(out)
        self._loss_mean.zero_()
        with torch.cuda.device(self.device):
            # d(mean loss)/d pred = grad / B   (train.py:308-309; the loss is always evaluated in fp32)
            _lib.call("argus_pose_loss", out, targets, None, self._loss_mean, grad, int(B), float(loss_scale) / B,
                      lib_stream)
            _lib.call("argus_model_zero_grads", model._handle.ptr, lib_stream)
            works = []
            buckets = gradient_buckets(model.flat_grads, self._stage_ranges)
            for stage in range(4):
                _lib.call("argus_model_backward", model._handle.ptr, grad, stage, stage + 1, lib_stream)
                if self.world > 1:
                    # NCCL runs on its own stream: it waits for this stage's kernels, the next stage overlaps with it
                    works.append(all_reduce_bucket(buckets[stage], self.group, async_op=True))
            for w in works:
                w.wait()
        return self._loss_mean[0]

    def optimizer_step(self, inv_loss_scale: float = 1.0, skip_nonfinite: bool = False) -> None:
        """clip_grad_norm_ + Adam on the flat arenas, then refresh the packed bf16 weights.
        skip_nonfinite: GradScaler protocol -- nothing is updated when the unscaled gradient norm is not finite."""
        model = self.model
        self.step_count += 1
        lib = _lib.load()
        fn = lib.argus_clip_adam_step_amp if skip_nonfinite else lib.argus_clip_adam_step
        with torch.cuda.device(self.device):
            _lib.check(fn(
                _lib.ptr(model.flat_params), _lib.ptr(model.flat_grads), _lib.ptr(self.exp_avg),
                _lib.ptr(self.exp_avg_sq), ctypes.c_int64(model.flat_params.numel()), _lib.ptr(self._scratch),
                ctypes.c_float(inv_loss_scale / self.grad_divisor), ctypes.c_float(self.max_grad_norm), ctypes.c_float(self.lr),
                ctypes.c_float(self.betas[0]), ctypes.c_float(self.betas[1]), ctypes.c_float(self.eps),
                ctypes.c_int(self.step_count), _lib.ptr(self._grad_norm), _lib.stream_ptr()))
        model.sync_weights(force=True)

    def step(self, images: torch.Tensor, targets: torch.Tensor) -> torch.Tensor:
        """One full training step; returns the (pre-update) mean loss as a device scalar. Without a GradScaler nothing
        synchronises; with one (amp mode) the gradient norm is read back, as `scaler.step` does in the reference."""
        scaler = self.scaler
        if scaler is None or not scaler.is_enabled():
            loss = self.forward_backward(images, targets)
            self.optimizer_step()
            return loss
        scale = scaler.get_scale()
        loss = self.forward_backward(images, targets, loss_scale=scale)
        self.optimizer_step(inv_loss_scale=1.0 / scale, skip_nonfinite=True)
        found_inf = not math.isfinite(float(self._grad_norm))      # host sync (train.py:319 does the same)
        if found_inf:
            self.step_count -= 1                                    # a skipped step does not advance Adam's counter
        scaler.update(found_inf)
        return loss

    # ------------------------------------------------------------------------------------------------------------
    def state_dict(self) -> dict:
        return {"step": self.step_count, "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(),
                "lr": self.lr}

    def load_state_dict(self, state: dict) -> None:
        self.step_count = int(state["step"])
        self.exp_avg.copy_(state["exp_avg"])
        self.exp_avg_sq.copy_(state["exp_avg_sq"])
        self.lr = float(state["lr"])
