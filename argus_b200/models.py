"""NCameraCNN on B200: same constructor, forward() contract and state_dict layout as the reference
(/root/reference/argus/models.py:13-90), with every FLOP executed by libargus_b200.so (sm_100a CUDA).

Differences that are deliberate and documented in DESIGN.md:
  * weights are randomly initialised (torchvision's defaults) — the reference downloads IMAGENET1K_V2
    (`weights="DEFAULT"`, models.py:43), which is impossible offline; `load_state_dict` accepts such a checkpoint;
  * the forward pass runs in bf16 with fp32 accumulation on the tensor cores and only exists on CUDA
    (no CPU fallback: calling the module with CPU tensors raises);
  * H and W must be powers of two >= 32 (the reference's default 256x256 and its 128x128 crop test both are).

Gradients flow to the parameters and to the input images, as with the reference: with `x.requires_grad_()`,
`loss.backward()` fills `x.grad` (the stem's transposed convolution runs on the tensor cores, argus_model_input_grad),
also when every parameter is frozen. A train-mode forward uses batch statistics. An eval-mode forward made with grad
enabled, while x or a parameter requires grad, is differentiable with the running statistics as constants
(argus_model_forward_frozen): its output is bit for bit the no-grad eval output, and it updates no running statistic
and no num_batches_tracked. This serves adversarial examples against the deployed network, fine-tuning with frozen
batch norm (also at batch size 1) and saliency maps. Under torch.no_grad() an eval-mode forward builds no graph.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass
from typing import Optional

import torch
import torch.nn as nn

from . import _lib


@dataclass(frozen=True)
class NCameraCNNConfig:
    """Configuration for the NCameraCNN model (reference: argus/models.py:13-23).

    Fields:
        n_cams: The number of cameras in the scene.
        resnet_output_dim: The output dimension of the ResNet model (before final FC layer).
    """

    n_cams: int = 2
    resnet_output_dim: int = 1024


class _Node(nn.Module):
    """Plain container used to rebuild the reference's module tree (resnet.layer1.0.conv1 ...)."""


class _BatchNormNode(nn.Module):
    eps = 1e-5
    momentum = 0.1


def _get_or_make(parent: nn.Module, name: str, cls=_Node) -> nn.Module:
    if name not in parent._modules:
        parent.add_module(name, cls())
    return parent._modules[name]


class _ModelHandle:
    """Owns the C-side `argus_model*`."""

    def __init__(self, n_cams: int, dim: int) -> None:
        self.ptr = ctypes.c_void_p()
        lib = _lib.load()
        lib.argus_model_create.restype = ctypes.c_int
        _lib.check(lib.argus_model_create(ctypes.byref(self.ptr), ctypes.c_int(n_cams), ctypes.c_int(dim)))

    def __del__(self) -> None:
        try:
            if self.ptr:
                _lib.load().argus_model_destroy(self.ptr)
                self.ptr = None
        except Exception:
            pass

    def counts(self):
        n_p, n_b = ctypes.c_int(), ctypes.c_int()
        e_p, e_b = ctypes.c_int64(), ctypes.c_int64()
        _lib.check(_lib.load().argus_model_counts(self.ptr, ctypes.byref(n_p), ctypes.byref(n_b), ctypes.byref(e_p),
                                                  ctypes.byref(e_b)))
        return n_p.value, n_b.value, e_p.value, e_b.value

    def tensor_info(self, is_buffer: bool, index: int):
        name = ctypes.create_string_buffer(128)
        off, numel, ndim = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int()
        shape = (ctypes.c_int64 * 4)()
        _lib.check(_lib.load().argus_model_tensor_info(self.ptr, ctypes.c_int(int(is_buffer)), ctypes.c_int(index), name,
                                                       ctypes.c_int(128), ctypes.byref(off), ctypes.byref(numel),
                                                       ctypes.byref(ndim), shape))
        return name.value.decode(), off.value, numel.value, tuple(shape[i] for i in range(ndim.value))

    def stage_range(self, stage: int):
        b, e = ctypes.c_int64(), ctypes.c_int64()
        _lib.check(_lib.load().argus_model_stage_range(self.ptr, ctypes.c_int(stage), ctypes.byref(b), ctypes.byref(e)))
        return b.value, e.value


class _NCameraCNNFunction(torch.autograd.Function):
    """Whole-network autograd node: forward = argus_model_forward (train mode) or argus_model_forward_frozen (eval
    mode), backward = argus_model_backward (+ argus_model_input_grad when x requires grad)."""

    @staticmethod
    def forward(ctx, model: "NCameraCNN", x: torch.Tensor, *params: torch.Tensor) -> torch.Tensor:
        training = model.training
        out = model._forward_impl(x, training, frozen=not training)
        ctx.model = model
        ctx.n_params = len(params)
        ctx.x_shape, ctx.x_dtype = x.shape, x.dtype
        return out

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        model = ctx.model
        grads = model._backward_impl(grad_out, ctx.needs_input_grad[2:])
        dx = model._input_grad_impl(ctx.x_shape).to(ctx.x_dtype) if ctx.needs_input_grad[1] else None
        return (None, dx) + tuple(grads)


class NCameraCNN(nn.Module):
    """A CNN which assumes N cameras are available in the scene (reference: argus/models.py:26-90).

    The inputs are N images of dimension HxW concatenated along the channel dimension; the outputs are 6-vectors in
    se(3) which must be sent to SE(3) via the exponential map.
    """

    def __init__(self, cfg: Optional[NCameraCNNConfig] = None) -> None:
        super().__init__()
        if cfg is None:
            cfg = NCameraCNNConfig()
        self.num_channels = 3 * cfg.n_cams
        self.resnet_output_dim = cfg.resnet_output_dim
        self.n_cams = cfg.n_cams

        self._handle = _ModelHandle(cfg.n_cams, cfg.resnet_output_dim)
        n_p, n_b, e_p, e_b = self._handle.counts()
        self._param_infos = [self._handle.tensor_info(False, i) for i in range(n_p)]
        self._buffer_infos = [self._handle.tensor_info(True, i) for i in range(n_b)]
        self._n_param_elems, self._n_buffer_elems = e_p, e_b

        flat_p = torch.zeros(e_p, dtype=torch.float32)
        flat_b = torch.zeros(e_b, dtype=torch.float32)
        n_bn = sum(1 for (name, *_rest) in self._buffer_infos if name.endswith("running_mean"))
        flat_nbt = torch.zeros(n_bn, dtype=torch.int64)
        self._build_tree(flat_p, flat_b, flat_nbt)
        self._set_flat(flat_p, flat_b, flat_nbt)
        self.reset_parameters()

        self._synced_version = -1
        self._bound_key = None
        self._flat_grads = None
        self._precision = "bf16"

    def set_precision(self, precision: str) -> "NCameraCNN":
        """"bf16" (default): tcgen05 tensor-core path. "fp32": the fp32 parity mode of the C library (same weights,
        same results layout; matches the reference's fp32 PyTorch forward / gradients to 1e-4 relative)."""
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        _lib.call("argus_model_set_precision", self._handle.ptr, 1 if precision == "fp32" else 0)
        self._precision = precision
        return self

    @property
    def precision(self) -> str:
        return self._precision

    # ------------------------------------------------------------------ module tree / flat arenas
    def _build_tree(self, flat_p, flat_b, flat_nbt) -> None:
        """Registers parameters and buffers under the reference's names, in the reference's state_dict order."""
        self._param_list: list[nn.Parameter] = []
        self._buffer_slots: list[tuple[nn.Module, str]] = []
        self._nbt_slots: list[tuple[nn.Module, str]] = []
        bn_buffers = {}
        for name, off, numel, shape in self._buffer_infos:
            bn_buffers.setdefault(name.rsplit(".", 1)[0], []).append((name, off, numel, shape))
        bn_index = 0
        seen_bn = set()
        for name, off, numel, shape in self._param_infos:
            path = name.split(".")
            mod_path, leaf = path[:-1], path[-1]
            prefix = ".".join(mod_path)
            is_bn = prefix in bn_buffers
            node: nn.Module = self
            for i, part in enumerate(mod_path):
                last = i == len(mod_path) - 1
                node = _get_or_make(node, part, _BatchNormNode if (last and is_bn) else _Node)
            p = nn.Parameter(flat_p[off:off + numel].view(shape))
            node.register_parameter(leaf, p)
            self._param_list.append(p)
            if is_bn and leaf == "bias" and prefix not in seen_bn:
                seen_bn.add(prefix)
                for bname, boff, bnumel, bshape in bn_buffers[prefix]:
                    bleaf = bname.rsplit(".", 1)[1]
                    node.register_buffer(bleaf, flat_b[boff:boff + bnumel].view(bshape))
                    self._buffer_slots.append((node, bleaf))
                node.register_buffer("num_batches_tracked", flat_nbt[bn_index])
                self._nbt_slots.append((node, "num_batches_tracked"))
                bn_index += 1

    def _set_flat(self, flat_p, flat_b, flat_nbt) -> None:
        """Makes every parameter / buffer a view into the given flat arenas (values must already be in place)."""
        self._flat_params, self._flat_buffers, self._flat_nbt = flat_p, flat_b, flat_nbt
        for p, (_name, off, numel, shape) in zip(self._param_list, self._param_infos):
            p.data = flat_p[off:off + numel].view(shape)
        for (node, leaf), (_name, off, numel, shape) in zip(self._buffer_slots, self._buffer_infos):
            node._buffers[leaf] = flat_b[off:off + numel].view(shape)
        for i, (node, leaf) in enumerate(self._nbt_slots):
            node._buffers[leaf] = flat_nbt[i]
        self._bound_key = None
        self._synced_version = -1

    def _apply(self, fn, recurse=True):
        """Module.to()/cuda()/cpu(): move tensor by tensor, then re-pack everything into fresh flat arenas."""
        super()._apply(fn, recurse)
        dev = self._param_list[0].device
        for p in self._param_list:
            if p.dtype != torch.float32:
                raise TypeError("argus_b200.NCameraCNN keeps fp32 master parameters; bf16 copies are internal")
        flat_p = torch.zeros(self._n_param_elems, dtype=torch.float32, device=dev)
        flat_b = torch.zeros(self._n_buffer_elems, dtype=torch.float32, device=dev)
        flat_nbt = torch.zeros(len(self._nbt_slots), dtype=torch.int64, device=dev)
        with torch.no_grad():
            for p, (_n, off, numel, shape) in zip(self._param_list, self._param_infos):
                flat_p[off:off + numel].view(shape).copy_(p.data)
            for (node, leaf), (_n, off, numel, shape) in zip(self._buffer_slots, self._buffer_infos):
                flat_b[off:off + numel].view(shape).copy_(node._buffers[leaf])
            for i, (node, leaf) in enumerate(self._nbt_slots):
                flat_nbt[i] = node._buffers[leaf]
        self._set_flat(flat_p, flat_b, flat_nbt)
        self._flat_grads = None
        return self

    def reset_parameters(self) -> None:
        """torchvision resnet50 / nn.Linear default initialisation (kaiming-normal fan_out convs, BN weight 1,
        bias 0, Linear kaiming-uniform(a=sqrt(5)))."""
        with torch.no_grad():
            for p, (name, _off, _numel, shape) in zip(self._param_list, self._param_infos):
                leaf = name.rsplit(".", 1)[1]
                if len(shape) == 4:
                    nn.init.kaiming_normal_(p, mode="fan_out", nonlinearity="relu")
                elif len(shape) == 2:
                    nn.init.kaiming_uniform_(p, a=math.sqrt(5))
                elif name.startswith("resnet.fc") or name.startswith("output_mlp"):
                    fan_in = {"resnet.fc.bias": 2048, "output_mlp.0.bias": self.n_cams * self.resnet_output_dim,
                              "output_mlp.2.bias": 128, "output_mlp.4.bias": 128}[name]
                    bound = 1 / math.sqrt(fan_in)
                    nn.init.uniform_(p, -bound, bound)
                elif leaf == "weight":
                    p.fill_(1.0)
                else:
                    p.zero_()
            for (node, leaf), _info in zip(self._buffer_slots, self._buffer_infos):
                node._buffers[leaf].fill_(1.0 if leaf == "running_var" else 0.0)
            self._flat_nbt.zero_()

    # ------------------------------------------------------------------ C-side binding
    @property
    def flat_params(self) -> torch.Tensor:
        return self._flat_params

    @property
    def flat_grads(self) -> torch.Tensor:
        self._ensure_bound()
        return self._flat_grads

    def stage_ranges(self) -> list[tuple[int, int]]:
        """Parameter-arena element ranges whose gradients are final after backward stage 0, 1, 2, 3."""
        return [self._handle.stage_range(s) for s in range(4)]

    def _ensure_bound(self) -> None:
        fp = self._flat_params
        if not fp.is_cuda:
            raise _lib.ArgusError("argus_b200.NCameraCNN runs on sm_100a GPUs only: move the module to CUDA "
                                  "(there is no CPU fallback)")
        key = (fp.data_ptr(), self._flat_buffers.data_ptr())
        if self._bound_key != key:
            if self._flat_grads is None or self._flat_grads.device != fp.device:
                self._flat_grads = torch.zeros_like(fp)
            with torch.cuda.device(fp.device):
                _lib.call("argus_model_bind", self._handle.ptr, fp, self._flat_grads, self._flat_buffers)
            self._bound_key = key
            self._synced_version = -1

    def _state_version(self) -> int:
        """Monotone fingerprint of every in-place update to a parameter or buffer. After `_set_flat` each Parameter /
        buffer is a separate view object with its OWN version counter (`p.data = view` detaches it from the flat
        tensor's counter), so updates made through the module tree -- `load_state_dict`, `torch.optim.*.step()` on
        `model.parameters()`, manual `p.data` edits, running-stat edits -- are only visible on the views."""
        v = self._flat_params._version + self._flat_buffers._version
        for p in self._param_list:
            v += p._version
        for node, leaf in self._buffer_slots:
            v += node._buffers[leaf]._version
        return v

    def sync_weights(self, force: bool = False) -> None:
        """Refresh the packed bf16 weights (and mark the eval-mode BN fold dirty) if any parameter or buffer changed
        since the last sync. Updates made by the library itself (TrainEngine's fused optimizer, running statistics of a
        training forward) do not go through torch and are handled on the C side / by `force=True`."""
        self._ensure_bound()
        v = self._state_version()
        if force or v != self._synced_version:
            _lib.call("argus_model_sync_weights", self._handle.ptr, _lib.stream_ptr())
            self._synced_version = v

    def mark_dirty(self) -> None:
        """Force a re-pack on the next forward (for edits torch cannot see, e.g. raw pointer writes into the arenas)."""
        self._synced_version = -1

    def _forward_impl(self, x: torch.Tensor, training: bool, aug_params: Optional[torch.Tensor] = None,
                      augment: bool = False, arc_mask: Optional[torch.Tensor] = None,
                      plasma_ws: Optional[torch.Tensor] = None, frozen: bool = False) -> torch.Tensor:
        """frozen (eval mode only): the differentiable eval-mode forward, argus_model_forward_frozen."""
        self._ensure_bound()
        if x.device != self._flat_params.device:
            raise _lib.ArgusError(f"input is on {x.device} but the model is on {self._flat_params.device}")
        is_u8 = x.dtype == torch.uint8
        if is_u8:
            # (B, n_cams, H, W, 3) uint8 HWC, the decoded-PNG layout
            assert x.dim() == 5 and x.shape[1] == self.n_cams and x.shape[-1] == 3
            B, _, H, W, _ = x.shape
        else:
            B, C, H, W = x.shape
            if C != self.num_channels:
                raise ValueError(f"expected {self.num_channels} channels, got {C}")
            x = x.to(torch.float32)
        x = x.contiguous()
        self.sync_weights()
        out = torch.empty((B, 6), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            if frozen:
                _lib.call("argus_model_forward_frozen", self._handle.ptr, x, int(is_u8), int(B), int(H), int(W), out,
                          _lib.stream_ptr())
            elif is_u8 and (augment or arc_mask is not None):
                # fused staging: arcs (bit mask) + augmentation (when `augment`) + /255 + bf16 space-to-depth packing
                if augment and plasma_ws is None:
                    plasma_ws = torch.empty((B * self.n_cams, H, W // 32), dtype=torch.int32, device=x.device)
                _lib.call("argus_model_stage_input_u8", self._handle.ptr, x, aug_params, arc_mask, plasma_ws, int(B),
                          int(H), int(W), int(training), int(augment), _lib.stream_ptr())
                _lib.call("argus_model_forward", self._handle.ptr, None, 0, int(B), int(H), int(W), int(training), out,
                          _lib.stream_ptr())
            else:
                _lib.call("argus_model_forward", self._handle.ptr, x, int(is_u8), int(B), int(H), int(W), int(training),
                          out, _lib.stream_ptr())
        if training:
            self._flat_nbt += 1
        return out

    def _forward_staged(self, B: int, H: int, W: int) -> torch.Tensor:
        """Training forward over a batch already staged by argus_model_stage_input_u8 (TrainEngine.prefetch)."""
        self._ensure_bound()
        self.sync_weights()
        dev = self._flat_params.device
        out = torch.empty((B, 6), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.call("argus_model_forward", self._handle.ptr, None, 0, int(B), int(H), int(W), 1, out, _lib.stream_ptr())
        self._flat_nbt += 1
        return out

    def _backward_impl(self, grad_out: torch.Tensor, needs_grad=None) -> list[Optional[torch.Tensor]]:
        """Parameter gradients of the last training or frozen forward; None for parameters whose `needs_grad` entry is
        False."""
        g = grad_out.contiguous().to(torch.float32)
        with torch.cuda.device(g.device):
            _lib.call("argus_model_zero_grads", self._handle.ptr, _lib.stream_ptr())
            _lib.call("argus_model_backward", self._handle.ptr, g, 0, 4, _lib.stream_ptr())
        fg = self._flat_grads
        if needs_grad is None:
            needs_grad = [True] * len(self._param_infos)
        return [fg[off:off + numel].view(shape).clone() if need else None
                for need, (_n, off, numel, shape) in zip(needs_grad, self._param_infos)]

    def _input_grad_impl(self, shape) -> torch.Tensor:
        """d loss / d x (fp32, `shape` = the input's) of the last training or frozen forward, after _backward_impl."""
        dx = torch.empty(shape, dtype=torch.float32, device=self._flat_params.device)
        with torch.cuda.device(dx.device):
            _lib.call("argus_model_input_grad", self._handle.ptr, dx, _lib.stream_ptr())
        return dx

    def probe_activation(self, index: int) -> torch.Tensor:
        """Test probe: activation of the last forward as a (rows, C) bf16 tensor (NHWC rows).
        index -1: pooled stem output, 0..15: bottleneck outputs, 16: pooled features, 17: resnet.fc output,
        100..115: act2 (the input of conv3) of each bottleneck."""
        self._ensure_bound()
        dev = self._flat_params.device
        cap = 1 << 28
        rows, C = ctypes.c_int64(), ctypes.c_int()
        # first ask for the size with a generous upper bound, then trim
        buf = torch.empty(cap, dtype=torch.bfloat16, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().argus_model_copy_activation(self._handle.ptr, ctypes.c_int(index), _lib.ptr(buf),
                                                               ctypes.c_int64(cap), ctypes.byref(rows),
                                                               ctypes.byref(C), _lib.stream_ptr()))
        return buf[: rows.value * C.value].view(rows.value, C.value).clone()

    # ------------------------------------------------------------------ public forward
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """Forward pass through the CNN (reference: argus/models.py:66-90).

        Args:
            x: The input images of shape (B, 3 * n_cams, H, W), concatenated along the channel dimension.

        Returns:
            pose: The predicted pose of the cube in the scene expressed in se(3).
        """
        assert len(x.shape) == 4 or x.dtype == torch.uint8, \
            "The input images must be of shape (B, C, H, W)! If B=1, add a dummy dimension."
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self._param_list)):
            return _NCameraCNNFunction.apply(self, x, *self._param_list)
        return self._forward_impl(x, self.training)
