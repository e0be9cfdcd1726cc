"""Pose utilities of the hot path (reference: /root/reference/argus/utils.py:110-145,153-171,179-189)."""
from __future__ import annotations

from typing import Callable

import torch

from . import _lib


def xyzwxyz_to_xyzxyzw_SE3(xyzwxyz: torch.Tensor) -> torch.Tensor:
    """Converts 7d poses with quats from (w, x, y, z) to (x, y, z, w) order (reference: argus/utils.py:110-126)."""
    return torch.cat((xyzwxyz[..., :3], xyzwxyz[..., -3:], xyzwxyz[..., -4:-3]), dim=-1)


def xyzxyzw_to_xyzwxyz_SE3(xyzxyzw: torch.Tensor) -> torch.Tensor:
    """Converts 7d poses with quats from (x, y, z, w) to (w, x, y, z) order (reference: argus/utils.py:129-145)."""
    return torch.cat((xyzxyzw[..., :3], xyzxyzw[..., -1:], xyzxyzw[..., -4:-1]), dim=-1)


def se3_exp(pred: torch.Tensor, wxyz: bool = False) -> torch.Tensor:
    """`pp.se3(pred).Exp()` on the GPU: (..., 6) se3 [tau, phi] -> (..., 7) [t, qx, qy, qz, qw].

    With wxyz=True the quaternion is emitted scalar-first, i.e. xyzxyzw_to_xyzwxyz_SE3 is fused in."""
    if not pred.is_cuda:
        raise _lib.ArgusError("se3_exp runs on sm_100a GPUs only (no CPU fallback)")
    p = pred.detach().to(torch.float32).reshape(-1, 6).contiguous()
    out = torch.empty((p.shape[0], 7), dtype=torch.float32, device=p.device)
    with torch.cuda.device(p.device):
        _lib.call("argus_pose_exp", p, out, int(p.shape[0]), int(wxyz), _lib.stream_ptr())
    return out.reshape(*pred.shape[:-1], 7)


def get_pose(images: torch.Tensor, model: torch.nn.Module) -> torch.Tensor:
    """Get the pose of the cube from the images (reference: argus/utils.py:179-189).

    Args:
        images: The images of shape (B, 3 * n_cams, W, H), concatenated along the channel dimension.
        model: The model to use.

    Returns:
        pose: The predicted pose as a 7d pose (x, y, z, qx, qy, qz, qw). The reference returns a pypose SE3
            LieTensor; pypose is not a dependency here, so a plain (B, 7) tensor with the same data is returned.
    """
    with torch.no_grad():   # inference: se3_exp detaches anyway, and an eval-mode forward with grad builds a graph
        return se3_exp(model(images))


def time_torch_fn(fn: Callable[[], torch.Tensor]) -> tuple[torch.Tensor, float]:
    """Time a torch function with CUDA events (reference: argus/utils.py:153-171). Returns (result, seconds)."""
    start = torch.cuda.Event(enable_timing=True)
    end = torch.cuda.Event(enable_timing=True)
    start.record()
    result = fn()
    end.record()
    torch.cuda.synchronize()
    return result, start.elapsed_time(end) / 1000


def _tree_lines(path: str, extension: str, indent: str = "") -> str:
    import fnmatch
    import os

    if not os.path.isdir(path):
        return ""
    items = sorted(i for i in os.listdir(path)
                   if os.path.isdir(os.path.join(path, i)) or fnmatch.fnmatch(i, f"*.{extension}"))
    out = ""
    for k, item in enumerate(items):
        last = k == len(items) - 1
        out += indent + ("└── " if last else "├── ") + item + "\n"
        full = os.path.join(path, item)
        if os.path.isdir(full):
            out += _tree_lines(full, extension, indent + ("    " if last else "│   "))
    return out


def get_tree_string(path: str, extension: str) -> str:
    """Directory tree of `path` restricted to `*.extension` leaves, in blue (reference: argus/utils.py:197-249; used by
    the config dataclasses' error messages). A missing directory yields just the header instead of raising."""
    return "\033[94m" + path + "\n" + _tree_lines(path, extension) + "\033[0m"


def draw_spaghetti(img, n_arcs: int = 10, width_range=(1.0, 5.0)):
    """Draws random black arcs on a PIL image (reference: argus/utils.py:252-275; CPU/PIL, uses numpy's global RNG
    exactly like the reference so that `np.random.seed` reproduces it)."""
    import numpy as np
    from PIL import ImageDraw

    for _ in range(n_arcs):
        x0, y0 = np.random.randint(0, img.width), np.random.randint(0, img.height)
        x1, y1 = np.random.randint(x0, img.width), np.random.randint(y0, img.height)
        start_angle, end_angle = np.random.randint(0, 360), np.random.randint(0, 360)
        width = np.random.uniform(*width_range)
        d = ImageDraw.Draw(img)
        d.arc((x0, y0, x1, y1), start_angle, end_angle, fill=(0, 0, 0), width=int(width))
    return img


class PoseEstimator:
    """Real-time inference pipeline for `get_pose` (reference: argus/utils.py:179-189, intended to run under
    `torch.compile(mode="reduce-overhead")`, i.e. CUDA graphs — scripts/timing.py:13-45).

    The whole chain uint8 image pair(s) -> /255 + packing -> eval forward -> se3 Exp (-> optional wxyz reorder for
    MuJoCo consumers, validate_real.py:73-76) is captured once into a CUDA graph for a fixed batch shape and replayed
    per call, so a call costs one host->device copy, one graph launch and one (B,7) read-back.
    """

    def __init__(self, model, batch: int, H: int, W: int, uint8_input: bool = True, wxyz: bool = False) -> None:
        dev = model.flat_params.device
        if dev.type != "cuda":
            raise _lib.ArgusError("PoseEstimator needs the model on a CUDA device (no CPU fallback)")
        self.model = model.eval()
        self.wxyz = wxyz
        n_cams = model.n_cams
        if uint8_input:
            self.static_in = torch.zeros((batch, n_cams, H, W, 3), dtype=torch.uint8, device=dev)
        else:
            self.static_in = torch.zeros((batch, 3 * n_cams, H, W), dtype=torch.float32, device=dev)
        self.static_out = torch.zeros((batch, 7), dtype=torch.float32, device=dev)
        model.sync_weights()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(2):  # builds the launch plan and the eval-mode BN fold outside the capture
                self._run_eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self._run_eager()

    def _run_eager(self) -> None:
        pred = self.model._forward_impl(self.static_in, False)
        self.static_out.copy_(se3_exp(pred, wxyz=self.wxyz))

    def __call__(self, images: torch.Tensor) -> torch.Tensor:
        """images: same shape/dtype as the session was built for (host or device). Returns (B, 7) poses."""
        self.static_in.copy_(images, non_blocking=True)
        self.graph.replay()
        return self.static_out
