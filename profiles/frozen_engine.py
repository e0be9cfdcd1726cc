"""Step time of TrainEngine with frozen batch-norm statistics (frozen_bn=True) against the training step, in one run.

Per configuration, two models and two engines: one training (train-mode batch norm), one frozen. Both take uint8 image
pairs with the training loop's augmentation (the reference's kornia chain and GPU spaghetti arcs) and stage the next
batch with prefetch() while the current step runs, as bench.py times the training step. The frozen model starts from the
training model's state after the warm-up steps, so its running statistics are real ones. Blocks of --steps steps of
each kind alternate --reps times; every block is timed with CUDA events around the enqueued steps and ends in a
synchronise. Reported: the per-step time of every block and the median per kind.

Configurations: B = 256 pairs at 256 x 256 (the bench configuration) and B = 16 pairs at 256 x 256 (a fine-tuning-sized
batch). Writes one JSON object (with the device name, power limit and max SM clock read in the same run) to --out.
    python profiles/frozen_engine.py --out profiles/frozen_engine.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from input_grad import device_info  # noqa: E402


def make_batches(B: int, H: int, n: int, dev) -> list:
    g = torch.Generator().manual_seed(B)
    out = []
    for _ in range(n):
        imgs = torch.randint(0, 256, (B, 2, H, H, 3), dtype=torch.uint8, generator=g)
        q = torch.randn(B, 4, generator=g)
        t = torch.cat([torch.randn(B, 3, generator=g), q / q.norm(dim=-1, keepdim=True)], -1)
        out.append((imgs.to(dev), t.to(dev)))
    return out


def time_block(engine, batches: list, steps: int) -> float:
    """ms per step over `steps` steps with look-ahead staging, after the first batch was staged untimed."""
    ring = len(batches)
    engine.prefetch(batches[0][0])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        engine.step(*batches[i % ring])
        engine.prefetch(batches[(i + 1) % ring][0])
    e1.record()
    e1.synchronize()
    # (the batch staged by the last prefetch is never consumed: the next block of this engine stages its first batch anew)
    return e0.elapsed_time(e1) / steps


def measure(B: int, H: int, steps: int, reps: int, warmup: int) -> dict:
    from argus_b200.data import Augmentation, AugmentationConfig
    from argus_b200.engine import TrainEngine
    from argus_b200.models import NCameraCNN

    dev = torch.device("cuda", 0)
    batches = make_batches(B, H, 3, dev)
    aug = lambda: Augmentation(AugmentationConfig(), train=True, seed=42, gpu_spaghetti=True).to(dev)
    torch.manual_seed(42)
    train_model = NCameraCNN().to(dev)
    train_engine = TrainEngine(train_model, lr=1e-4, max_grad_norm=1.0, augmentation=aug(), distributed=False)
    for i in range(warmup):
        train_engine.step(*batches[i % 3])
    frozen_model = NCameraCNN().to(dev)
    frozen_model.load_state_dict(train_model.state_dict(), strict=True)
    frozen_model.eval()
    frozen_engine = TrainEngine(frozen_model, lr=1e-4, max_grad_norm=1.0, augmentation=aug(), distributed=False,
                                frozen_bn=True)
    for i in range(warmup):
        frozen_engine.step(*batches[i % 3])
    torch.cuda.synchronize()
    running0 = frozen_model._flat_buffers.clone()
    blocks = {"train": [], "frozen": []}
    for _ in range(reps):
        blocks["train"].append(round(time_block(train_engine, batches, steps), 3))
        blocks["frozen"].append(round(time_block(frozen_engine, batches, steps), 3))
    assert torch.equal(frozen_model._flat_buffers, running0), "frozen steps changed the running statistics"
    assert torch.isfinite(frozen_model.flat_params).all() and torch.isfinite(train_model.flat_params).all()
    res = {"B": B, "H": H, "W": H, "steps_per_block": steps, "blocks": reps,
           "train_step_ms_median": round(statistics.median(blocks["train"]), 3),
           "frozen_step_ms_median": round(statistics.median(blocks["frozen"]), 3),
           "train_step_ms_blocks": blocks["train"], "frozen_step_ms_blocks": blocks["frozen"]}
    res["frozen_over_train"] = round(res["frozen_step_ms_median"] / res["train_step_ms_median"], 3)
    del train_engine, frozen_engine, train_model, frozen_model, batches
    torch.cuda.empty_cache()
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 16])
    ap.add_argument("--steps", type=int, nargs="+", default=[10, 40], help="steps per block, one per batch size")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: timings are only meaningful on the B200")
    if len(args.steps) != len(args.batches):
        raise SystemExit("--steps needs one value per batch size")
    res = {"what": "TrainEngine.step with frozen batch-norm statistics (frozen_bn=True) against the training step: uint8 "
                   "input, augmentation + GPU spaghetti, look-ahead prefetch; alternating blocks, CUDA events"}
    res.update(device_info())
    res["configs"] = [measure(B, args.size, s, args.reps, args.warmup) for B, s in zip(args.batches, args.steps)]
    text = json.dumps(res, indent=1)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
