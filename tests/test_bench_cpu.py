"""CPU: bench.py --dump-outputs writes float32 arrays within 64 MB, and the parameter and gradient samples take the same
fixed positions on every run (stand-in tensors of the model's real arena sizes)."""
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
N_PARAMS, N_BN_STATS = 25_885_766, 53_120


def test_dump_outputs_are_float32_bounded_and_reproducible(tmp_path):
    import bench

    params = torch.arange(N_PARAMS, dtype=torch.float32)
    model = SimpleNamespace(flat_params=params, flat_grads=-params, _flat_buffers=torch.ones(N_BN_STATS))
    engine = SimpleNamespace(last_grad_norm=torch.tensor([2.5]))
    for run in ("a", "b"):
        bench.dump_step_outputs(str(tmp_path / run), model, engine, torch.tensor(0.75))
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["bn_running_stats.npy", "grad_norm.npy", "grads_sample.npy", "loss.npy", "params_sample.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 << 20
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["loss"].tolist() == [0.75] and a["grad_norm"].tolist() == [2.5]
    pos = a["params_sample"]                                                 # (positions above 2**24 round in fp32)
    assert pos.shape == (bench.DUMP_SAMPLE,) and np.all(np.diff(pos) >= 0) and pos[-1] > 0.99 * N_PARAMS
    assert np.array_equal(a["grads_sample"], -pos)                           # the same positions in both arenas
    for name, v in a.items():
        assert np.array_equal(np.load(tmp_path / "b" / f"{name}.npy"), v), name


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps" in r.stderr
