"""The opt-in kernel modes kept for A/B measurements (DESIGN.md section 4) must stay correct: each is selected by an
environment variable the library reads once, so the covered tests are re-run in a child process with it set."""
import os
import subprocess
import sys
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _rerun(env_extra, selection):
    env = dict(os.environ, **env_extra)
    r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", *selection],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


def test_without_programmatic_dependent_launch(cuda_device):
    """ARGUS_PDL=0: plain stream order instead of the default programmatic edges between back-to-back kernels (they wait
    in their prologue); gradients and the reproducibility tests must not change."""
    _rerun({"ARGUS_PDL": "0"}, ["tests/test_model_gpu.py", "tests/test_train_gpu.py", "-k",
                                 "train_forward_backward or reproducible or prefetch"])


def test_fused_bn_reduction_modes(cuda_device):
    """ARGUS_BN_REDUCE_FUSED=2 (BN-backward sums in the dgrad epilogues, every eligible layer) and ARGUS_FUSED_TAIL=0
    (separate bn_apply block tail): the gradient and reproducibility tests must hold in both."""
    _rerun({"ARGUS_BN_REDUCE_FUSED": "2"}, ["tests/test_model_gpu.py", "tests/test_train_gpu.py", "-k",
                                            "train_forward_backward or reproducible or prefetch"])
    _rerun({"ARGUS_FUSED_TAIL": "0"}, ["tests/test_model_gpu.py", "tests/test_train_gpu.py", "-k",
                                       "train_forward_backward or reproducible or prefetch"])
