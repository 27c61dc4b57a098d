"""GPU, >= 2 devices: feature-sharded fit over NCCL must reproduce the oracle (and the 1-GPU model)."""
import pytest

from test_dist_host_logic import run_workers

pytestmark = pytest.mark.gpu


def test_feature_sharded_fit_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = run_workers("nccl", 2, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert r.stdout.count("worst=") == 18  # (3 NIPALS + 6 other-method cases) x 2 ranks
    assert r.stdout.count("fold-parallel CV ok") == 2
