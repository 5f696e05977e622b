"""N>1 on real GPUs (runs only where >= 2 CUDA devices are visible)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _ngpu():
    try:
        import torch

        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_ngpu() < 2, reason="needs >= 2 GPUs")
def test_two_gpu_ba_and_pair_sharding():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29633", os.path.join(HERE, "mgpu_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    if out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-6000:])
    assert out.returncode == 0
    assert "MGPU_OK" in out.stdout
