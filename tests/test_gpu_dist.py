"""-m gpu, needs >= 2 GPUs (skipped otherwise): the multi-GPU modes on REAL ranks -- one process per GPU launched with
torch.distributed.run, NCCL all-reduces over NVLink -- where tests/test_gpu_multi.py emulates the ranks on one GPU.
Run on a machine with two or more GPUs: `python -m pytest tests/test_gpu_dist.py -m gpu`."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _run(mode, world):
    port = 29500 + (os.getpid() % 500)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "dist_worker.py"), mode]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and f"DIST_OK {mode} world={world}" in p.stdout, (p.stdout[-2000:], p.stderr[-4000:])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("mode", ["dp", "pop"])
def test_real_ranks_over_nccl(mode):
    _run(mode, min(torch.cuda.device_count(), 4) if mode == "dp" else 2)
