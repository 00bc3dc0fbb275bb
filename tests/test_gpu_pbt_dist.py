"""-m gpu, needs >= 2 GPUs (skipped otherwise): the exploit step of population-based training across REAL ranks (one process
per GPU, torch.distributed.run, NCCL all_to_all_single) against the unsharded population (tests/pbt_dist_worker.py)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_exploit_across_real_ranks_equals_the_unsharded_population():
    world = min(torch.cuda.device_count(), 4)
    port = 29500 + (os.getpid() % 500) + 7
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "pbt_dist_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and f"DIST_OK pbt world={world}" in p.stdout, (p.stdout[-2000:], p.stderr[-4000:])
