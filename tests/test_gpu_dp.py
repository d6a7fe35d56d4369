"""2-rank NCCL data-parallel correctness (needs two GPUs; one rank per GPU -- never two ranks on one device)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (one rank per GPU)")
def test_nccl_gradient_equivalence_world2():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29641", os.path.join(ROOT, "tests", "dp_equivalence.py")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    assert r.stdout.count("dp equivalence ok") == 2, r.stdout[-4000:]
