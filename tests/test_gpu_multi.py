"""Multi-GPU checks that need more than one B200 (skipped on a single-GPU machine): run with
`python -m pytest tests/test_gpu_multi.py -m gpu` on a machine with two or more B200s."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_fused_gather_matches_nccl_all_gather():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.join(ROOT, "tests", "multi_gpu_fused_gather.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "FUSED_GATHER_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
