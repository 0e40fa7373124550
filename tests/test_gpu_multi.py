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


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_plan_and_resampler_on_another_device_keep_the_current_device():
    """Plans and resamplers live on their own device, but no call on them changes the caller's current device."""
    from audio_classification_icbhi_b200.plan import LogMelPlan
    from audio_classification_icbhi_b200.resample import Resampler

    last = torch.cuda.device_count() - 1
    torch.cuda.set_device(0)
    plan = LogMelPlan(n_fft=1024, hop_length=256, target_length=16000, device=f"cuda:{last}")
    assert torch.cuda.current_device() == 0
    B, T = 3, plan.target_length
    g = torch.Generator().manual_seed(0)
    clips = torch.randn(B * T, generator=g) * 0.1
    offset = torch.arange(B, dtype=torch.int64) * T
    length = torch.full((B,), T, dtype=torch.int32)
    want = plan.forward(clips.to(plan.device), offset.to(plan.device), length.to(plan.device))
    torch.cuda.synchronize(plan.device)
    assert torch.cuda.current_device() == 0
    got = plan.forward_host(clips, offset, length)
    assert torch.cuda.current_device() == 0
    assert torch.equal(got, want.cpu())
    plan.close()
    assert torch.cuda.current_device() == 0
    rs = Resampler(44100, 16000, device=f"cuda:{last}")
    assert torch.cuda.current_device() == 0
    rs.close()
    assert torch.cuda.current_device() == 0
