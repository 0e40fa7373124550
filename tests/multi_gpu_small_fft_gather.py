"""Launched by tests/test_gpu_small_fft.py under torchrun with one rank per GPU: the fused feature all-gather
(lm_forward_gather) at n_fft = 256 and 512 must equal lm_forward's features of every rank, bit for bit."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main() -> None:
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from audio_classification_icbhi_b200 import FusedGather, LogMelPlan

    modes = []
    for sr, n_fft, hop, n_mels in ((4000, 256, 64, 64), (16000, 512, 128, 128)):
        plan = LogMelPlan(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, target_length=5 * sr, device=dev)
        B = 333
        g = torch.Generator(device=dev).manual_seed(100 + rank)
        lens = torch.randint(100, 7 * sr, (B,), generator=g, device=dev, dtype=torch.int64)
        starts = torch.cumsum((lens + 7) // 8 * 8, 0) - (lens + 7) // 8 * 8
        wave = torch.randn(int(starts[-1] + lens[-1]) + 8, generator=g, device=dev) * 0.1
        offset, length = starts.contiguous(), lens.to(torch.int32)
        own = plan.forward(wave, offset, length)
        ref = torch.empty((world * B, 1, plan.n_mels, plan.frames), device=dev)
        dist.all_gather_into_tensor(ref, own)
        for use_mc in (True, False):
            fg = FusedGather(plan, B, use_multicast=use_mc)
            fg.full.fill_(float("nan"))
            torch.cuda.synchronize()
            dist.barrier()
            fg.run(wave, offset, length)
            full = fg.finish()
            torch.cuda.synchronize()
            assert torch.equal(full, ref), f"rank {rank}, n_fft {n_fft}: fused gather ({fg.mode}) differs from lm_forward"
            modes.append(f"{n_fft}:{fg.mode}")
    dist.barrier()
    if rank == 0:
        print("SMALL_FFT_GATHER_OK", world, "ranks;", " | ".join(modes))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
