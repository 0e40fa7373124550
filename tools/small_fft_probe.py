#!/usr/bin/env python3
"""Throughput of the 1024- / 512- / 256-point STFT paths against the 2048 / 512 headline, and the same batches through
torchaudio on the same GPU (T.MelSpectrogram(...).cuda() -> T.AmplitudeToDB() -> per-clip (x - mean) / (std + eps)).

4096 five-second clips of N(0, 0.1^2) per configuration, resident in HBM (0.33 .. 1.31 GB, above the 126 MB L2).
Kernel and torch times: CUDA events around each launch, 5 warm-up launches, median of --reps timed launches.
One JSON object per configuration; the GPU name and power limit are read in the same run (nvidia-smi, read only).

    python tools/small_fft_probe.py [--reps 30] [--out small_fft_probe.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from audio_classification_icbhi_b200.plan import LogMelPlan  # noqa: E402

# (label, sample_rate, n_fft, hop, n_mels)
CONFIGS = [
    ("16k_1024_256_m128", 16000, 1024, 256, 128),
    ("16k_512_128_m128", 16000, 512, 128, 128),
    ("8k_512_128_m64", 8000, 512, 128, 64),
    ("4k_256_64_m64", 4000, 256, 64, 64),
    ("16k_2048_512_m128 (headline)", 16000, 2048, 512, 128),
]
B, SECONDS = 4096, 5


def gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in q.split(","))
    except Exception as e:  # the probe still reports the device name torch sees
        name, power = torch.cuda.get_device_name(0), f"unknown ({e.__class__.__name__})"
    return {"gpu": name, "power_limit": power}


def median_ms(fn, reps: int, warm: int = 5) -> float:
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    times.sort()
    return times[len(times) // 2]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("small_fft_probe: needs a CUDA device")
    import torchaudio.transforms as TT
    info = gpu_info()
    dev = torch.device("cuda", 0)
    lines = []
    for label, sr, n_fft, hop, n_mels in CONFIGS:
        T = sr * SECONDS
        plan = LogMelPlan(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, target_length=T, device=dev)
        g = torch.Generator(device=dev).manual_seed(0)
        clips = torch.randn(B, T, generator=g, device=dev) * 0.1
        offset = torch.arange(B, device=dev, dtype=torch.int64) * T
        length = torch.full((B,), T, device=dev, dtype=torch.int32)
        out = torch.empty(plan.out_shape(B), device=dev)
        flat = clips.view(-1)
        ms = median_ms(lambda: plan.forward(flat, offset, length, out=out), args.reps)

        mel = TT.MelSpectrogram(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels).to(dev)
        to_db = TT.AmplitudeToDB().to(dev)

        def torch_path():
            db = to_db(mel(clips))
            f = db.reshape(B, -1)
            return ((f - f.mean(dim=1, keepdim=True)) / (f.std(dim=1, keepdim=True) + 1e-8)).reshape(B, 1, n_mels, -1)

        with torch.no_grad():
            ref = torch_path()
            torch_ms = median_ms(torch_path, args.reps)
        max_diff = (ref - out).abs().max().item()
        rec = {"config": label, "sample_rate": sr, "n_fft": n_fft, "hop": hop, "n_mels": n_mels, "clips": B,
               "clip_seconds": SECONDS, "frames": plan.frames, "ms": round(ms, 4),
               "clips_per_s": round(B / ms * 1e3), "frames_per_s": round(B * plan.frames / ms * 1e3),
               "torch_gpu_ms": round(torch_ms, 3), "speedup_vs_torch_gpu": round(torch_ms / ms, 2),
               "max_abs_diff_vs_torch_gpu": max_diff, "timing": f"median of {args.reps} launches, CUDA events", **info}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        plan.close()
        del clips, out, ref, mel, to_db
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
