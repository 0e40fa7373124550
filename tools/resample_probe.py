#!/usr/bin/env python3
"""GPU box: throughput of the polyphase resampler, 5 s clips at the ICBHI rates -> 16 kHz, and at 384 kHz, a rate pair
whose tiled span is over 96 KB: lm_resample runs the one-output-per-thread kernel there."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from audio_classification_icbhi_b200 import get_resampler
dev = torch.device("cuda:0")
for sr in (44100, 10000, 4000, 384000):
    r = get_resampler(sr, 16000, dev)
    B = 512
    x = torch.randn(B, 5 * sr, device=dev) * 0.1
    for _ in range(2):
        y = r(x)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        y = r(x)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    print(f"{sr:6d} -> 16000: {B} x 5 s clips in {ms:8.3f} ms = {B / ms * 1e3:12,.0f} clips/s  ({ms / B * 4096:7.2f} ms per 4096 clips)")
