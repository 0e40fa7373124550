#!/usr/bin/env python3
"""GPU box: log-mel of clips at their native rate, fused (`lm_forward_resampled`, one launch) against the two-step
path (`lm_resample` then `lm_forward`; int16 input: `lm_pcm16_decode` first).  Both paths run on the same batches in
the same process, alternated, and their outputs are compared bit for bit.

  1. 4096 x 5 s clips resident in HBM at 44.1, 10 and 4 kHz, fp32 and int16, -> 16 kHz, n_fft 2048 / hop 512 / 128 mels.
     Two-step: one lm_resample_rows launch over the batch (all rows of one length) + one lm_forward.
  2. ICBHI-shaped: 20 s recordings at 44.1 kHz, 5 s centre crop.  The two-step path resamples whole recordings.
  3. GpuCollate wall time for batches of 32 mixed-rate host items of 20 s: the per-item path (H2D + lm_resample per
     item, pack, lm_forward) against GpuCollate, with a synchronise after each batch.  The ICBHI mix (44.1 / 10 / 4 kHz)
     is one lm_forward_resampled; a mix of 10 foreign rates and 16 kHz is more than one launch takes.

Every input set is larger than the 126 MB L2 (sizes printed).  Times: median of >= 20 launches per path.
    python tools/resampled_probe.py [--reps 21]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import audio_classification_icbhi_b200 as A
from audio_classification_icbhi_b200.resample import get_resampler

DEV = torch.device("cuda:0")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the query is informative only
        q = f"nvidia-smi unavailable ({e})"
    return f"{name}; power limit, max SM clock: {q}"


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def alternate(old, new, reps):
    for _ in range(2):   # warm-up of every shape
        old(); new()
    torch.cuda.synchronize()
    t_old, t_new = [], []
    for _ in range(reps):
        a, out_old = timed(old)
        b, out_new = timed(new)
        t_old.append(a); t_new.append(b)
    same = torch.equal(out_old.view(torch.int32), out_new.view(torch.int32))
    return float(np.median(t_old)), float(np.median(t_new)), same


def row(name, B, mb, t_old, t_new, same):
    print(f"{name:34s} B={B:5d} in={mb:8.0f} MB  two-step {t_old:8.3f} ms ({B / t_old * 1e3:11,.0f} clips/s)  "
          f"fused {t_new:8.3f} ms ({B / t_new * 1e3:11,.0f} clips/s)  x{t_old / t_new:5.2f}  bit-identical={same}",
          flush=True)


def resident(plan, sr, secs, B, pcm16, reps, name):
    r = get_resampler(sr, 16000, DEV)
    n = int(sr * secs)
    g = torch.Generator(device=DEV).manual_seed(sr)
    x = torch.randn(B, n, device=DEV, generator=g) * 0.1
    if pcm16:
        x = (x * 32767).round().clamp(-32768, 32767).to(torch.int16)
    off = torch.arange(B, device=DEV, dtype=torch.int64) * n
    ln = torch.full((B,), n, device=DEV, dtype=torch.int32)
    src = torch.zeros(B, dtype=torch.int32, device=DEV)
    n_out = r.out_len(n)
    y = torch.empty(B, n_out, device=DEV)
    xf = torch.empty(B, n, device=DEV) if pcm16 else x
    out_old = torch.empty(plan.out_shape(B), device=DEV)
    out_new = torch.empty(plan.out_shape(B), device=DEV)
    yoff = torch.arange(B, device=DEV, dtype=torch.int64) * n_out
    yln = torch.full((B,), n_out, device=DEV, dtype=torch.int32)
    lib, s = r._lib, torch.cuda.current_stream(DEV)
    import ctypes as C

    def old():
        if pcm16:
            plan.pcm16_decode(x.view(-1), out=xf.view(-1))
        A._lib.check(lib.lm_resample_rows(r._h, xf.data_ptr(), n, n, B, y.data_ptr(), n_out, C.c_void_p(s.cuda_stream)))
        return plan.forward(y.view(-1), yoff, yln, out=out_old)

    def new():
        return plan.forward_resampled(x.view(-1), off, ln, src, [r], out=out_new)

    t_old, t_new, same = alternate(old, new, reps)
    row(name, B, x.numel() * x.element_size() / 2**20, t_old, t_new, same)
    return t_old, t_new, same


def collate_wall(pre, reps, rates, name):
    rs = np.random.RandomState(3)
    batches = []
    for k in range(4):
        items = []
        for i, sr in enumerate(rates):
            items.append((torch.from_numpy((rs.standard_normal((1, int(sr * 20))) * 0.1).astype(np.float32)), sr, i % 4))
        rs.shuffle(items)
        batches.append(items)
    mb = sum(w.numel() * 4 for b in batches for w, _, _ in b) / 2**20
    collate = A.GpuCollate(pre)

    def old(batch):
        waves = [pre.resample_to_target(w, sr) for w, sr, _ in batch]
        return pre.preprocess_batch(waves)

    def new(batch):
        return collate(batch)[0]

    for b in batches:   # warm-up
        old(b); new(b)
    torch.cuda.synchronize()
    t_old, t_new, same = [], [], True
    for i in range(reps):
        b = batches[i % len(batches)]
        t0 = time.perf_counter(); fo = old(b); torch.cuda.synchronize(); t1 = time.perf_counter()
        fn = new(b); torch.cuda.synchronize(); t2 = time.perf_counter()
        t_old.append((t1 - t0) * 1e3); t_new.append((t2 - t1) * 1e3)
        same &= torch.equal(fo.view(torch.int32), fn.view(torch.int32))
    a, b = float(np.median(t_old)), float(np.median(t_new))
    print(f"{name:34s} B={len(rates):5d} in={mb:8.0f} MB  per-item {a:8.3f} ms/batch  "
          f"fused {b:8.3f} ms/batch  x{a / b:5.2f}  bit-identical={same}  (4 distinct batches, wall clock + sync)",
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--batch", type=int, default=4096)
    args = ap.parse_args()
    print(card())
    print(f"torch {torch.__version__}, CUDA {torch.version.cuda}; medians of {args.reps} alternated launches")
    plan = A.LogMelPlan(sample_rate=16000, n_fft=2048, hop_length=512, n_mels=128, target_length=80000, device=DEV)
    print("1. 5 s clips resident in HBM -> 16 kHz, 2048 / 512 / 128 mels")
    for sr in (44100, 10000, 4000):
        for pcm16 in (False, True):
            resident(plan, sr, 5, args.batch, pcm16, args.reps, f"{sr} Hz {'int16' if pcm16 else 'fp32'}")
            torch.cuda.empty_cache()
    print("2. ICBHI-shaped: 20 s recordings at 44.1 kHz, 5 s centre crop")
    resident(plan, 44100, 20, args.batch // 2, False, args.reps, "44100 Hz fp32, 20 s")
    torch.cuda.empty_cache()
    print("3. GpuCollate")
    icbhi = [44100] * 22 + [10000] * 5 + [4000] * 5   # ICBHI: most recordings at 44.1 kHz
    collate_wall(A.AudioPreprocessor(), args.reps, icbhi, "GpuCollate, 32 x 20 s host items")
    many = ([44100, 48000, 32000, 24000, 22050, 12000, 11025, 10000, 8000, 4000, 16000] * 3)[:32]
    collate_wall(A.AudioPreprocessor(), args.reps, many, "GpuCollate, 32 x 20 s at 11 rates")


if __name__ == "__main__":
    main()
