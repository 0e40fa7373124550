#!/usr/bin/env python3
"""GPU box: what a training batch costs from the files on, for whole-recording raw items (`raw()`: decode the whole file
to fp32, `GpuCollate` packs and uploads every sample, one `lm_forward_resampled`) against span items (`raw(spans=True)`:
read only the samples the features use, as int16 for PCM16 files, one int16 upload, one `lm_forward_spans`).

  1. the DESIGN.md 4.5 batch: 32 recordings of 20 s, 22 at 44.1 kHz, 5 at 10 kHz, 5 at 4 kHz;
  2. 32 segmented 16 kHz cycles of 0.2 - 16 s (the ICBHISegmentedDataset shape);
  3. the cost of the stored-span check inside the kernel: 1024 x 20 s int16 recordings resident in HBM at 44.1 / 22.05 /
     11.025 kHz (q = 160 / 320 / 640 output phases) -> 16 kHz, `forward_resampled` on the whole clips against
     `forward_spans` on the same buffer with each stored span the whole clip, CUDA events, alternated.

Per batch: GpuCollate wall time with a synchronise after each batch (medians over 4 distinct batches, the two item kinds
alternated), the sample bytes uploaded, and the worker-side time per item (`raw_item` / `raw_span_item`, files in the page
cache).  The features of the two paths are compared bit for bit.  The files are 16-bit PCM wavs written to a temporary
directory.
    python tools/span_collate_probe.py [--reps 41]
"""
import argparse
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import audio_classification_icbhi_b200 as A
from audio_classification_icbhi_b200 import wavio


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the query is informative only
        q = f"nvidia-smi unavailable ({e})"
    return f"{name}; power limit, max SM clock: {q}"


def write_batches(d, rates_secs, n_batches, seed):
    """n_batches lists of (path, label) of fresh PCM16 recordings."""
    rs = np.random.RandomState(seed)
    batches = []
    for b in range(n_batches):
        items = []
        for i, (sr, s) in enumerate(rates_secs(rs)):
            path = os.path.join(d, f"{seed}_{b}_{i}.wav")
            wavio.write_wav_pcm16(path, (rs.standard_normal(int(sr * s)) * 0.1).clip(-1, 1), sr)
            items.append((path, i % 4))
        batches.append(items)
    return batches


def probe(name, ds, batches, reps):
    collate = A.GpuCollate(ds.preprocessor)

    def items(batch, spans):
        ds.data = batch
        get = ds.raw_span_item if spans else ds.raw_item
        return [get(i) for i in range(len(batch))]

    # worker side: decode time per item, medians over the items of every batch, 3 passes
    t_item = {False: [], True: []}
    for _ in range(3):
        for batch in batches:
            for spans in (False, True):
                ds.data = batch
                get = ds.raw_span_item if spans else ds.raw_item
                for i in range(len(batch)):
                    t0 = time.perf_counter()
                    get(i)
                    t_item[spans].append((time.perf_counter() - t0) * 1e3)
    raw = {s: [items(b, s) for b in batches] for s in (False, True)}
    up_old = np.mean([sum(int(w.numel()) * 4 for w, _, _ in r) for r in raw[False]]) / 2**20
    up_new = np.mean([sum(int(it.samples.nbytes) for it in r) for r in raw[True]]) / 2**20
    for k in range(len(batches)):   # warm-up of every batch
        collate(raw[False][k]); collate(raw[True][k])
    torch.cuda.synchronize()
    t_old, t_new, same = [], [], True
    for i in range(reps):
        k = i % len(batches)
        t0 = time.perf_counter(); fo, lo = collate(raw[False][k]); torch.cuda.synchronize(); t1 = time.perf_counter()
        fn, ln = collate(raw[True][k]); torch.cuda.synchronize(); t2 = time.perf_counter()
        t_old.append((t1 - t0) * 1e3); t_new.append((t2 - t1) * 1e3)
        same &= torch.equal(fo.view(torch.int32), fn.view(torch.int32)) and torch.equal(lo, ln)
    a, b = float(np.median(t_old)), float(np.median(t_new))
    print(f"{name}")
    print(f"  GpuCollate wall + sync   whole recordings {a:8.3f} ms/batch   spans {b:8.3f} ms/batch   x{a / b:5.2f}   "
          f"bit-identical={same}")
    print(f"  samples uploaded         whole recordings {up_old:8.2f} MB/batch   spans {up_new:8.2f} MB/batch   x{up_old / up_new:5.2f}")
    print(f"  worker time per item     raw_item {np.median(t_item[False]):8.3f} ms   raw_span_item {np.median(t_item[True]):8.3f} ms   "
          f"x{np.median(t_item[False]) / np.median(t_item[True]):5.2f}", flush=True)


def span_check_cost(plan, sr, B, reps):
    from audio_classification_icbhi_b200.resample import get_resampler
    r = get_resampler(sr, 16000, plan.device)
    n = 20 * sr
    g = torch.Generator(device=plan.device).manual_seed(sr)
    x = (torch.randn(B, n, device=plan.device, generator=g) * 3000).round().to(torch.int16)
    off = torch.arange(B, device=plan.device, dtype=torch.int64) * n
    ln = torch.full((B,), n, device=plan.device, dtype=torch.int32)
    src = torch.zeros(B, dtype=torch.int32, device=plan.device)
    first = torch.zeros(B, dtype=torch.int64, device=plan.device)
    outs = [torch.empty(plan.out_shape(B), device=plan.device) for _ in range(2)]
    calls = [lambda: plan.forward_resampled(x.view(-1), off, ln, src, [r], out=outs[0]),
             lambda: plan.forward_spans(x.view(-1), off, first, ln, ln, src, [r], out=outs[1])]
    for _ in range(2):
        for c in calls:
            c()
    ts = [[], []]
    for _ in range(reps):
        for k, c in enumerate(calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); c(); e1.record()
            torch.cuda.synchronize()
            ts[k].append(e0.elapsed_time(e1))
    a, b = float(np.median(ts[0])), float(np.median(ts[1]))
    same = torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
    print(f"  {sr:6d} Hz (q = {16000 // int(np.gcd(sr, 16000)):4d})  "
          f"forward_resampled {a:8.3f} ms   forward_spans {b:8.3f} ms   spans / resampled time {b / a:6.4f}   "
          f"bit-identical={same}   ({B} x 20 s int16, {x.numel() * 2 / 2**20:.0f} MB)", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=41)
    args = ap.parse_args()
    print(card())
    print(f"torch {torch.__version__}, CUDA {torch.version.cuda}; medians of {args.reps} alternated batches")
    d = tempfile.mkdtemp(prefix="span_probe_")
    try:
        os.makedirs(os.path.join(d, "audio_and_txt_files"))
        ds = A.ICBHIDataset(d, "test")
        icbhi = lambda rs: [(sr, 20.0) for sr in [44100] * 22 + [10000] * 5 + [4000] * 5]
        probe("1. 32 x 20 s recordings (22 at 44.1 kHz, 5 at 10 kHz, 5 at 4 kHz) -> 16 kHz, 5 s crop, 2048 / 512 / 128",
              ds, write_batches(d, icbhi, 4, 1), args.reps)
        cycles = lambda rs: [(16000, float(s)) for s in rs.uniform(0.2, 16.0, 32)]
        probe("2. 32 segmented cycles at 16 kHz of 0.2 - 16 s -> 5 s pad / crop", ds, write_batches(d, cycles, 4, 2),
              args.reps)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    print("3. the stored-span check: forward_spans (each span the whole clip) against forward_resampled, resident in HBM")
    plan = A.LogMelPlan(sample_rate=16000, n_fft=2048, hop_length=512, n_mels=128, target_length=80000)
    for sr in (44100, 22050, 11025):
        span_check_cost(plan, sr, 1024, args.reps)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
