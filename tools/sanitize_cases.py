#!/usr/bin/env python3
"""Small workload for compute-sanitizer (memcheck / racecheck / initcheck): every staging path,
all four FFT sizes, several clips per CTA, clip-end normalisation, resize and PCM16 kernels."""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import audio_classification_icbhi_b200 as A

rs = np.random.RandomState(0)
def clips(lens):
    return [(rs.standard_normal(n) * 0.1).astype(np.float32) for n in lens]

p = A.AudioPreprocessor(duration=1.0)                      # 2 tiles per clip
p.plan.set("max_ctas", 2)                                  # several clips per CTA
out = p.preprocess_batch(clips([16000, 9000, 0, 16001, 40000, 16000, 1, 16000, 12345]))
p.plan.set("tma", 0)
out2 = p.preprocess_batch(clips([16000, 16000, 16000]))
pa = A.AudioPreprocessor(duration=1.0, augment=True)
pa.plan.set("max_ctas", 1)
out3 = pa.preprocess_batch(clips([16000] * 5))
out3b = pa.preprocess_batch(clips([16000] * 3), fast_augment=True)
f = A.FlexibleAudioPreprocessor(duration=0.5)              # n_fft 1024 path
f.plan.set("max_ctas", 2)
out4 = f.preprocess_batch(clips([8000, 7000, 8000, 8001, 100]))
f8 = A.FlexibleAudioPreprocessor(duration=2.048, hop_length=512)   # T % hop == 0 -> resize kernel
out5 = f8.preprocess_batch(clips([32768, 20000]))
sw = A.SlidingWindowLogMel(segment_duration=1.0, overlap=0.5, emulate_pcm16=True)
out6, _ = sw(clips([50000])[0])
small = []
for sr, n_fft, hop, n_mels in ((16000, 512, 128, 64), (4000, 256, 64, 64), (4000, 256, 50, 128)):   # 512 / 256 paths
    kw = dict(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, duration=1.0)
    ps = A.AudioPreprocessor(**kw)
    ps.plan.set("max_ctas", 2)
    small.append(ps.preprocess_batch(clips([sr, sr // 3, 0, sr + 1, 40000, 1])))
    ps.plan.set("tma", 0)
    small.append(ps.preprocess_batch(clips([sr, sr - 7])))
    psa = A.AudioPreprocessor(augment=True, **kw)
    psa.plan.set("max_ctas", 1)
    small.append(psa.preprocess_batch(clips([sr] * 3)))
    small.append(psa.preprocess_batch(clips([sr] * 3), fast_augment=True))
torch.cuda.synchronize()
for o in (out, out2, out3, out3b, out4, out5, out6, *small):
    assert torch.isfinite(o).all()
print("sanitize cases ok", [tuple(o.shape) for o in (out, out2, out3, out3b, out4, out5, out6, *small)])
