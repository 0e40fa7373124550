"""Sliding-window log-mel for the realtime analyzers, without the temp-wav round trip.

Reference: `segment_audio` (R/realtime_analyzer_parallel.py:134-161, same code in
realtime_analyzer.py:141-182, _spec.py:121-148, _timeline.py:117-144) cuts a recording into
overlapping windows, and `process_segments_batch` (:171-191) writes every window to a temporary
.wav and calls `preprocessor.preprocess(path)` on it.  Here the recording is uploaded once and
every window is an (offset, length) pair into that one device buffer: `lm_forward` pads the
short tail window with zeros and reflect-pads every window on its own, exactly as independent
clips would be.  There is no 15 s cap (:126).
"""
from __future__ import annotations

import ctypes as C
from functools import partial
from typing import List, Optional, Tuple, Union

import numpy as np
import torch

from . import _lib
from .preprocessing_flexible import FlexibleAudioPreprocessor

__all__ = ["segment_offsets", "SlidingWindowLogMel"]


def segment_offsets(n_samples: int, sample_rate: int, segment_duration: float, overlap: float
                    ) -> Tuple[np.ndarray, np.ndarray, List[Tuple[float, float]]]:
    """Window table of `segment_audio`: (start samples int64, valid lengths int32, (t0, t1) seconds).
    Full windows while start + S <= n, then one zero-padded tail window if start < n."""
    seg = int(segment_duration * sample_rate)
    hop = int(seg * (1 - overlap))
    if seg <= 0 or hop <= 0:
        raise ValueError("segment_duration and overlap must give a positive window and hop")
    n_full = 0 if n_samples < seg else (n_samples - seg) // hop + 1
    starts = np.arange(n_full, dtype=np.int64) * hop
    lengths = np.full(n_full, seg, dtype=np.int32)
    times = [(int(s) / sample_rate, (int(s) + seg) / sample_rate) for s in starts]
    tail = n_full * hop
    if tail < n_samples:
        starts = np.append(starts, np.int64(tail))
        lengths = np.append(lengths, np.int32(n_samples - tail))
        times.append((tail / sample_rate, n_samples / sample_rate))
    return starts, lengths, times


class SlidingWindowLogMel:
    """Features for every window of a recording in one batched call.

    Mirrors the preprocessor the analyzers build (R/realtime_analyzer_parallel.py:74-81):
    FlexibleAudioPreprocessor(n_fft=min(2048, int(sr*seg/2)), hop=256 if seg < 1 else 512,
    duration=seg, augment=False)."""

    def __init__(self, sample_rate: int = 16000, n_mels: int = 128, segment_duration: float = 1.0,
                 overlap: float = 0.5, emulate_pcm16: bool = False, device=None):
        self.sample_rate, self.segment_duration, self.overlap = sample_rate, segment_duration, overlap
        self.emulate_pcm16 = emulate_pcm16
        self.preprocessor = FlexibleAudioPreprocessor(
            sample_rate=sample_rate, n_mels=n_mels, n_fft=min(2048, int(sample_rate * segment_duration / 2)),
            hop_length=256 if segment_duration < 1.0 else 512, duration=segment_duration, augment=False,
            device=device)

    def windows(self, n_samples: int):
        return segment_offsets(n_samples, self.sample_rate, self.segment_duration, self.overlap)

    def __call__(self, recording: Union[torch.Tensor, np.ndarray], window_range: Optional[Tuple[int, int]] = None):
        """recording: 1-D float32 (host or device).  Returns (features [W,1,n_mels,frames] on the GPU,
        [(t0, t1)] per window).  `window_range=(lo, hi)` restricts to a shard of the windows."""
        plan = self.preprocessor.plan
        rec = torch.as_tensor(recording).reshape(-1).to(device=plan.device, dtype=torch.float32)
        starts, lengths, times = self.windows(int(rec.numel()))
        if window_range is not None:
            lo, hi = window_range
            starts, lengths, times = starts[lo:hi], lengths[lo:hi], times[lo:hi]
        if self.emulate_pcm16 and rec.numel():
            q = torch.empty_like(rec)
            _lib.check(_lib.load().lm_pcm16_roundtrip(rec.data_ptr(), q.data_ptr(), int(rec.numel()),
                                                      C.c_void_p(torch.cuda.current_stream(plan.device).cuda_stream)))
            rec = q
        if len(starts) == 0:
            return torch.empty(plan.out_shape(0), device=plan.device), times
        offset = torch.from_numpy(starts).to(plan.device)
        length = torch.from_numpy(lengths).to(plan.device)
        if rec.numel() < 4:
            rec = torch.nn.functional.pad(rec, (0, 4 - rec.numel()))
        feats = self.preprocessor._finish(plan, partial(plan.forward, rec.contiguous(), offset, length), None, None)
        return feats, times
