"""Drop-in `FlexibleAudioPreprocessor` (reference: R/data/preprocessing_flexible.py:9-192).

Differences from `AudioPreprocessor`, all kept:
  * durations below 1 s shrink the transform: n_fft = min(1024, int(sr*duration/2)), hop = n_fft//4
    (:33-36);
  * `resize_spectrogram` (:118-154) sits between the dB stage and the masks: the feature map is
    bilinearly resized to max(ceil(T/hop), 32) time steps.  That is a no-op for 0.5/1/3/5 s and
    turns 251 frames into 250 for the 8 s config.

When no resize is needed the whole clip is one launch of the fused kernel; otherwise the fused
kernel stops at dB and `lm_resize_finish` (CUDA) does resize + masks + normalisation.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from .plan import LogMelPlan
from .preprocessing import AudioPreprocessor

__all__ = ["FlexibleAudioPreprocessor"]


class FlexibleAudioPreprocessor(AudioPreprocessor):
    """Audio preprocessor that handles variable segment durations."""

    flexible = True

    def __init__(self, sample_rate=16000, n_mels=128, n_fft=2048, hop_length=512, duration=5.0,
                 augment=False, min_duration=0.5, device=None):
        super().__init__(sample_rate=sample_rate, n_mels=n_mels, n_fft=n_fft, hop_length=hop_length,
                         duration=duration, augment=augment, device=device)
        self.min_duration = min_duration
        if duration < 1.0:   # adjust n_fft and hop_length for short segments
            self.n_fft = min(1024, int(sample_rate * duration / 2))
            self.hop_length = self.n_fft // 4

    @property
    def frames(self) -> int:
        return self.target_time_steps()

    def target_time_steps(self) -> int:
        return max(int(math.ceil(self.target_length / self.hop_length)), 32)

    def resize_spectrogram(self, mel_spec, target_time_steps=None):
        """Bilinear resize along time on whatever device `mel_spec` lives on
        (preprocessing_flexible.py:118-154).  GPU tensors go through `lm_resize_finish`."""
        if target_time_steps is None:
            target_time_steps = int(math.ceil(self.target_length / self.hop_length))
        target_time_steps = max(target_time_steps, 32)
        if mel_spec.shape[-1] == target_time_steps:
            return mel_spec
        squeeze = mel_spec.dim()
        x = mel_spec.reshape(-1, mel_spec.shape[-2], mel_spec.shape[-1]).to(torch.float32)
        if not x.is_cuda:
            x = x.to(self.plan.device)
        out = self._resize_finish(x.contiguous(), target_time_steps, None, normalize=False)
        out = out.to(mel_spec.device)
        if squeeze == 2:
            return out[0]
        return out.reshape(tuple(mel_spec.shape[:-1]) + (target_time_steps,))

    def _resize_finish(self, db: torch.Tensor, fout: int, aug_d, normalize: bool) -> torch.Tensor:
        lib = _lib.load()
        B, n_mels, fin = db.shape[0], db.shape[-2], db.shape[-1]
        out = torch.empty((B,) + tuple(db.shape[1:-1]) + (fout,), dtype=torch.float32, device=db.device)
        stream = torch.cuda.current_stream(db.device).cuda_stream
        _lib.check(lib.lm_resize_finish(db.data_ptr(), B, n_mels, fin, fout,
                                        None if aug_d is None else aug_d.data_ptr(), out.data_ptr(),
                                        1 if normalize else 0, 1e-8, C.c_void_p(stream)))
        return out

    def _finish(self, plan: LogMelPlan, forward, aug, noise) -> torch.Tensor:
        fout = self.target_time_steps()
        if plan.frames == fout:
            return super()._finish(plan, forward, aug, noise)
        # fused kernel up to dB with the waveform augmentation only; masks act on the resized map
        aug_d = wave_aug = None
        if aug is not None:
            aug_d = plan.upload_aug(aug)
            wave_aug = aug.copy()
            wave_aug["f0"] = wave_aug["f1"] = wave_aug["t0"] = wave_aug["t1"] = 0
        wave_aug_d, noise_d = self._upload(plan, wave_aug, noise)
        db = forward(aug=wave_aug_d, noise=noise_d, normalize=False)
        return self._resize_finish(db, fout, aug_d, normalize=True)
