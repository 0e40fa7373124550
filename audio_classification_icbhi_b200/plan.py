"""LogMelPlan: Python handle on one ``lm_plan`` (include/logmel_b200.h).

The plan owns the constants ``AudioPreprocessor.__init__`` builds in the reference
(R/src/data/preprocessing.py:37-47): the periodic Hann window and the HTK mel filterbank of
``T.MelSpectrogram`` and the ``T.AmplitudeToDB`` scalars.  They are produced with the same torch
calls torchaudio makes, so the uploaded bits equal the reference's registered buffers.

torch is used for memory and streams only; all arithmetic runs in liblogmel_b200.so.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib

__all__ = ["LogMelPlan", "reference_window", "reference_filterbank", "make_aug_array", "clip_span"]


def reference_window(n_fft: int) -> torch.Tensor:
    """``torch.hann_window(n_fft)`` -- the ``window`` buffer of T.Spectrogram
    (torchaudio/transforms/_transforms.py:86-87)."""
    return torch.hann_window(n_fft, dtype=torch.float32)


def reference_filterbank(n_freqs: int, n_mels: int, sample_rate: int,
                         f_min: float = 0.0, f_max: Optional[float] = None) -> torch.Tensor:
    """``fb`` buffer of T.MelScale: melscale_fbanks(n_freqs, f_min, f_max, n_mels, sr, None, "htk")
    (torchaudio/transforms/_transforms.py:402-405).  Uses torchaudio's own builder when it
    imports (bit-identical to the reference); otherwise the same torch float32 ops in the same
    order (torchaudio/functional/functional.py:563-576)."""
    f_max = float(sample_rate // 2) if f_max is None else float(f_max)
    try:
        from torchaudio.functional import melscale_fbanks
        return melscale_fbanks(n_freqs, f_min, f_max, n_mels, sample_rate, None, "htk").to(torch.float32)
    except Exception:  # torchaudio absent: identical torch op sequence
        all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
        m_min = 2595.0 * math.log10(1.0 + f_min / 700.0)
        m_max = 2595.0 * math.log10(1.0 + f_max / 700.0)
        m_pts = torch.linspace(m_min, m_max, n_mels + 2)
        f_pts = 700.0 * (10.0 ** (m_pts / 2595.0) - 1.0)
        f_diff = f_pts[1:] - f_pts[:-1]
        slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
        down = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
        up = slopes[:, 2:] / f_diff[1:]
        return torch.max(torch.zeros(1), torch.min(down, up)).to(torch.float32)


def make_aug_array(n: int) -> np.ndarray:
    """[n] structured array laid out as ``lm_aug`` with identity defaults."""
    a = np.zeros(n, dtype=_lib.AUG_DTYPE)
    a["gain"] = 1.0
    return a


def clip_span(orig_freq: int, new_freq: int, target_len: int, length: int) -> Tuple[int, int]:
    """(first, count): the native samples [first, first + count) that the features of a clip of `length` samples at
    `orig_freq` read when a plan at `new_freq` crops to `target_len` (`lm_clip_span`).  Host arithmetic only -- no
    GPU, no CUDA call -- so DataLoader workers can read just those samples from a file for `forward_spans`."""
    first, count = C.c_int64(), C.c_int64()
    _lib.check(_lib.load().lm_clip_span(int(orig_freq), int(new_freq), int(target_len), int(length),
                                        C.byref(first), C.byref(count)))
    return first.value, count.value


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class LogMelPlan:
    """One preprocessor configuration on one GPU."""

    def __init__(self, sample_rate: int = 16000, n_fft: int = 2048, hop_length: int = 512, n_mels: int = 128,
                 target_length: int = 80000, device: Union[int, str, torch.device, None] = None,
                 db_multiplier: float = 10.0, amin: float = 1e-10, db_offset: float = 0.0,
                 norm_eps: float = 1e-8, fb: Optional[torch.Tensor] = None,
                 window: Optional[torch.Tensor] = None):
        self._lib = _lib.load()          # raises if the .so is missing
        if not torch.cuda.is_available():
            raise RuntimeError("LogMelPlan needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError(f"LogMelPlan needs a CUDA device, got {dev}")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.sample_rate, self.n_fft, self.hop_length, self.n_mels = sample_rate, n_fft, hop_length, n_mels
        self.target_length = int(target_length)
        self.n_freqs = n_fft // 2 + 1
        win = reference_window(n_fft) if window is None else window.to(torch.float32).cpu()
        fbt = reference_filterbank(self.n_freqs, n_mels, sample_rate) if fb is None else fb.to(torch.float32).cpu()
        if tuple(fbt.shape) != (self.n_freqs, n_mels) or win.numel() != n_fft:
            raise ValueError("window / fb shape mismatch")
        self._win = np.ascontiguousarray(win.numpy())
        self._fb = np.ascontiguousarray(fbt.numpy())
        cfg = _lib.LmConfig(n_fft, hop_length, n_mels, self.target_length,
                            self._win.ctypes.data_as(C.POINTER(C.c_float)),
                            self._fb.ctypes.data_as(C.POINTER(C.c_float)),
                            db_multiplier, amin, db_offset, norm_eps)
        handle = C.c_void_p()
        _lib.check(self._lib.lm_plan_create(C.byref(cfg), dev.index, C.byref(handle)))
        self._h = handle
        self.frames = self._lib.lm_plan_frames(self._h)

    # -- lifetime --------------------------------------------------------------------------
    def close(self) -> None:
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.lm_plan_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- introspection -----------------------------------------------------------------------
    def info(self) -> dict:
        i = _lib.LmInfo()
        _lib.check(self._lib.lm_plan_info(self._h, C.byref(i)))
        return {k: getattr(i, k) for k, _ in _lib.LmInfo._fields_}

    def set(self, key: str, value: int) -> None:
        _lib.check(self._lib.lm_plan_set(self._h, key.encode(), int(value)))

    @property
    def bytes_per_clip(self) -> int:
        return 4 * self.target_length + 4 * self.n_mels * self.frames

    def out_shape(self, batch: int) -> Tuple[int, int, int, int]:
        return (batch, 1, self.n_mels, self.frames)

    # -- device path -----------------------------------------------------------------------
    def _check_device_inputs(self, samples: Tuple[str, torch.Tensor, torch.dtype], offset: torch.Tensor,
                             length: torch.Tensor, aug: Optional[torch.Tensor], noise: Optional[torch.Tensor],
                             outs=(), resamplers: Optional[list] = None, source: Optional[torch.Tensor] = None,
                             first: Optional[torch.Tensor] = None, stored: Optional[torch.Tensor] = None) -> int:
        """Raises ValueError unless the tensors of one device call fit this plan; returns the batch size B.
        `samples` is (name, tensor, dtype) of the packed clips, `outs` (name, tensor or None) of the outputs;
        `forward_resampled` adds its resamplers, per-clip `source` indices and optional stored spans."""
        B = int(offset.numel())
        for name, t, dt in (samples, ("offset", offset, torch.int64), ("length", length, torch.int32)):
            if t.device != self.device or t.dtype != dt or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous {dt} tensor on {self.device}")
        if length.numel() != B:
            raise ValueError("offset / length size mismatch")
        for name, t in outs:
            if t is not None and (t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous()
                                  or t.numel() != B * self.n_mels * self.frames):
                raise ValueError(f"{name} must be contiguous fp32 [B,1,n_mels,frames] on {self.device}")
        if aug is not None and (aug.device != self.device or aug.numel() * aug.element_size() != 40 * B):
            raise ValueError("aug must hold B lm_aug records (40 bytes each) on the plan's device")
        if noise is not None and (noise.device != self.device or noise.dtype != torch.float32
                                  or noise.numel() != B * self.target_length or not noise.is_contiguous()):
            raise ValueError("noise must be contiguous fp32 [B, target_length] on the plan's device")
        if resamplers is None:
            return B
        if len(resamplers) > _lib.LM_MAX_RESAMPLERS:
            raise ValueError(f"at most {_lib.LM_MAX_RESAMPLERS} resamplers per call")
        for r in resamplers:
            if r.new_freq != self.sample_rate:
                raise ValueError(f"resampler {r.orig_freq} -> {r.new_freq} Hz does not produce the plan's {self.sample_rate} Hz")
            if torch.device("cuda", r.device.index or 0) != self.device:
                raise ValueError(f"resampler on {r.device}, plan on {self.device}")
        if source.dtype != torch.int32 or source.numel() != B or source.dim() != 1 or source.device.type not in ("cpu", "cuda") \
                or (source.is_cuda and source.device != self.device):
            raise ValueError(f"source must be an int32 [B] tensor on the host or on {self.device}")
        if B and (int(source.min()) < -1 or int(source.max()) >= len(resamplers)):
            raise ValueError(f"source values must lie in [-1, {len(resamplers)})")
        for name, t, dt in (("first", first, torch.int64), ("stored", stored, torch.int32)):
            if t is not None and (t.device != self.device or t.dtype != dt or not t.is_contiguous() or t.numel() != B):
                raise ValueError(f"{name} must be a contiguous {dt} [B] tensor on {self.device}")
        return B

    def _launch(self, fn, B: int, args: tuple, out: Optional[torch.Tensor], tail: tuple,
                stream: Optional[torch.cuda.Stream]) -> torch.Tensor:
        """The checked call fn(plan, *args, out, *tail, stream) of one device entry point.  Tensors are passed as their
        data pointers; `out` is allocated as [B, 1, n_mels, frames] when None, `stream` defaults to the current stream
        of the plan's device.  Returns `out`."""
        if out is None:
            out = torch.empty(self.out_shape(B), dtype=torch.float32, device=self.device)
        s = torch.cuda.current_stream(self.device) if stream is None else stream
        ptrs = [a.data_ptr() if isinstance(a, torch.Tensor) else a for a in (*args, out, *tail)]
        _lib.check(fn(self._h, *ptrs, C.c_void_p(s.cuda_stream)))
        return out

    def forward(self, wave: torch.Tensor, offset: torch.Tensor, length: torch.Tensor,
                aug: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None,
                normalize: bool = True, out: Optional[torch.Tensor] = None,
                out_db: Optional[torch.Tensor] = None, out_melpow: Optional[torch.Tensor] = None,
                stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """Batched log-mel on device tensors.

        wave: fp32 1-D packed samples; offset int64 [B]; length int32 [B];
        aug: uint8 [B*40] device tensor holding ``lm_aug`` records (see ``upload_aug``);
        noise: fp32 [B, target_length].  Returns ``out`` = [B, 1, n_mels, frames] fp32."""
        B = self._check_device_inputs(("wave", wave, torch.float32), offset, length, aug, noise,
                                      (("out", out), ("out_db", out_db), ("out_melpow", out_melpow)))
        return self._launch(self._lib.lm_forward, B, (wave, offset, length, B, aug, noise), out,
                            (out_db, out_melpow, 1 if normalize else 0), stream)

    def forward_pcm16(self, pcm: torch.Tensor, offset: torch.Tensor, length: torch.Tensor,
                      aug: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None,
                      normalize: bool = True, out: Optional[torch.Tensor] = None,
                      stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """`forward` on packed int16 samples (the ICBHI wav sample format; R/src/data/preprocessing.py:55-68 is
        torchaudio.load, i.e. x / 32768): one kernel, 2 bytes per sample across HBM, bit-identical to decoding
        first.  Clip starts that are multiples of 8 samples take the bulk-copy staging path."""
        B = self._check_device_inputs(("pcm", pcm, torch.int16), offset, length, aug, noise, (("out", out),))
        return self._launch(self._lib.lm_forward_pcm16, B, (pcm, offset, length, B, aug, noise), out,
                            (1 if normalize else 0,), stream)

    def forward_resampled(self, wave: torch.Tensor, offset: torch.Tensor, length: torch.Tensor, source: torch.Tensor,
                          resamplers: Sequence["Resampler"], aug: Optional[torch.Tensor] = None,
                          noise: Optional[torch.Tensor] = None, normalize: bool = True, out: Optional[torch.Tensor] = None,
                          stream: Optional[torch.cuda.Stream] = None, *, first: Optional[torch.Tensor] = None,
                          stored: Optional[torch.Tensor] = None) -> torch.Tensor:
        """`forward` on clips at their own sample rates, resampled to the plan's rate inside the kernel: one launch for
        a batch that mixes rates.  `wave` is fp32 or int16 (x / 32768) packed samples; `offset` / `length` count
        samples at the clip's own rate; `source` int32 [B] (on the host or on the plan's device) holds each clip's
        index into `resamplers` (`Resampler(clip_rate, plan.sample_rate)`, at most LM_MAX_RESAMPLERS), or -1 for a clip
        already at the plan's rate.  Bit-identical to resampling each clip with its `Resampler`, packing the results
        and calling `forward` (`forward_pcm16` for int16 clips with source -1).
        With `first` and `stored` (both or neither) only a span of each clip is stored: see `forward_spans`."""
        if (first is None) != (stored is None):
            raise ValueError("first and stored must be given together")
        if wave.dtype not in (torch.float32, torch.int16):
            raise ValueError("wave must be fp32 samples or int16 PCM")
        resamplers = list(resamplers)
        B = self._check_device_inputs(("wave", wave, wave.dtype), offset, length, aug, noise, (("out", out),),
                                      resamplers, source, first, stored)
        if not source.is_cuda:
            source = source.contiguous().to(self.device, non_blocking=True)
        source = source.contiguous()
        handles = (C.c_void_p * max(len(resamplers), 1))(*[r._h.value for r in resamplers])
        # lm_forward_spans is lm_forward_resampled's argument list with first / stored after offset
        spans = () if first is None else (first, stored)
        fn = self._lib.lm_forward_spans if spans else self._lib.lm_forward_resampled
        return self._launch(fn, B, (handles, len(resamplers), wave, 1 if wave.dtype == torch.int16 else 0, offset, *spans,
                                    length, source, B, aug, noise), out, (1 if normalize else 0,), stream)

    def forward_spans(self, wave: torch.Tensor, offset: torch.Tensor, first: torch.Tensor, stored: torch.Tensor,
                      length: torch.Tensor, source: torch.Tensor, resamplers: Sequence["Resampler"],
                      aug: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None, normalize: bool = True,
                      out: Optional[torch.Tensor] = None, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """`forward_resampled` on clips of which only a span of native samples is stored: clip i has `length[i]`
        samples, of which [first[i], first[i] + stored[i]) sit at wave[offset[i] ...].  `first` int64 [B] and `stored`
        int32 [B] live on the plan's device.  When every stored span contains `clip_span(clip rate, plan rate,
        target_length, length[i])`, the output is bit-identical to `forward_resampled` on the whole clips; a clip whose
        stored span misses a sample it needs comes out as a zero-length clip, and nothing outside the spans is read."""
        return self.forward_resampled(wave, offset, length, source, resamplers, aug, noise, normalize, out, stream,
                                      first=first, stored=stored)

    def forward_gather(self, wave: torch.Tensor, offset: torch.Tensor, length: torch.Tensor, out_slice_ptr: int,
                       peer_slice_ptrs=(), mc_slice_ptr: int = 0, aug: Optional[torch.Tensor] = None,
                       noise: Optional[torch.Tensor] = None, stream: Optional[torch.cuda.Stream] = None) -> None:
        """`forward` fused with the feature all-gather: the normalised features also go to the same slice of
        the other ranks' gathered buffers (`peer_slice_ptrs`: device addresses mapped into this process, e.g.
        `torch.distributed._symmetric_memory` buffer pointers + slice offset) or through the multicast address
        `mc_slice_ptr`.  See `sharding.FusedGather`."""
        B = self._check_device_inputs(("wave", wave, torch.float32), offset, length, aug, noise)
        peers = [int(x) for x in peer_slice_ptrs]
        arr = (C.c_void_p * max(len(peers), 1))(*peers) if peers else None
        self._launch(self._lib.lm_forward_gather, B, (wave, offset, length, B, aug, noise), C.c_void_p(int(out_slice_ptr)),
                     (arr, len(peers), C.c_void_p(int(mc_slice_ptr)) if mc_slice_ptr else None), stream)

    @property
    def launches(self) -> int:
        """Kernels launched through this plan so far (counted inside the library)."""
        return int(self._lib.lm_plan_launch_count(self._h))

    def upload_aug(self, aug: np.ndarray) -> torch.Tensor:
        """Host ``lm_aug`` structured array -> device byte tensor."""
        if aug.dtype != np.dtype(_lib.AUG_DTYPE):
            raise ValueError("aug must use the lm_aug dtype (make_aug_array)")
        raw = torch.from_numpy(np.ascontiguousarray(aug).view(np.uint8).copy())
        return raw.to(self.device, non_blocking=False)

    def forward_dense(self, clips: torch.Tensor, **kw) -> torch.Tensor:
        """Convenience: ``clips`` [B, len] (same length each) already on the device."""
        if clips.dim() != 2:
            raise ValueError("clips must be [B, len]")
        B, n = clips.shape
        clips = clips.contiguous()
        offset = torch.arange(B, device=self.device, dtype=torch.int64) * n
        length = torch.full((B,), n, device=self.device, dtype=torch.int32)
        return self.forward(clips.view(-1), offset, length, **kw)

    # -- host path (the call a reference user makes: CPU in, CPU out) ------------------------------
    def forward_host(self, wave: torch.Tensor, offset: torch.Tensor, length: torch.Tensor,
                     aug: Optional[np.ndarray] = None, noise: Optional[torch.Tensor] = None,
                     normalize: bool = True, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Host tensors in, host features out; H2D / kernel / D2H are pipelined inside the
        library on plan-owned streams.  Pinned tensors make the copies asynchronous.
        ``wave`` is fp32 samples or int16 PCM (expanded to x / 32768 inside the kernel: half the PCIe bytes)."""
        B = int(offset.numel())
        if wave.dtype not in (torch.float32, torch.int16):
            raise ValueError("wave must be fp32 samples or int16 PCM")
        for name, t, dt in (("wave", wave, wave.dtype), ("offset", offset, torch.int64), ("length", length, torch.int32)):
            if t.device.type != "cpu" or t.dtype != dt or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous CPU {dt} tensor")
        if out is None:
            out = torch.empty(self.out_shape(B), dtype=torch.float32, pin_memory=True)
        if out.device.type != "cpu" or out.dtype != torch.float32 or out.numel() != B * self.n_mels * self.frames:
            raise ValueError("out must be CPU fp32 [B,1,n_mels,frames]")
        aug_ptr = None
        if aug is not None:
            if aug.dtype != np.dtype(_lib.AUG_DTYPE) or aug.shape != (B,):
                raise ValueError("aug must be a [B] lm_aug array")
            aug = np.ascontiguousarray(aug)
            aug_ptr = aug.ctypes.data
        if noise is not None and (noise.device.type != "cpu" or noise.dtype != torch.float32
                                  or noise.numel() != B * self.target_length or not noise.is_contiguous()):
            raise ValueError("noise must be contiguous CPU fp32 [B, target_length]")
        fn = self._lib.lm_forward_host_pcm16 if wave.dtype == torch.int16 else self._lib.lm_forward_host
        _lib.check(fn(self._h, wave.data_ptr(), int(wave.numel()), offset.data_ptr(), length.data_ptr(), B, aug_ptr,
                      _ptr(noise), out.data_ptr(), 1 if normalize else 0))
        return out

    def pcm16_decode(self, pcm: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Device int16 PCM -> fp32 in [-1, 1) (x / 32768), what ``torchaudio.load`` returns for a 16-bit wav."""
        if pcm.device != self.device or pcm.dtype != torch.int16 or not pcm.is_contiguous():
            raise ValueError(f"pcm must be a contiguous int16 tensor on {self.device}")
        if out is None:
            out = torch.empty(pcm.shape, dtype=torch.float32, device=self.device)
        s = torch.cuda.current_stream(self.device)
        _lib.check(self._lib.lm_pcm16_decode(pcm.data_ptr(), out.data_ptr(), int(pcm.numel()), C.c_void_p(s.cuda_stream)))
        return out
