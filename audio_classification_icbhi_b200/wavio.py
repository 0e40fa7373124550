"""Minimal RIFF/WAVE reader and writer (stdlib only) for the file-facing ends of the drop-in API.

The reference decodes with torchaudio.load (R/src/data/preprocessing.py:57) and librosa/soundfile
(R/preprocess_icbhi.py:126,166).  torchaudio >= 2.9 needs torchcodec for that and librosa /
soundfile are not in the image, so the host I/O is done here.  Values are scaled the way
torchaudio.load(normalize=True) scales integer PCM (divide by 2**(bits-1)).  This is host-side
file plumbing, not part of the measured path.
"""
from __future__ import annotations

import os
import struct
import wave
from typing import NamedTuple, Tuple

import numpy as np


def read_wav(path: str) -> Tuple[np.ndarray, int]:
    """-> (float32 [channels, frames], sample_rate).  PCM 8/16/24/32-bit and IEEE float32."""
    with open(path, "rb") as f:
        data = f.read()
    if data[:4] != b"RIFF" or data[8:12] != b"WAVE":
        raise ValueError(f"{path}: not a RIFF/WAVE file")
    pos, fmt, payload = 12, None, None
    while pos + 8 <= len(data):
        cid, size = data[pos:pos + 4], struct.unpack("<I", data[pos + 4:pos + 8])[0]
        body = data[pos + 8:pos + 8 + size]
        if cid == b"fmt ":
            fmt = struct.unpack("<HHIIHH", body[:16])
            if fmt[0] == 0xFFFE and len(body) >= 26:   # WAVE_FORMAT_EXTENSIBLE: real tag in the GUID
                fmt = (struct.unpack("<H", body[24:26])[0],) + fmt[1:]
        elif cid == b"data":
            payload = body
        pos += 8 + size + (size & 1)
    if fmt is None or payload is None:
        raise ValueError(f"{path}: missing fmt/data chunk")
    tag, channels, rate, _, _, bits = fmt
    x = _decode(path, payload, tag, bits)
    n = len(x) // channels
    return np.ascontiguousarray(x[:n * channels].reshape(n, channels).T), int(rate)


class WavInfo(NamedTuple):
    tag: int          # 1 = integer PCM, 3 = IEEE float
    channels: int
    rate: int
    bits: int
    frames: int       # samples per channel
    data_offset: int  # byte offset of the first sample in the file


def wav_info(path: str) -> WavInfo:
    """The format of a RIFF/WAVE file from its chunk headers: nothing of the sample data is read."""
    with open(path, "rb") as f:
        head = f.read(12)
        if head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            raise ValueError(f"{path}: not a RIFF/WAVE file")
        size_file = os.fstat(f.fileno()).st_size
        pos, fmt, data = 12, None, None
        while pos + 8 <= size_file:
            f.seek(pos)
            cid, size = f.read(4), struct.unpack("<I", f.read(4))[0]
            if cid == b"fmt ":
                body = f.read(min(size, 40))
                fmt = struct.unpack("<HHIIHH", body[:16])
                if fmt[0] == 0xFFFE and len(body) >= 26:   # WAVE_FORMAT_EXTENSIBLE: real tag in the GUID
                    fmt = (struct.unpack("<H", body[24:26])[0],) + fmt[1:]
            elif cid == b"data":
                data = (pos + 8, min(size, size_file - pos - 8))
            pos += 8 + size + (size & 1)
    if fmt is None or data is None:
        raise ValueError(f"{path}: missing fmt/data chunk")
    tag, channels, rate, _, _, bits = fmt
    return WavInfo(tag, channels, int(rate), bits, data[1] // (channels * (bits // 8)), data[0])


def read_wav_span(path: str, first: int, count: int) -> np.ndarray:
    """Mono samples [first, first + count) of a file, reading only those bytes.  A mono 16-bit PCM file gives its raw
    int16 samples (x / 32768 is what `read_wav` returns for them); any other encoding gives float32 scaled as `read_wav`
    scales it, channels averaged the way `AudioPreprocessor.decode_audio` averages them (torch.mean over channels)."""
    info = wav_info(path)
    first, count = int(first), int(count)
    if first < 0 or count < 0 or first + count > info.frames:
        raise ValueError(f"{path}: samples [{first}, {first + count}) outside [0, {info.frames})")
    block = info.channels * (info.bits // 8)
    with open(path, "rb") as f:
        f.seek(info.data_offset + first * block)
        payload = f.read(count * block)
    if info.channels == 1 and info.tag == 1 and info.bits == 16:
        return np.frombuffer(payload, dtype="<i2").astype(np.int16)
    x = _decode(path, payload, info.tag, info.bits).reshape(count, info.channels).T
    if info.channels == 1:
        return np.ascontiguousarray(x[0])
    import torch
    return torch.mean(torch.from_numpy(np.ascontiguousarray(x)), dim=0).numpy()


def _decode(path: str, payload: bytes, tag: int, bits: int) -> np.ndarray:
    """Interleaved sample bytes -> float32, integer PCM divided by 2**(bits-1) (8-bit: offset binary)."""
    if tag == 3 and bits == 32:
        return np.frombuffer(payload, dtype="<f4").astype(np.float32)
    if tag == 1 and bits == 16:
        return np.frombuffer(payload, dtype="<i2").astype(np.float32) / 32768.0
    if tag == 1 and bits == 32:
        return np.frombuffer(payload, dtype="<i4").astype(np.float32) / 2147483648.0
    if tag == 1 and bits == 24:
        b = np.frombuffer(payload[:len(payload) // 3 * 3], dtype=np.uint8).reshape(-1, 3).astype(np.int32)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
        v = np.where(v >= 1 << 23, v - (1 << 24), v)
        return v.astype(np.float32) / 8388608.0
    if tag == 1 and bits == 8:
        return (np.frombuffer(payload, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
    raise ValueError(f"{path}: unsupported WAV encoding (tag {tag}, {bits} bits)")


def write_wav_pcm16(path: str, samples: np.ndarray, sample_rate: int) -> None:
    """Mono float -> PCM_16, the subtype soundfile.write picks for .wav (R/preprocess_icbhi.py:166)."""
    x = np.clip(np.asarray(samples, dtype=np.float64).reshape(-1), -1.0, 1.0)
    q = np.rint(x * 32767.0).astype("<i2")
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(int(sample_rate))
        w.writeframes(q.tobytes())
