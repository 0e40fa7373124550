"""Host side of the span path, without a GPU: lm_clip_span (the native samples a clip's features read) against a
brute-force read set of the resampler's taps, wav_info / read_wav_span against read_wav, and raw(spans=True) through
forked DataLoader workers."""
import ctypes as C
import math
import struct

import numpy as np
import pytest
import torch

import audio_classification_icbhi_b200 as A
from audio_classification_icbhi_b200 import wavio
from oracle import logmel_oracle as O

RATES = [44100, 10000, 4000, 8000, 22050, 48000]   # the rate pairs of tests/golden/resample_golden.npz
PLAN_SR, T = 16000, 80000


@pytest.fixture(scope="module")
def lib():
    from audio_classification_icbhi_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


_designs = {}


def design(orig, new):
    """The tap geometry the library derives (logmel_capi.cu rs_design) restated on the float64 oracle kernel rounded
    to float32: per phase the taps with |w| > 1e-12 from k0 on, ntaps the widest phase, padded to nt4 float4."""
    if (orig, new) not in _designs:
        kern, width, o, q = O.sinc_resample_kernel(orig, new)
        w32 = kern.astype(np.float32)
        K = w32.shape[1]
        k0, ntaps = [], 1
        for p in range(q):
            nz = np.nonzero(np.abs(w32[p]) > np.float32(1e-12))[0]
            lo, hi = (int(nz[0]), int(nz[-1])) if len(nz) else (0, 0)
            k0.append(lo)
            ntaps = max(ntaps, hi - lo + 1)
        k0 = [max(0, K - ntaps) if k + ntaps > K else k for k in k0]
        nt4 = (ntaps + 3) // 4
        taps = np.zeros((q, 4 * nt4), np.float32)   # the padded taps the fmaf chain walks
        for p in range(q):
            m = min(ntaps, K - k0[p])
            taps[p, :m] = w32[p, k0[p]:k0[p] + m]
        _designs[(orig, new)] = (o, q, width, nt4, np.array(k0), taps)
    return _designs[(orig, new)]


def out_len(orig, n):
    if orig == PLAN_SR:
        return n
    o, q = design(orig, PLAN_SR)[:2]
    return (q * n + o - 1) // o


def crop_of(lp):
    return ((lp - T) // 2 if lp > T else 0), min(lp, T)


def chain_reads(orig, n):
    """Brute force: for every staged output y[crop + i], i < lc, the native indices its chain touches inside [0, n) and
    with which weight.  Returns (indices, weights) of all (output, tap) pairs."""
    o, q, width, nt4, k0, taps = design(orig, PLAN_SR)
    crop, lc = crop_of(out_len(orig, n))
    mp = np.arange(crop, crop + lc, dtype=np.int64)
    m, ph = mp // q, mp % q
    base = m * o + k0[ph] - width
    idx = base[:, None] + np.arange(4 * nt4)[None, :]
    w = taps[ph]
    keep = (idx >= 0) & (idx < n)
    return idx[keep], w[keep]


def edge_lengths(sr):
    """0 and 1 samples, L' < T, L' == T, the smallest L' > T with an odd crop, 20 s and one hour."""
    if sr == PLAN_SR:
        return [0, 1, T // 2 + 3, T, T + 1, 20 * sr, 3600 * sr]
    guess = T * sr // PLAN_SR
    cand = range(max(guess - 8, 1), guess + 16)
    eq = next(n for n in cand if out_len(sr, n) == T)
    odd = [n for n in cand if out_len(sr, n) > T and (out_len(sr, n) - T) % 2 == 1]
    return [0, 1, guess // 2 + 3, eq, (odd or [n for n in cand if out_len(sr, n) > T])[0], 20 * sr, 3600 * sr]


def span(lib, orig, n, new=PLAN_SR, target=T):
    first, count = C.c_int64(-7), C.c_int64(-7)
    assert lib.lm_clip_span(orig, new, target, n, C.byref(first), C.byref(count)) == 0
    return first.value, count.value


@pytest.mark.parametrize("sr", RATES + [PLAN_SR])
def test_clip_span_is_the_brute_force_read_set(lib, sr):
    for n in edge_lengths(sr):
        first, count = span(lib, sr, n)
        assert A.clip_span(sr, PLAN_SR, T, n) == (first, count)
        if sr == PLAN_SR:
            crop, lc = crop_of(n)
            assert (first, count) == ((crop, lc) if n else (0, 0)), n
            continue
        idx, _ = chain_reads(sr, n)
        if len(idx) == 0:
            assert (first, count) == (0, 0), n
            continue
        read = np.unique(idx)
        assert read[0] == first and read[-1] == first + count - 1, (n, first, count, read[0], read[-1])
        assert len(read) == count, "the read set is one contiguous span"


@pytest.mark.parametrize("sr", RATES)
def test_clip_span_is_minimal(lib, sr):
    """Zeroing the first sample of the span changes the float64 oracle's cropped output.  At the far end the span runs
    past the last sample a non-zero tap weighs by the float4 padding of the taps: those few samples are read with weight
    0 only (a non-finite value there still reaches the sum), and zeroing the last weighted one changes the output."""
    rs = np.random.RandomState(sr % 1000)
    for n in (20 * sr, edge_lengths(sr)[4], edge_lengths(sr)[2]):
        first, count = span(lib, sr, n)
        x = rs.standard_normal(n)
        crop, lc = crop_of(out_len(sr, n))
        ref = O.resample(x, sr, PLAN_SR)[crop:crop + lc]

        def changes(j):
            x2 = x.copy()
            x2[j] = 0.0
            return bool(np.any(O.resample(x2, sr, PLAN_SR)[crop:crop + lc] != ref))

        assert changes(first), (n, first)
        idx, w = chain_reads(sr, n)
        last_weighted = int(idx[w != 0].max())
        assert first + count - 1 - last_weighted < 8
        assert changes(last_weighted), (n, last_weighted)
        tail = (idx > last_weighted)
        assert np.all(w[tail] == 0) and int(idx.max()) == first + count - 1


def test_clip_span_rejects_bad_arguments(lib):
    f, c = C.c_int64(), C.c_int64()
    for args in ((0, 16000, T, 10), (44100, 0, T, 10), (44100, 16000, 0, 10), (44100, 16000, T, -1),
                 (16000, 16000, T, -1)):
        assert lib.lm_clip_span(*args, C.byref(f), C.byref(c)) == -1, args
    assert lib.lm_clip_span(44100, 16000, T, 10, None, C.byref(c)) == -1
    assert lib.lm_clip_span(44100, 16000, T, 10, C.byref(f), None) == -1
    with pytest.raises(RuntimeError, match="invalid argument"):
        A.clip_span(44100, 16000, T, -1)


def test_forward_spans_refuses_bad_arguments_without_a_device(lib):
    fake_plan = C.create_string_buffer(64)   # never dereferenced by the checks below
    buf = C.create_string_buffer(64)
    p = C.addressof(buf)

    def call(plan=fake_plan, rs=None, n=0, pcm16=0, B=1, **ptrs):
        a = {k: ptrs.get(k, p) for k in ("wave", "offset", "first", "stored", "length", "source", "out")}
        return lib.lm_forward_spans(plan, rs, n, a["wave"], pcm16, a["offset"], a["first"], a["stored"], a["length"],
                                    a["source"], B, None, None, a["out"], 1, None)

    assert call(plan=None) == -1
    assert call(n=-1) == -1
    assert call(n=9) == -1
    assert call(n=1, rs=None) == -1
    assert call(n=1, rs=(C.c_void_p * 1)(None)) == -1
    assert call(pcm16=2) == -1
    assert call(B=-1) == -1
    for name in ("wave", "offset", "first", "stored", "length", "source", "out"):
        assert call(**{name: None}) == -1, name
    assert call(B=0) == 0


# ---- wav files --------------------------------------------------------------------------------------------------------

def write_wav(path, x, rate, tag, bits, channels=1):
    """x: [frames, channels] float in [-1, 1)."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, channels)
    if tag == 3:
        payload = x.astype("<f4").tobytes()
    elif bits == 8:
        payload = np.clip(np.rint(x * 128 + 128), 0, 255).astype(np.uint8).tobytes()
    elif bits == 16:
        payload = np.clip(np.rint(x * 32768), -32768, 32767).astype("<i2").tobytes()
    elif bits == 32:
        payload = np.clip(np.rint(x * 2**31), -2**31, 2**31 - 1).astype("<i4").tobytes()
    else:
        v = np.clip(np.rint(x * 2**23), -2**23, 2**23 - 1).astype(np.int64).reshape(-1) & 0xFFFFFF
        payload = np.stack([v & 0xFF, (v >> 8) & 0xFF, v >> 16], axis=1).astype(np.uint8).tobytes()
    block = channels * bits // 8
    fmt = struct.pack("<HHIIHH", tag, channels, rate, rate * block, block, bits)
    extra = b"LIST" + struct.pack("<I", 5) + b"abcde\0"      # an odd-sized chunk before the data
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + extra + b"data" + struct.pack("<I", len(payload)) + payload
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


@pytest.mark.parametrize("tag,bits,channels", [(1, 8, 1), (1, 16, 1), (1, 24, 1), (1, 32, 1), (3, 32, 1), (1, 16, 2),
                                               (3, 32, 3)], ids=["pcm8", "pcm16", "pcm24", "pcm32", "float", "stereo",
                                                                 "3ch_float"])
def test_read_wav_span_is_a_slice_of_read_wav(tmp_path, tag, bits, channels):
    rs = np.random.RandomState(bits + channels)
    n = 10007
    path = str(tmp_path / "x.wav")
    write_wav(path, (rs.standard_normal((n, channels)) * 0.2).clip(-0.99, 0.99), 10000, tag, bits, channels)
    full, rate = wavio.read_wav(path)
    info = wavio.wav_info(path)
    assert (info.rate, info.channels, info.bits, info.frames) == (rate, channels, bits, n)
    mono = torch.mean(torch.from_numpy(full), dim=0).numpy()   # AudioPreprocessor.decode_audio's channel mean
    for first, count in ((0, n), (0, 0), (1, 1), (3, 5000), (n - 17, 17), (4444, 1)):
        got = wavio.read_wav_span(path, first, count)
        if (tag, bits, channels) == (1, 16, 1):
            assert got.dtype == np.int16
            got = got.astype(np.float32) / 32768.0
        else:
            assert got.dtype == np.float32
        assert got.shape == (count,)
        assert np.array_equal(got.view(np.int32), np.ascontiguousarray(mono[first:first + count]).view(np.int32))
    with pytest.raises(ValueError, match="outside"):
        wavio.read_wav_span(path, n - 3, 4)


def test_raw_span_items_through_forked_workers_without_a_gpu(tmp_path):
    """raw(spans=True) is what forked DataLoader workers run: header, span arithmetic and a partial read, no CUDA and no
    plan.  A PCM16 file comes back as its int16 samples of clip_span's span."""
    d = tmp_path / "audio_and_txt_files"
    d.mkdir()
    rs = np.random.RandomState(7)
    rates = [44100, 4000, 10000, 16000]
    secs = [20, 3, 12, 7]
    for i, (sr, s) in enumerate(zip(rates, secs)):
        wavio.write_wav_pcm16(str(d / f"{100 + i}_r.wav"), (rs.standard_normal(sr * s) * 0.1).clip(-1, 1), sr)
        (d / f"{100 + i}_r.txt").write_text("0.0\t1.0\t1\t0\n")
    cfg = {"data": dict(sample_rate=16000, n_mels=128, n_fft=2048, hop_length=512, duration=5.0)}
    ds = A.ICBHIDataset(tmp_path, "train", cfg)
    ds.data = [(str(d / f"{100 + i}_r.wav"), i % 4) for i in range(4)]
    loader = torch.utils.data.DataLoader(ds.raw(spans=True), batch_size=2, num_workers=2, collate_fn=A.raw_collate,
                                         multiprocessing_context="fork")
    got = [item for batch in loader for item in batch]
    assert ds.preprocessor._plan is None and not torch.cuda.is_initialized()
    for i, (it, sr, s) in enumerate(zip(got, rates, secs)):
        assert isinstance(it, A.SpanItem)
        assert (it.rate, it.length, it.label) == (sr, sr * s, i % 4)
        first, count = A.clip_span(sr, 16000, 80000, sr * s)
        assert it.first == first and it.samples.dtype == np.int16 and it.samples.shape == (count,)
        full, _ = wavio.read_wav(ds.data[i][0])
        assert np.array_equal(it.samples.astype(np.float32) / 32768.0, full[0, first:first + count])
    assert got[0].samples.shape[0] < 0.3 * rates[0] * secs[0]   # a 20 s 44.1 kHz recording: about a quarter is read
    assert ds.raw()[0][1] == 44100                               # the classic view is unchanged


def test_gpu_collate_refuses_span_items_cut_for_another_target(tmp_path):
    """A span item is checked against clip_span on the host before anything reaches the GPU: one cut for a 3 s target
    misses samples a 5 s preprocessor reads."""
    d = tmp_path / "audio_and_txt_files"
    d.mkdir()
    rs = np.random.RandomState(8)
    wavio.write_wav_pcm16(str(d / "100_r.wav"), (rs.standard_normal(44100 * 20) * 0.1).clip(-1, 1), 44100)
    (d / "100_r.txt").write_text("0.0\t1.0\t1\t0\n")
    cfg = {"data": dict(sample_rate=16000, n_mels=128, n_fft=2048, hop_length=512, duration=3.0)}
    ds = A.ICBHIDataset(tmp_path, "train", cfg)
    ds.data = [(str(d / "100_r.wav"), 1)]
    item = ds.raw_span_item(0)
    pre5 = A.AudioPreprocessor()
    with pytest.raises(ValueError, match="misses samples"):
        A.GpuCollate(pre5)([item])
    first, count = A.clip_span(44100, 16000, 80000, item.length)
    short = item._replace(first=first + 1, samples=np.zeros(count, np.int16))
    with pytest.raises(ValueError, match="misses samples"):
        A.GpuCollate(pre5)([short])
    assert pre5._plan is None and not torch.cuda.is_initialized()
