"""GPU tests of lm_forward_spans / LogMelPlan.forward_spans and of GpuCollate on span items (raw(spans=True)): clips of
which only the native samples their features read are stored.  The contract is byte-for-byte equality with
lm_forward_resampled on the whole clips when each stored span contains lm_clip_span's span, and the zero-length-clip
output, with nothing outside the stored span read, when it does not."""
import ctypes as C

import numpy as np
import pytest
import torch

import audio_classification_icbhi_b200 as A
from audio_classification_icbhi_b200 import _lib, wavio
from audio_classification_icbhi_b200.resample import get_resampler
from tests.test_gpu_resampled import (DEV, GUARD_F32, GUARD_I16, RATES, assert_bytes_equal, edge_lengths, fused, get_plan,
                                      make_clips, seeded_aug)

pytestmark = pytest.mark.gpu


def rate_args(plan, rates):
    foreign = sorted({r for r in rates if r != plan.sample_rate})
    source = torch.tensor([foreign.index(r) if r != plan.sample_rate else -1 for r in rates], dtype=torch.int32)
    return source, [get_resampler(r, plan.sample_rate, DEV) for r in foreign]


def spans_of(plan, clips, rates, rs, widen=False, short=None):
    """(lo, hi) stored per clip: clip_span's span, widened by random amounts, or one sample short at `short` ("left" /
    "right") for the clips marked True in `short`'s mask."""
    out = []
    for i, (c, r) in enumerate(zip(clips, rates)):
        n = c.numel()
        first, count = A.clip_span(r, plan.sample_rate, plan.target_length, n)
        lo, hi = first, first + count
        if widen:
            lo, hi = max(0, lo - int(rs.randint(0, 40))), min(n, hi + int(rs.randint(0, 40)))
        if short is not None and short[1][i] and count > 0:
            lo, hi = (lo + 1, hi) if short[0] == "left" else (lo, hi - 1)
        out.append((lo, hi))
    return out


def forward_spans(plan, clips, rates, pcm16, rs, spans, aug=None, noise=None, normalize=True):
    """Stored spans packed at odd offsets with guard values between them; one launch."""
    source, resamplers = rate_args(plan, rates)
    offs, pos = [], 1
    for lo, hi in spans:
        offs.append(pos)
        pos += hi - lo + 1 + int(rs.randint(0, 7))
    buf = torch.full((pos + 5,), GUARD_I16 if pcm16 else GUARD_F32, dtype=torch.int16 if pcm16 else torch.float32)
    for o, c, (lo, hi) in zip(offs, clips, spans):
        buf[o:o + hi - lo] = c[lo:hi]
    t = lambda v, dt: torch.tensor(v, dtype=dt, device=DEV)
    n0 = plan.launches
    out = plan.forward_spans(buf.to(DEV), t(offs, torch.int64), t([lo for lo, _ in spans], torch.int64),
                             t([hi - lo for lo, hi in spans], torch.int32), t([c.numel() for c in clips], torch.int32),
                             source.to(DEV), resamplers, aug=aug, noise=noise, normalize=normalize)
    assert plan.launches == n0 + 1, "one kernel launch per call"
    return out


def check_all_spans(plan, clips, rates, pcm16, rs, aug=None, noise=None, normalize=True):
    """Minimal spans and widened ones equal forward_resampled on the whole clips; one sample short on either side gives
    the zero-length clip for the clips cut short (and leaves the others alone)."""
    ref = fused(plan, clips, rates, pcm16, rs, aug=aug, noise=noise, normalize=normalize)
    for widen in (False, True):
        got = forward_spans(plan, clips, rates, pcm16, rs, spans_of(plan, clips, rates, rs, widen=widen), aug=aug,
                            noise=noise, normalize=normalize)
        assert_bytes_equal(got, ref)
    cut = np.array([c.numel() > 0 for c in clips]) & (np.arange(len(clips)) % 2 == 0)
    empty = [c[:0] if k else c for c, k in zip(clips, cut)]
    ref_cut = fused(plan, empty, rates, pcm16, rs, aug=aug, noise=noise, normalize=normalize)
    for side in ("left", "right"):
        got = forward_spans(plan, clips, rates, pcm16, rs, spans_of(plan, clips, rates, rs, short=(side, cut)), aug=aug,
                            noise=noise, normalize=normalize)
        assert_bytes_equal(got, ref_cut)


# ---- the contract ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pcm16", [False, True], ids=["fp32", "int16"])
def test_every_rate_pair_at_2048(pcm16):
    plan = get_plan(16000, 2048, 512, 128)
    rs = np.random.RandomState(31)
    lengths, rates = [], []
    for sr in RATES:
        ls = edge_lengths(sr, 16000, plan.target_length)
        lengths += ls
        rates += [sr] * len(ls)
    lengths += [0, 1, 50000, 80000, 80001, 320000]   # at the plan's rate (source -1)
    rates += [16000] * 6
    clips = make_clips(rs, lengths, pcm16)
    for normalize in (True, False):
        check_all_spans(plan, clips, rates, pcm16, rs, normalize=normalize)


@pytest.mark.parametrize("pcm16", [False, True], ids=["fp32", "int16"])
def test_one_hour_recordings(pcm16):
    plan = get_plan(16000, 2048, 512, 128)
    rs = np.random.RandomState(32)
    rates = [44100, 4000, 16000]
    clips = make_clips(rs, [3600 * r for r in rates], pcm16)
    check_all_spans(plan, clips, rates, pcm16, rs)


@pytest.mark.parametrize("plan_cfg,rates", [
    ((16000, 1024, 256, 128), [44100, 10000, 4000]),
    ((16000, 512, 128, 128), [44100, 10000, 4000]),
    ((4000, 256, 64, 64), [44100, 10000, 4000]),
], ids=["1024", "512", "256"])
@pytest.mark.parametrize("pcm16", [False, True], ids=["fp32", "int16"])
def test_other_fft_sizes(plan_cfg, rates, pcm16):
    sr, n_fft, hop, n_mels = plan_cfg
    plan = get_plan(sr, n_fft, hop, n_mels)
    rs = np.random.RandomState(33)
    lengths, rr = [], []
    for r in rates:
        ls = edge_lengths(r, sr, plan.target_length)
        lengths += ls
        rr += [r] * len(ls)
    clips = make_clips(rs, lengths, pcm16)
    check_all_spans(plan, clips, rr, pcm16, rs)
    check_all_spans(plan, clips, rr, pcm16, rs, aug=plan.upload_aug(seeded_aug(plan, len(clips), 34)))


@pytest.mark.parametrize("noise_kind", ["host", "philox"])
@pytest.mark.parametrize("pcm16", [False, True], ids=["fp32", "int16"])
def test_augmentation(noise_kind, pcm16):
    plan = get_plan(16000, 2048, 512, 128)
    rs = np.random.RandomState(35)
    rates = [44100, 10000, 4000, 16000, 44100, 22050, 16000, 48000]
    clips = make_clips(rs, [44100 * 3, 10000 * 7, 4000 * 5, 80000, 44100 * 20, 22050 * 4 + 3, 5000, 48000 * 5], pcm16)
    aug = plan.upload_aug(seeded_aug(plan, len(clips), 36))
    noise = torch.randn(len(clips), plan.target_length, device=DEV) if noise_kind == "host" else None
    for normalize in (True, False):
        check_all_spans(plan, clips, rates, pcm16, rs, aug=aug, noise=noise, normalize=normalize)


@pytest.mark.parametrize("B", [1, 3])
def test_split_batches(B):
    plan = A.LogMelPlan(sample_rate=16000, n_fft=2048, hop_length=512, n_mels=128, target_length=80000, device=DEV)
    rs = np.random.RandomState(37)
    rates = [44100, 4000, 16000][:B]
    clips = make_clips(rs, [44100 * 20, 4000 * 30, 170000][:B], False)
    aug = plan.upload_aug(seeded_aug(plan, B, 38))
    for a in (None, aug):
        check_all_spans(plan, clips, rates, False, rs, aug=a)
        plan.set("split", 1)
        check_all_spans(plan, clips, rates, False, rs, aug=a)
        plan.set("split", 0)
    plan.close()


# ---- GpuCollate on span items ---------------------------------------------------------------------------------------------

def write_recordings(tmp_path, rates, secs, seed):
    d = tmp_path / "audio_and_txt_files"
    d.mkdir()
    rs = np.random.RandomState(seed)
    for i, (sr, s) in enumerate(zip(rates, secs)):
        wavio.write_wav_pcm16(str(d / f"{100 + i}_r.wav"), (rs.standard_normal(int(sr * s)) * 0.1).clip(-1, 1), sr)
        (d / f"{100 + i}_r.txt").write_text(f"0.0\t1.0\t{i % 2}\t{(i // 2) % 2}\n")
    return [(str(d / f"{100 + i}_r.wav"), (i % 4)) for i in range(len(rates))]


def collate_both(ds, collate, lo, hi, seed=None):
    """(features, labels) of items lo..hi-1 as classic raw items and as span items, each from a fresh seed when given."""
    res = []
    for raw in (ds.raw(), ds.raw(spans=True)):
        batch = [raw[i] for i in range(lo, hi)]
        if seed is not None:
            np.random.seed(seed)
            torch.manual_seed(seed)
        res.append(collate(batch))
    return res


@pytest.mark.parametrize("cfg", [None, dict(sample_rate=4000, n_mels=64, n_fft=256, hop_length=64, duration=5.0)],
                         ids=["16k", "4k_256"])
def test_gpu_collate_spans_equal_classic_items(tmp_path, cfg):
    rates = [4000, 10000, 16000, 44100, 44100, 10000, 4000, 16000]
    secs = [20, 7.5, 5, 21.3, 3, 12, 2.5, 8]
    data = write_recordings(tmp_path, rates, secs, 41)
    ds = A.ICBHIDataset(tmp_path, "test", {"data": cfg} if cfg else None)
    ds.data = data
    span = ds.raw(spans=True)[3]
    assert span.samples.dtype == np.int16 and span.samples.shape[0] < 0.3 * span.length
    collate = A.GpuCollate(ds.preprocessor)
    plan = ds.preprocessor.plan
    for lo, hi in ((0, 4), (4, 8), (0, 8)):
        n0 = plan.launches
        (fc, lc), (fs, ls) = collate_both(ds, collate, lo, hi)
        assert plan.launches == n0 + 2   # one launch each
        assert ls.tolist() == lc.tolist() == [y for _, y in ds.data[lo:hi]]
        assert_bytes_equal(fs, fc)


def test_gpu_collate_spans_with_augmentation(tmp_path):
    rates = [44100, 4000, 16000, 10000, 44100, 16000]
    data = write_recordings(tmp_path, rates, [20, 9, 5, 30, 4, 2], 42)
    ds = A.ICBHIDataset(tmp_path, "train", None, augment=True)
    ds.data = data
    # the reference-stream draws (global numpy / torch generators) replay from a seed; fast_augment draws from a fresh
    # Generator per batch, so two calls can only be compared through forward_spans itself (test_augmentation)
    collate = A.GpuCollate(ds.preprocessor)
    (fc, _), (fs, _) = collate_both(ds, collate, 0, 6, seed=43)
    assert_bytes_equal(fs, fc)


def test_gpu_collate_spans_beyond_max_resamplers(tmp_path):
    rates = [8000, 11025, 12000, 22050, 24000, 32000, 44100, 48000, 10000, 16000, 4000, 44100]
    assert len(set(rates) - {16000}) > _lib.LM_MAX_RESAMPLERS
    data = write_recordings(tmp_path, rates, [3.3 + 2 * (i % 5) for i in range(len(rates))], 44)
    ds = A.ICBHIDataset(tmp_path, "test")
    ds.data = data
    pre = ds.preprocessor
    collate = A.GpuCollate(pre)
    n0 = pre.plan.launches
    spans = [ds.raw(spans=True)[i] for i in range(len(rates))]
    fs, ls = collate(spans)
    assert pre.plan.launches == n0 + 2   # 10 foreign rates: two groups of at most 8
    (fc, lc), _ = collate_both(ds, collate, 0, len(rates))
    assert ls.tolist() == lc.tolist()
    assert_bytes_equal(fs, fc)


def test_gpu_collate_spans_flexible_8s(tmp_path):
    rates = [44100, 4000, 16000, 10000]
    data = write_recordings(tmp_path, rates, [9.1, 4.0, 8.0, 20.0], 45)
    ds = A.ICBHIDataset(tmp_path, "test")
    ds.data = data
    ds.preprocessor = A.FlexibleAudioPreprocessor(duration=8.0)
    assert ds.preprocessor.plan.frames != ds.preprocessor.target_time_steps()   # the resize path
    collate = A.GpuCollate(ds.preprocessor)
    (fc, _), (fs, _) = collate_both(ds, collate, 0, 4)
    assert fs.shape == (4, 1, 128, ds.preprocessor.target_time_steps())
    assert_bytes_equal(fs, fc)


def test_gpu_collate_mixed_int16_and_fp32_items(tmp_path):
    data = write_recordings(tmp_path, [44100, 4000, 16000], [20, 6, 7], 46)
    ds = A.ICBHIDataset(tmp_path, "test")
    ds.data = data
    collate = A.GpuCollate(ds.preprocessor)
    spans = [ds.raw(spans=True)[i] for i in range(3)]
    as_f32 = spans[1]._replace(samples=spans[1].samples.astype(np.float32) / np.float32(32768.0))
    assert_bytes_equal(collate([spans[0], as_f32, spans[2]])[0], collate(spans)[0])
    with pytest.raises(ValueError, match="mixes"):
        collate([spans[0], ds.raw()[1]])


# ---- error paths ----------------------------------------------------------------------------------------------------------

def test_error_paths():
    plan = get_plan(16000, 2048, 512, 128)
    lib = _lib.load()
    wave = torch.zeros(1000, device=DEV)
    off = torch.zeros(1, dtype=torch.int64, device=DEV)
    first = torch.zeros(1, dtype=torch.int64, device=DEV)
    stored = torch.full((1,), 1000, dtype=torch.int32, device=DEV)
    ln = torch.full((1,), 1000, dtype=torch.int32, device=DEV)
    src = torch.zeros(1, dtype=torch.int32, device=DEV)
    out = torch.empty(plan.out_shape(1), device=DEV)
    r = get_resampler(44100, 16000, DEV)
    handles = (C.c_void_p * 9)(*([r._h.value] * 9))

    def call(arr=handles, n=1, first_p=first.data_ptr(), stored_p=stored.data_ptr()):
        return lib.lm_forward_spans(plan._h, arr, n, wave.data_ptr(), 0, off.data_ptr(), first_p, stored_p,
                                    ln.data_ptr(), src.data_ptr(), 1, None, None, out.data_ptr(), 1, None)

    assert call(n=9) == -1
    assert call(n=-1) == -1
    assert call(arr=None) == -1
    assert call(arr=(C.c_void_p * 2)(r._h.value, None), n=2) == -1
    assert call(first_p=None) == -1
    assert call(stored_p=None) == -1
    assert call() == 0
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="first must be"):
        plan.forward_spans(wave, off, first.to(torch.int32), stored, ln, src, [r])
    with pytest.raises(ValueError, match="stored must be"):
        plan.forward_spans(wave, off, first, stored.cpu(), ln, src, [r])
    with pytest.raises(ValueError, match="stored must be"):
        plan.forward_spans(wave, off, first, torch.zeros(2, dtype=torch.int32, device=DEV), ln, src, [r])
    with pytest.raises(ValueError, match="source values"):
        plan.forward_spans(wave, off, first, stored, ln, torch.tensor([1], dtype=torch.int32), [r])
    with pytest.raises(ValueError, match="plan's 16000 Hz"):
        plan.forward_spans(wave, off, first, stored, ln, src, [get_resampler(44100, 8000, DEV)])
    with pytest.raises(ValueError, match="at most 8"):
        plan.forward_spans(wave, off, first, stored, ln, src, [r] * 9)
    with pytest.raises(ValueError, match="first and stored must be given together"):
        plan.forward_resampled(wave, off, ln, src, [r], first=first)
    with pytest.raises(ValueError, match="first and stored must be given together"):
        plan.forward_resampled(wave, off, ln, src, [r], stored=stored)
