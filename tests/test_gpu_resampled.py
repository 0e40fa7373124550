"""GPU tests of lm_forward_resampled / LogMelPlan.forward_resampled: clips at their own sample rates resampled inside the
log-mel kernel's staging.  The contract is byte-for-byte equality with the two-step composition users ran before:
per-clip `Resampler` (lm_resample), pack, `forward` -- and, for clips already at the plan's rate (source -1), with
`forward` / `forward_pcm16` on their own.  Plus the drop-in paths built on it (preprocess_batch(sample_rates=...),
FlexibleAudioPreprocessor, GpuCollate) and torchaudio on the CPU as an outside reference."""
import ctypes as C

import numpy as np
import pytest
import torch

import audio_classification_icbhi_b200 as A
from audio_classification_icbhi_b200 import _lib, wavio
from audio_classification_icbhi_b200.resample import get_resampler
from oracle import logmel_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RATES = [44100, 10000, 4000, 8000, 22050, 48000]
UNTILED_RATE = 384000   # its tiled span (99.6 KB) is over 96 KB: lm_resample runs the one-output-per-thread kernel
GUARD_F32 = 1.0e6      # fills the gaps between packed clips: a read outside a clip would show up in every feature
GUARD_I16 = 32767

_plans = {}


def get_plan(sr, n_fft, hop, n_mels, T=None):
    T = 5 * sr if T is None else T
    key = (sr, n_fft, hop, n_mels, T)
    if key not in _plans:
        _plans[key] = A.LogMelPlan(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, target_length=T, device=DEV)
    return _plans[key]


def out_len(sr, plan_sr, n):
    return get_resampler(sr, plan_sr, DEV).out_len(n)


def edge_lengths(sr, plan_sr, T):
    """Native lengths of 0 and 1 samples, L' < T, L' == T, the smallest L' > T with an odd crop (or the smallest L' > T
    when the rate pair cannot reach one), and a 20 s recording."""
    guess = T * sr // plan_sr
    cand = range(max(guess - 8, 1), guess + 16)
    eq = next(n for n in cand if out_len(sr, plan_sr, n) == T) if sr != plan_sr else T
    over = [n for n in cand if out_len(sr, plan_sr, n) > T]
    odd = [n for n in over if (out_len(sr, plan_sr, n) - T) % 2 == 1]
    return [0, 1, guess // 2 + 3, eq, (odd or over)[0], 20 * sr]


def make_clips(rs, lengths, pcm16):
    if pcm16:
        return [torch.from_numpy(rs.randint(-20000, 20000, n).astype(np.int16)) for n in lengths]
    return [torch.from_numpy((rs.standard_normal(n) * 0.1).astype(np.float32)) for n in lengths]


def pack_unaligned(rs, clips, pcm16):
    """Clips at odd offsets with guard values around each one."""
    offs, pos = [], 1
    for c in clips:
        offs.append(pos)
        pos += c.numel() + 1 + int(rs.randint(0, 7))
    dt = torch.int16 if pcm16 else torch.float32
    buf = torch.full((pos + 5,), GUARD_I16 if pcm16 else GUARD_F32, dtype=dt)
    for o, c in zip(offs, clips):
        buf[o:o + c.numel()] = c
    return (buf.to(DEV), torch.tensor(offs, dtype=torch.int64, device=DEV),
            torch.tensor([c.numel() for c in clips], dtype=torch.int32, device=DEV))


def fused(plan, clips, rates, pcm16, rs, aug=None, noise=None, normalize=True):
    foreign = sorted({r for r in rates if r != plan.sample_rate})
    resamplers = [get_resampler(r, plan.sample_rate, DEV) for r in foreign]
    source = torch.tensor([foreign.index(r) if r != plan.sample_rate else -1 for r in rates], dtype=torch.int32)
    wave, off, ln = pack_unaligned(rs, clips, pcm16)
    n0 = plan.launches
    out = plan.forward_resampled(wave, off, ln, source.to(DEV), resamplers, aug=aug, noise=noise, normalize=normalize)
    assert plan.launches == n0 + 1, "one kernel launch per call"
    return out


def two_step(plan, clips, rates, aug=None, noise=None, normalize=True):
    """The composition the fused path replaces: decode, lm_resample per clip, pack (4-aligned), lm_forward."""
    ys = []
    for c, r in zip(clips, rates):
        x = c.float() / 32768.0 if c.dtype == torch.int16 else c
        x = x.to(DEV)
        ys.append(x if r == plan.sample_rate else get_resampler(r, plan.sample_rate, DEV)(x))
    offs, pos = [], 0
    for y in ys:
        offs.append(pos)
        pos += (y.numel() + 3) & ~3
    buf = torch.zeros(max(pos, 4), dtype=torch.float32, device=DEV)
    for o, y in zip(offs, ys):
        buf[o:o + y.numel()] = y
    off = torch.tensor(offs, dtype=torch.int64, device=DEV)
    ln = torch.tensor([y.numel() for y in ys], dtype=torch.int32, device=DEV)
    return plan.forward(buf, off, ln, aug=aug, noise=noise, normalize=normalize)


def assert_bytes_equal(a, b):
    a, b = a.cpu(), b.cpu()
    assert a.shape == b.shape
    same = torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert same, f"max |diff| {float((a - b).abs().max())}, differing {(a != b).sum().item()} of {a.numel()}"


def seeded_aug(plan, B, seed, noise_on=True):
    rs = np.random.RandomState(seed)
    a = A.make_aug_array(B)
    a["shift"] = rs.randint(-plan.target_length // 5, plan.target_length // 5, B)
    a["gain"] = rs.uniform(0.5, 1.5, B).astype(np.float32)
    a["noise_scale"] = np.where(rs.rand(B) < 0.7, 0.005, 0.0) if noise_on else 0.0
    a["f0"] = rs.randint(0, plan.n_mels // 2, B)
    a["f1"] = a["f0"] + rs.randint(0, 15, B)
    a["t0"] = rs.randint(0, plan.frames // 2, B)
    a["t1"] = a["t0"] + rs.randint(0, 35, B)
    a["seed"] = rs.randint(1, 2**62, B, dtype=np.int64).astype(np.uint64)
    a[0] = A.make_aug_array(1)[0]   # one un-augmented clip: its silent tiles are skipped
    return a


# ---- the contract: every rate pair, edge lengths, both sample formats -------------------------------------------------

@pytest.mark.parametrize("pcm16", [False, True], ids=["fp32", "int16"])
@pytest.mark.parametrize("n_fft,hop,n_mels", [(2048, 512, 128)])
def test_rate_pairs_and_edge_lengths_equal_two_step(n_fft, hop, n_mels, pcm16):
    plan = get_plan(16000, n_fft, hop, n_mels)
    rs = np.random.RandomState(11)
    lengths, rates = [], []
    for sr in RATES + [UNTILED_RATE]:
        ls = edge_lengths(sr, 16000, plan.target_length)
        lengths += ls
        rates += [sr] * len(ls)
    lengths += [0, 1, 50000, 80000, 80001, 200001]   # clips at the plan's rate (source -1)
    rates += [16000] * 6
    clips = make_clips(rs, lengths, pcm16)
    for normalize in (True, False):
        got = fused(plan, clips, rates, pcm16, rs, normalize=normalize)
        assert_bytes_equal(got, two_step(plan, clips, rates, normalize=normalize))


@pytest.mark.parametrize("pcm16", [False, True], ids=["fp32", "int16"])
def test_source_minus_one_equals_plain_forward(pcm16):
    plan = get_plan(16000, 2048, 512, 128)
    rs = np.random.RandomState(12)
    lengths = [80000, 31000, 123457, 44100 * 5, 17, 10000 * 5]
    rates = [16000, 16000, 16000, 44100, 16000, 10000]
    clips = make_clips(rs, lengths, pcm16)
    got = fused(plan, clips, rates, pcm16, rs)
    assert_bytes_equal(got, two_step(plan, clips, rates))
    for i, r in enumerate(rates):
        if r != 16000:
            continue
        wave, off, ln = pack_unaligned(rs, [clips[i]], pcm16)
        own = plan.forward_pcm16(wave, off, ln) if pcm16 else plan.forward(wave, off, ln)
        assert_bytes_equal(got[i:i + 1], own)


@pytest.mark.parametrize("noise_kind", ["host", "philox"])
@pytest.mark.parametrize("normalize", [True, False])
def test_augmentation_equals_two_step(noise_kind, normalize):
    plan = get_plan(16000, 2048, 512, 128)
    rs = np.random.RandomState(13)
    rates = [44100, 10000, 4000, 16000, 44100, 22050, 16000, 48000]
    lengths = [44100 * 3, 10000 * 7, 4000 * 5, 80000, 44100 * 20, 22050 * 4 + 3, 5000, 48000 * 5]
    clips = make_clips(rs, lengths, False)
    aug = plan.upload_aug(seeded_aug(plan, len(clips), 5))
    noise = torch.randn(len(clips), plan.target_length, device=DEV) if noise_kind == "host" else None
    got = fused(plan, clips, rates, False, rs, aug=aug, noise=noise, normalize=normalize)
    assert_bytes_equal(got, two_step(plan, clips, rates, aug=aug, noise=noise, normalize=normalize))


@pytest.mark.parametrize("plan_cfg,rates", [
    ((4000, 256, 64, 64), [44100, 10000, 4000]),
    ((8000, 512, 128, 128), [44100, 10000, 4000, 8000]),
    ((16000, 1024, 256, 128), [44100, 10000, 4000, 16000]),
    ((16000, 512, 128, 128), [44100, 4000, 16000]),
], ids=["4k_256", "8k_512", "16k_1024", "16k_512"])
@pytest.mark.parametrize("pcm16", [False, True], ids=["fp32", "int16"])
def test_other_fft_sizes_equal_two_step(plan_cfg, rates, pcm16):
    sr, n_fft, hop, n_mels = plan_cfg
    plan = get_plan(sr, n_fft, hop, n_mels)
    rs = np.random.RandomState(14)
    lengths, rr = [], []
    for r in rates:
        ls = edge_lengths(r, sr, plan.target_length)
        lengths += ls
        rr += [r] * len(ls)
    clips = make_clips(rs, lengths, pcm16)
    assert_bytes_equal(fused(plan, clips, rr, pcm16, rs), two_step(plan, clips, rr))
    aug = plan.upload_aug(seeded_aug(plan, len(clips), 6))
    assert_bytes_equal(fused(plan, clips, rr, pcm16, rs, aug=aug), two_step(plan, clips, rr, aug=aug))


@pytest.mark.parametrize("B", [1, 3])
def test_small_batch_split_equals_unsplit(B):
    plan = A.LogMelPlan(sample_rate=16000, n_fft=2048, hop_length=512, n_mels=128, target_length=80000, device=DEV)
    rs = np.random.RandomState(15)
    rates = [44100, 4000, 16000][:B]
    clips = make_clips(rs, [44100 * 20, 4000 * 3, 70000][:B], False)
    auto = fused(plan, clips, rates, False, rs)
    assert_bytes_equal(auto, two_step(plan, clips, rates))
    plan.set("split", 1)
    assert_bytes_equal(fused(plan, clips, rates, False, rs), auto)
    plan.close()


def test_against_torchaudio_on_cpu():
    import torchaudio.transforms as TT
    plan = get_plan(16000, 2048, 512, 128)
    rs = np.random.RandomState(16)
    rates = [44100, 10000, 4000, 16000]
    clips = make_clips(rs, [44100 * 6, 10000 * 4, 4000 * 5, 70000], False)
    got = fused(plan, clips, rates, False, rs).cpu().numpy()
    ocfg = O.OracleConfig(sample_rate=16000, n_fft=2048, hop_length=512, n_mels=128, duration=5.0)
    fb = A.reference_filterbank(1025, 128, 16000).numpy()
    for i, r in enumerate(rates):
        x = clips[i] if r == 16000 else TT.Resample(r, 16000)(clips[i].unsqueeze(0))[0]
        ref = O.logmel(x.numpy(), ocfg, fb=fb)
        # bands above the resampler's cut-off are nearly empty: a 1e-6 waveform difference moves their dB visibly
        tol = 2e-4 if r == 16000 else 5e-3
        assert np.abs(got[i, 0] - ref).max() < tol, (i, r)


# ---- drop-in paths ------------------------------------------------------------------------------------------------------

def _write_icbhi(tmp_path, rates, secs, seed):
    d = tmp_path / "audio_and_txt_files"
    d.mkdir()
    rs = np.random.RandomState(seed)
    for i, (sr, s) in enumerate(zip(rates, secs)):
        x = (rs.standard_normal(int(sr * s)) * 0.1).clip(-1, 1)
        wavio.write_wav_pcm16(str(d / f"{100 + i}_r.wav"), x, sr)
        (d / f"{100 + i}_r.txt").write_text(f"0.0\t1.0\t{i % 2}\t0\n")
    return [(str(d / f"{100 + i}_r.wav"), i % 2) for i in range(len(rates))]


def _old_collate(pre, batch):
    """GpuCollate before resampling moved into the kernel: lm_resample per item, then one lm_forward."""
    waves = [pre.resample_to_target(w, sr) for w, sr, _ in batch]
    return pre.preprocess_batch(waves)


def test_gpu_collate_one_launch_per_batch_equals_per_item_path(tmp_path):
    rates = [4000, 10000, 16000, 44100, 44100, 10000, 4000, 16000]
    secs = [20, 7.5, 5, 21.3, 3, 12, 2.5, 8]
    data = _write_icbhi(tmp_path, rates, secs, 21)
    ds = A.ICBHIDataset(tmp_path, "test")
    ds.data = data
    raw = ds.raw()
    pre = ds.preprocessor
    collate = A.GpuCollate(pre)
    for lo in (0, 4):
        batch = [raw[i] for i in range(lo, lo + 4)]
        n0 = pre.plan.launches
        feats, labels = collate(batch)
        assert pre.plan.launches == n0 + 1
        assert labels.tolist() == [y for _, _, y in batch]
        assert_bytes_equal(feats, _old_collate(pre, batch))


def test_gpu_collate_groups_beyond_max_resamplers(monkeypatch):
    pre = A.AudioPreprocessor()
    rs = np.random.RandomState(22)
    rates = [8000, 11025, 12000, 22050, 24000, 32000, 44100, 48000, 10000, 16000]
    assert len(set(rates) - {16000}) > _lib.LM_MAX_RESAMPLERS
    batch = [(torch.from_numpy((rs.standard_normal((1, int(r * 3.3))) * 0.1).astype(np.float32)), r, i % 4)
             for i, r in enumerate(rates)]
    ref = _old_collate(pre, batch)

    def no_per_item_resampling(*args):
        raise AssertionError("resampled item by item")
    monkeypatch.setattr(pre, "resample_to_target", no_per_item_resampling)
    n0 = pre.plan.launches
    feats, _ = A.GpuCollate(pre)(batch)
    assert pre.plan.launches == n0 + 2   # 9 foreign rates: two groups of at most 8, no lm_resample
    assert_bytes_equal(feats, ref)
    # the same items split into batches of <= 8 foreign rates take the fused path, with the same features
    feats2 = torch.cat([A.GpuCollate(pre)(batch[:5])[0], A.GpuCollate(pre)(batch[5:])[0]])
    assert_bytes_equal(feats2, feats)
    # preprocess_batch takes any number of rates, too
    waves = [w for w, _, _ in batch]
    assert_bytes_equal(pre.preprocess_batch(waves, sample_rates=rates), ref)
    split = [pre.preprocess_batch(waves[:5], sample_rates=rates[:5]),
             pre.preprocess_batch(waves[5:], sample_rates=rates[5:])]
    assert_bytes_equal(torch.cat(split), ref)


def test_flexible_8s_mixed_rates_equals_two_step():
    f = A.FlexibleAudioPreprocessor(duration=8.0)
    assert f.plan.frames != f.target_time_steps()   # the resize path
    rs = np.random.RandomState(23)
    rates = [44100, 4000, 16000, 10000]
    clips = [torch.from_numpy((rs.standard_normal(int(r * s)) * 0.1).astype(np.float32))
             for r, s in zip(rates, [9.1, 4.0, 8.0, 20.0])]
    got = f.preprocess_batch(clips, sample_rates=rates)
    ref = f.preprocess_batch([f.resample_to_target(c, r) for c, r in zip(clips, rates)])
    assert got.shape == (4, 1, 128, f.target_time_steps())
    assert_bytes_equal(got, ref)


def test_preprocess_batch_at_the_plan_rate_is_unchanged():
    pre = A.AudioPreprocessor()
    rs = np.random.RandomState(24)
    clips = [torch.from_numpy((rs.standard_normal(n) * 0.1).astype(np.float32)) for n in (80000, 12345)]
    assert_bytes_equal(pre.preprocess_batch(clips, sample_rates=[16000, 16000]), pre.preprocess_batch(clips))


# ---- error paths --------------------------------------------------------------------------------------------------------

def test_error_paths():
    plan = get_plan(16000, 2048, 512, 128)
    lib = _lib.load()
    wave = torch.zeros(1000, device=DEV)
    off = torch.zeros(1, dtype=torch.int64, device=DEV)
    ln = torch.full((1,), 1000, dtype=torch.int32, device=DEV)
    src = torch.zeros(1, dtype=torch.int32, device=DEV)
    out = torch.empty(plan.out_shape(1), device=DEV)
    r = get_resampler(44100, 16000, DEV)
    handles = (C.c_void_p * 9)(*([r._h.value] * 9))
    call = lambda arr, n: lib.lm_forward_resampled(plan._h, arr, n, wave.data_ptr(), 0, off.data_ptr(), ln.data_ptr(),
                                                    src.data_ptr(), 1, None, None, out.data_ptr(), 1, None)
    assert call(handles, 9) == -1
    assert call(handles, -1) == -1
    assert call(None, 1) == -1
    assert call((C.c_void_p * 2)(r._h.value, None), 2) == -1
    assert call(handles, 1) == 0
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="source values"):
        plan.forward_resampled(wave, off, ln, torch.tensor([1], dtype=torch.int32), [r])
    with pytest.raises(ValueError, match="source values"):
        plan.forward_resampled(wave, off, ln, torch.tensor([-2], dtype=torch.int32, device=DEV), [r])
    with pytest.raises(ValueError, match="plan's 16000 Hz"):
        plan.forward_resampled(wave, off, ln, src, [get_resampler(44100, 8000, DEV)])
    with pytest.raises(ValueError, match="at most 8"):
        plan.forward_resampled(wave, off, ln, src, [r] * 9)


def test_invalid_device_source_reads_nothing():
    """source is device data the host does not check on the C path: an index outside [-1, n) is an empty clip."""
    plan = get_plan(16000, 2048, 512, 128)
    lib = _lib.load()
    rs = np.random.RandomState(25)
    clips = make_clips(rs, [44100 * 5, 44100 * 5], False)
    wave, off, ln = pack_unaligned(rs, clips, False)
    r = get_resampler(44100, 16000, DEV)
    src = torch.tensor([7, -5], dtype=torch.int32, device=DEV)
    out = torch.empty(plan.out_shape(2), device=DEV)
    assert lib.lm_forward_resampled(plan._h, (C.c_void_p * 1)(r._h.value), 1, wave.data_ptr(), 0, off.data_ptr(),
                                    ln.data_ptr(), src.data_ptr(), 2, None, None, out.data_ptr(), 1, None) == 0
    empty = plan.forward(torch.zeros(4, device=DEV), torch.zeros(2, dtype=torch.int64, device=DEV),
                         torch.zeros(2, dtype=torch.int32, device=DEV))
    assert_bytes_equal(out, empty)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_resampler_on_another_device_is_refused():
    plan = get_plan(16000, 2048, 512, 128)
    other = A.Resampler(44100, 16000, f"cuda:{torch.cuda.device_count() - 1}")
    wave = torch.zeros(1000, device=DEV)
    off = torch.zeros(1, dtype=torch.int64, device=DEV)
    ln = torch.full((1,), 1000, dtype=torch.int32, device=DEV)
    src = torch.zeros(1, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError, match="resampler on"):
        plan.forward_resampled(wave, off, ln, src, [other])
    out = torch.empty(plan.out_shape(1), device=DEV)
    assert _lib.load().lm_forward_resampled(plan._h, (C.c_void_p * 1)(other._h.value), 1, wave.data_ptr(), 0,
                                            off.data_ptr(), ln.data_ptr(), src.data_ptr(), 1, None, None,
                                            out.data_ptr(), 1, None) == -1
    other.close()
