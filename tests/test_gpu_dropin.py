"""GPU tests of the drop-in layer: the reference's class contract, served by the CUDA path.
Run on the B200 box: pytest -m gpu."""
import random

import numpy as np
import pytest
import torch

import audio_classification_icbhi_b200 as A
from audio_classification_icbhi_b200 import wavio
from oracle import logmel_oracle as O
from tests.golden.make_golden import PLAIN_CASES, golden_input

pytestmark = pytest.mark.gpu
NORM_ATOL = 2e-4
DB_ATOL = 1e-3


def set_seed(seed):   # R/src/utils/config.py:31-33
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)


def test_preprocess_file_returns_the_reference_contract(tmp_path, golden):
    """preprocess(path) -> fresh float32 CPU tensor [1, n_mels, frames] (R/diagnose_data.py:55-66)."""
    x = golden_input(0, 80000)
    path = str(tmp_path / "clip.wav")
    wavio.write_wav_pcm16(path, x, 16000)
    p = A.AudioPreprocessor()
    out = p.preprocess(path)
    assert isinstance(out, torch.Tensor) and out.device.type == "cpu" and out.dtype == torch.float32
    assert tuple(out.shape) == (1, 128, 157) and torch.isfinite(out).all()
    xq = np.rint(x.astype(np.float64) * 32767) / 32768.0           # what the PCM_16 file holds
    assert np.abs(out[0].numpy() - O.logmel(xq.astype(np.float32), O.OracleConfig())).max() < NORM_ATOL
    # and an in-memory clip reproduces the reference's own output
    out2 = p.preprocess_waveform(torch.from_numpy(x).unsqueeze(0))
    assert np.abs(out2[0].numpy() - golden["headline_5s/norm"]).max() < NORM_ATOL
    # stereo input is averaged to mono like load_audio does
    out3 = p.preprocess_waveform(torch.from_numpy(np.stack([x, x])))
    assert torch.equal(out3, out2)


@pytest.mark.parametrize("tag,dur", [("aug_3s", 3.0), ("aug_5s", 5.0)])
def test_seeded_training_path_reproduces_the_reference(golden, tag, dur):
    """Config 4: set_seed(42), augment=True, clips one by one (the reference's call pattern) and as
    one batch: both give the reference's seeded outputs."""
    T = int(16000 * dur)
    clips = [golden_input(100 + c, T) for c in range(6)]
    set_seed(42)
    p = A.AudioPreprocessor(duration=dur, augment=True)
    one_by_one = [p.preprocess_waveform(torch.from_numpy(c).unsqueeze(0)) for c in clips]
    set_seed(42)
    batched = p.preprocess_batch(clips).cpu()
    for c in range(6):
        ref = golden[f"{tag}/clip{c}/norm"]
        assert np.abs(one_by_one[c][0].numpy() - ref).max() < NORM_ATOL
        assert torch.equal(batched[c], one_by_one[c])
    # throughput mode: on-device noise, private RNG -- valid features, masks inside the bounds
    fast = p.preprocess_batch(clips, fast_augment=True)
    assert torch.isfinite(fast).all() and fast.shape == batched.shape


def test_flexible_resize_8s_matches_reference(golden):
    x = golden_input(7, 128000)
    f = A.FlexibleAudioPreprocessor(duration=8.0)
    out = f.preprocess_waveform(x)
    assert tuple(out.shape) == (1, 128, 250)
    assert np.abs(out[0].numpy() - golden["flex_8s_resize/norm"]).max() < NORM_ATOL
    # resize_spectrogram on its own, host tensor in -> host tensor out, equals F.interpolate
    db = torch.from_numpy(golden["cfg_8s/db"]).unsqueeze(0)
    r = f.resize_spectrogram(db)
    assert r.device.type == "cpu" and tuple(r.shape) == (1, 128, 250)
    ref = torch.nn.functional.interpolate(db.unsqueeze(0), size=(128, 250), mode="bilinear", align_corners=False)[0]
    assert (r - ref).abs().max().item() < 1e-4
    assert np.abs(r[0].numpy() - golden["flex_8s_resize/db"]).max() < DB_ATOL
    assert f.resize_spectrogram(torch.zeros(1, 128, 250)).shape[-1] == 250      # no-op when sizes agree


def test_flexible_resize_with_masks_acts_on_resized_axis():
    set_seed(3)
    f = A.FlexibleAudioPreprocessor(duration=8.0, augment=True)
    x = golden_input(12, 128000)
    set_seed(3)
    aug, noise = A.draw_reference_augmentation(1, 128000, 128, 250)
    set_seed(3)
    out = f.preprocess_batch([x]).cpu().numpy()[0, 0]
    a = aug[0]
    ref = O.logmel(x, O.OracleConfig(duration=8.0), flexible=True, shift=int(a["shift"]),
                   noise=None if noise is None else noise[0].numpy(), noise_scale=float(a["noise_scale"]),
                   masks=(int(a["f0"]), int(a["f1"]), int(a["t0"]), int(a["t1"])))
    assert out.shape == (128, 250)
    assert np.abs(out - ref).max() < NORM_ATOL


@pytest.mark.parametrize("seg,overlap,n_fft", [(1.0, 0.5, 2048), (0.5, 0.75, 1024)])
def test_sliding_windows_match_per_window_oracle(seg, overlap, n_fft):
    """Config 5 in miniature: every window is an independent clip (own reflect padding, own
    normalisation), the tail window is zero padded."""
    sw = A.SlidingWindowLogMel(segment_duration=seg, overlap=overlap)
    assert sw.preprocessor.n_fft == n_fft
    rs = np.random.RandomState(9)
    n = 15 * 16000 + 1234
    rec = (rs.standard_normal(n) * 0.1).astype(np.float32)
    feats, times = sw(rec)
    starts, lengths, times2 = A.segment_offsets(n, 16000, seg, overlap)
    assert feats.shape == (len(starts), 1, 128, 32) and times == times2
    n_fft_o, hop_o = O.flexible_fft_params(16000, min(2048, int(16000 * seg / 2)), 256 if seg < 1 else 512, seg)
    cfg = O.OracleConfig(n_fft=n_fft_o, hop_length=hop_o, duration=seg)
    got = feats.cpu().numpy()
    for w in (0, 1, len(starts) // 2, len(starts) - 2, len(starts) - 1):
        s, l = int(starts[w]), int(lengths[w])
        assert np.abs(got[w, 0] - O.logmel(rec[s:s + l], cfg)).max() < NORM_ATOL, w
    # a shard of the windows equals the same rows of the full run (multi-GPU layout)
    part, _ = sw(rec, window_range=(5, 17))
    assert torch.equal(part, feats[5:17])
    # optional PCM_16 round-trip emulation
    swq = A.SlidingWindowLogMel(segment_duration=seg, overlap=overlap, emulate_pcm16=True)
    fq, _ = swq(rec)
    recq = (np.rint(np.clip(rec, -1, 1).astype(np.float64) * 32767) / 32768.0).astype(np.float32)
    s, l = int(starts[3]), int(lengths[3])
    assert np.abs(fq[3, 0].cpu().numpy() - O.logmel(recq[s:s + l], cfg)).max() < NORM_ATOL


def test_hour_long_recording_window_count_and_spot_checks():
    """Config 5 at full size: 1 h at 16 kHz, 1 s windows, 50 % overlap -> 7200 windows."""
    sw = A.SlidingWindowLogMel(segment_duration=1.0, overlap=0.5)
    g = torch.Generator(device="cuda").manual_seed(2)
    rec = torch.randn(3600 * 16000, generator=g, device="cuda") * 0.1
    feats, times = sw(rec)
    torch.cuda.synchronize()
    assert feats.shape == (7200, 1, 128, 32) and times[-1] == (3599.5, 3600.0)
    assert torch.isfinite(feats).all()
    flat = feats.view(7200, -1).double()
    assert flat.mean(dim=1).abs().max().item() < 1e-5 and (flat.std(dim=1) - 1).abs().max().item() < 1e-5
    cfg = O.OracleConfig(duration=1.0)
    for w in (0, 3333, 7198, 7199):
        s = w * 8000
        ref = O.logmel(rec[s:s + 16000].cpu().numpy(), cfg)
        assert np.abs(feats[w, 0].cpu().numpy() - ref).max() < NORM_ATOL


def test_datasets_end_to_end_with_gpu_collate(tmp_path):
    d = tmp_path / "audio_and_txt_files"
    d.mkdir()
    rs = np.random.RandomState(1)
    sigs = []
    for i in range(10):
        x = (rs.standard_normal(16000 * (2 + i % 3)) * 0.1).clip(-1, 1)
        sigs.append(x)
        wavio.write_wav_pcm16(str(d / f"{100 + i}_r.wav"), x, 16000)
        (d / f"{100 + i}_r.txt").write_text(f"0.0\t1.0\t{i % 2}\t0\n")
    cfg = {"data": dict(sample_rate=16000, n_mels=128, n_fft=2048, hop_length=512, duration=3.0)}
    ds = A.ICBHIDataset(tmp_path, "train", cfg, augment=False)
    mel, label = ds[2]                                   # the reference's __getitem__ contract
    assert mel.device.type == "cpu" and tuple(mel.shape) == (1, 128, 94) and label == 0
    loader = torch.utils.data.DataLoader(ds.raw(), batch_size=4, shuffle=False, num_workers=0,
                                         collate_fn=A.GpuCollate(ds.preprocessor))
    feats, labels = next(iter(loader))
    assert feats.is_cuda and feats.shape == (4, 1, 128, 94) and labels.tolist() == [0, 1, 0, 1]
    assert torch.allclose(feats[2].cpu(), mel, atol=1e-6)
    xq = (np.rint(sigs[2] * 32767) / 32768.0).astype(np.float32)
    assert np.abs(mel[0].numpy() - O.logmel(xq, O.OracleConfig(duration=3.0))).max() < NORM_ATOL


def test_segmenter_gpu_shortcut(tmp_path):
    rs = np.random.RandomState(4)
    x = (rs.standard_normal(16000 * 9) * 0.1).clip(-1, 1)
    wavio.write_wav_pcm16(str(tmp_path / "a.wav"), x, 16000)
    (tmp_path / "a.txt").write_text("0.1\t2.6\t0\t0\n2.6\t2.9\t1\t0\n2.9\t8.95\t1\t1\n")
    seg = A.ICBHISegmenter(tmp_path, tmp_path / "out")
    p = A.AudioPreprocessor()
    feats, labels = seg.segments_to_features(tmp_path / "a.wav", tmp_path / "a.txt", p)
    assert labels == ["normal", "both"] and feats.shape == (2, 1, 128, 157)
    xq = (np.rint(x * 32767) / 32768.0).astype(np.float32)
    for i, (a, b) in enumerate(((0.1, 2.6), (2.9, 8.95))):
        ref = O.logmel(xq[int(a * 16000):int(b * 16000)], O.OracleConfig())
        assert np.abs(feats[i, 0].cpu().numpy() - ref).max() < NORM_ATOL


@pytest.mark.parametrize("n_mels,hop,dur", [(64, 512, 2.0), (40, 256, 1.5), (128, 128, 1.0), (200, 512, 2.0)])
def test_other_configurations_match_oracle(n_mels, hop, dur):
    """The config keys are inputs, not constants: other n_mels / hop values go through the same kernel."""
    p = A.AudioPreprocessor(n_mels=n_mels, hop_length=hop, duration=dur)
    x = golden_input(31, int(16000 * dur) + 777)
    out = p.preprocess_waveform(x)[0].numpy()
    cfg = O.OracleConfig(n_mels=n_mels, hop_length=hop, duration=dur)
    assert out.shape == (n_mels, cfg.frames)
    fb = A.reference_filterbank(1025, n_mels, 16000).numpy()
    assert np.abs(out - O.logmel(x, cfg, fb=fb)).max() < NORM_ATOL


def test_unsupported_configurations_fail_loudly():
    for kw in (dict(n_fft=4096), dict(n_fft=2000), dict(hop_length=511), dict(hop_length=1024), dict(n_mels=300)):
        with pytest.raises(RuntimeError, match="unsupported configuration"):
            A.AudioPreprocessor(**kw).plan
    with pytest.raises(RuntimeError, match="target_len must exceed"):
        A.AudioPreprocessor(duration=0.05).plan


@pytest.mark.parametrize("sr", [4000, 10000, 44100, 8000, 22050, 48000])
def test_gpu_resampler_matches_torchaudio_golden_and_oracle(sr):
    """lm_resample (CUDA polyphase sinc) against T.Resample(sr, 16000) as the reference calls it
    (golden, generated from torchaudio) and against the float64 oracle: 1e-5 / 2e-6 of full scale."""
    import os
    from oracle import logmel_oracle as O
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "resample_golden.npz"))
    x = g[f"in/{sr}"]
    r = A.get_resampler(sr, 16000)
    y = r(torch.from_numpy(x)).cpu().numpy()
    assert y.shape == g[f"out/{sr}"].shape and r.out_len(len(x)) == len(y)
    assert np.abs(y - g[f"out/{sr}"]).max() < 1e-5
    assert np.abs(y - O.resample(x, sr, 16000)).max() < 2e-6
    y2 = r(torch.from_numpy(np.stack([x, 0.5 * x]))).cpu().numpy()      # [channels, len]
    np.testing.assert_array_equal(y2[0], y)
    assert r(torch.zeros(0)).numel() == 0


def test_load_audio_resamples_on_the_gpu(tmp_path):
    """load_audio of a 4 kHz PCM16 wav -> 16 kHz mono through the CUDA resampler (preprocessing.py:55-68)."""
    from oracle import logmel_oracle as O
    rs = np.random.RandomState(3)
    x = (rs.standard_normal(4000) * 0.2).clip(-1, 1)
    path = str(tmp_path / "lo.wav")
    wavio.write_wav_pcm16(path, x, 4000)
    p = A.AudioPreprocessor()
    w = p.load_audio(path)
    assert w.shape == (1, 16000) and w.dtype == torch.float32 and w.device.type == "cpu"
    q = np.rint(x * 32767) / 32768.0
    assert np.abs(w[0].numpy() - O.resample(q, 4000, 16000)).max() < 2e-6
    feats = p.preprocess(path)
    assert feats.shape == (1, 128, 157)


def test_randomised_geometries_match_oracle():
    """Seeded sweep over plan geometries (n_fft, hop, n_mels, target length down to just above n_fft/2, i.e. one
    or two tiles, a last tile with a single frame, ...) and ragged clip lengths (empty, shorter than a hop,
    cropped), several clips per group: the kernel against the oracle fed with torchaudio's filterbank."""
    rs = np.random.RandomState(2024)
    for trial in range(14):
        n_fft = int(rs.choice([2048, 2048, 1024]))
        hop = int(rs.choice([64, 128, 160, 256, 400, 512])) if n_fft == 2048 else int(rs.choice([64, 100, 128, 256]))
        n_mels = int(rs.choice([24, 40, 64, 80, 128, 136, 256 if n_fft == 2048 else 96]))
        T = int(rs.choice([n_fft // 2 + 1, n_fft // 2 + 7, n_fft, 3000, 7 * hop + 5, 8 * hop, 8 * hop - 1, 16001, 48000]))
        T = max(T, n_fft // 2 + 1)
        plan = A.LogMelPlan(n_fft=n_fft, hop_length=hop, n_mels=n_mels, target_length=T, device="cuda:0")
        plan.set("max_ctas", int(rs.choice([1, 2, 148])))
        cfg = O.OracleConfig(n_mels=n_mels, n_fft=n_fft, hop_length=hop, duration=T / 16000.0)
        assert cfg.target_length == T or abs(cfg.target_length - T) <= 1
        lens = [0, 1, hop - 1, T, T + 1, 3 * T + 11] + [int(v) for v in rs.randint(1, 2 * T, 5)]
        clips = [(rs.standard_normal(n) * 0.1).astype(np.float32) for n in lens]
        starts, pos = [], 0
        for c in clips:
            starts.append(pos)
            pos += (len(c) + 3) // 4 * 4 + (4 if trial % 2 else 1)      # every other trial: unaligned starts
        packed = np.zeros(pos + 4, dtype=np.float32)
        for s, c in zip(starts, clips):
            packed[s:s + len(c)] = c
        dev = plan.device
        out = plan.forward(torch.from_numpy(packed).to(dev), torch.tensor(starts, dtype=torch.int64, device=dev),
                           torch.tensor(lens, dtype=torch.int32, device=dev)).cpu().numpy()[:, 0]
        fb = A.reference_filterbank(n_fft // 2 + 1, n_mels, 16000).numpy().astype(np.float64)
        frames = 1 + T // hop
        assert out.shape == (len(clips), n_mels, frames), (trial, out.shape)
        for i, c in enumerate(clips):
            w = O.pad_or_crop(c.astype(np.float64), T)
            db = O.amplitude_to_db(O.mel_power(O.stft_power(w, n_fft, hop), fb))
            ref = O.normalize(db)
            assert np.abs(out[i] - ref).max() < NORM_ATOL, (trial, n_fft, hop, n_mels, T, lens[i])
        # the same clips as 16-bit PCM: the fused staging (bulk copy + in-place expansion, or the gather path for the
        # unaligned trials) against decode-then-forward, bit for bit, at this geometry
        q = np.clip(np.rint(packed * 32768.0), -32768, 32767).astype(np.int16)
        if trial % 2 == 0:                                  # aligned trials: starts on 8-sample boundaries for the bulk path
            starts8, pos8 = [], 0
            for c in clips:
                starts8.append(pos8)
                pos8 += (len(c) + 7) // 8 * 8
            q8 = np.zeros(pos8 + 8, dtype=np.int16)
            for s8, s4, c in zip(starts8, starts, clips):
                q8[s8:s8 + len(c)] = q[s4:s4 + len(c)]
            q, qstarts = q8, starts8
        else:
            qstarts = starts
        d_q = torch.from_numpy(q).to(dev)
        d_off = torch.tensor(qstarts, dtype=torch.int64, device=dev)
        d_len = torch.tensor(lens, dtype=torch.int32, device=dev)
        want = plan.forward(plan.pcm16_decode(d_q), d_off, d_len)
        got = plan.forward_pcm16(d_q, d_off, d_len)
        torch.cuda.synchronize()
        assert torch.equal(got, want), ("pcm16", trial, n_fft, hop, n_mels, T)
        plan.close()


def test_forked_workers_decode_and_the_gpu_resamples_and_collates(tmp_path):
    """The training-loop pattern of INTEGRATION.md section 3 with real forked workers: 44.1 / 4 / 10 kHz recordings are
    decoded in the workers (no CUDA there), resampled and turned into features in this process, one launch per batch."""
    d = tmp_path / "audio_and_txt_files"
    d.mkdir()
    rs = np.random.RandomState(6)
    rates = [44100, 4000, 10000, 16000, 44100, 16000]
    sigs = []
    for i, sr in enumerate(rates):
        x = (rs.standard_normal(sr * 2) * 0.1).clip(-1, 1)
        sigs.append(x)
        wavio.write_wav_pcm16(str(d / f"{100 + i}_r.wav"), x, sr)
        (d / f"{100 + i}_r.txt").write_text(f"0.0\t1.0\t{i % 2}\t0\n")
    cfg = {"data": dict(sample_rate=16000, n_mels=128, n_fft=2048, hop_length=512, duration=3.0)}
    ds = A.ICBHIDataset(tmp_path, "test", cfg)
    ds.data = [(str(d / f"{100 + i}_r.wav"), i % 2) for i in range(6)]
    torch.cuda.init()
    _ = ds.preprocessor.plan                                  # the parent owns a CUDA context before the fork
    loader = torch.utils.data.DataLoader(ds.raw(), batch_size=3, num_workers=2, collate_fn=A.raw_collate,
                                         multiprocessing_context="fork")
    feats, labels = [], []
    launches0 = ds.preprocessor.plan.launches
    for f, y in A.GpuLoader(loader, A.GpuCollate(ds.preprocessor)):
        assert f.is_cuda and f.shape == (3, 1, 128, 94)
        feats.append(f)
        labels += y.tolist()
    assert ds.preprocessor.plan.launches - launches0 == 2 and labels == [0, 1, 0, 1, 0, 1]
    feats = torch.cat(feats).cpu().numpy()
    for i, sr in enumerate(rates):
        xq = (np.rint(sigs[i] * 32767) / 32768.0).astype(np.float32)
        x16 = xq if sr == 16000 else O.resample(xq, sr, 16000).astype(np.float32)
        # a resampled clip has almost no energy above the resampler's cut-off: there a 1e-6 waveform difference between
        # the fp32 kernel and the float64 oracle resampler moves the dB value of an (empty) band visibly
        tol = NORM_ATOL if sr == 16000 else 5e-3
        assert np.abs(feats[i, 0] - O.logmel(x16, O.OracleConfig(duration=3.0))).max() < tol


def test_transform_attributes_of_the_reference_class(golden):
    """The reference object exposes its torchaudio transforms as attributes (R/src/data/preprocessing.py:38-53); callers
    such as tests/golden/make_golden.py use them directly.  Here they are GPU-backed: mel_spectrogram against the
    reference's mel power, amplitude_to_db against its dB stage, the masks against torchaudio's own draws."""
    p = A.AudioPreprocessor(augment=True)
    for name, seed, n in (("headline_5s", 1, 80000), ("short_1p3s_pad_5s", 2, 20800)):
        case = [c for c in PLAIN_CASES if c[0] == name][0]
        w = p.pad_or_crop(torch.from_numpy(golden_input(case[3], case[4], case[5])).unsqueeze(0))
        melp = p.mel_spectrogram(w)
        assert melp.device.type == "cpu" and tuple(melp.shape) == (1, 128, 157)
        ref = golden[f"{name}/mel_power"]
        floor = max(1e-6 * np.abs(ref).max(), 1e-30)
        assert (np.abs(melp[0].numpy() - ref) / np.maximum(np.abs(ref), floor)).max() < 1e-4
        db = p.amplitude_to_db(torch.from_numpy(ref).unsqueeze(0))
        assert np.abs(db[0].numpy() - golden[f"{name}/db"]).max() < 1e-4
        assert np.abs(p.normalize(db)[0].numpy() - golden[f"{name}/norm"]).max() < NORM_ATOL
    x = torch.randn(1, 48000) * 0.1                     # another length: the attribute neither pads nor crops
    assert tuple(p.mel_spectrogram(x).shape) == (1, 128, 94)
    import torchaudio.transforms as T
    spec = torch.randn(1, 128, 157)
    torch.manual_seed(3)
    a = p.time_mask(p.freq_mask(spec))
    torch.manual_seed(3)
    b = T.TimeMasking(time_mask_param=35)(T.FrequencyMasking(freq_mask_param=15)(spec))
    assert torch.equal(a, b)
    assert not hasattr(A.AudioPreprocessor(augment=False), "freq_mask")       # as in the reference: only with augment


@pytest.mark.parametrize("sr", [44100, 4000, 10000, 22050, 48000, 384000])
def test_tiled_resampler_is_bit_identical_to_the_plain_kernel(sr, monkeypatch):
    """The shared-memory tiled resampler and the one-output-per-thread kernel run the same chain over the same padded
    taps, so they agree bit for bit, on non-finite samples too (a zero padding tap over inf gives NaN in both).  384 kHz
    takes the plain kernel by default (its tiled span is over 96 KB)."""
    from audio_classification_icbhi_b200.resample import Resampler
    x = torch.from_numpy(np.random.RandomState(sr).standard_normal((3, 2 * sr + 123)).astype(np.float32) * 0.1)
    x[0, [7, sr // 3, sr + 1]] = float("inf")
    x[0, sr // 2] = float("nan")
    x[2, [0, sr - 2, 2 * sr + 122]] = float("-inf")
    tiled = Resampler(sr, 16000)(x)
    monkeypatch.setenv("LM_RESAMPLE_UNTILED", "1")
    plain = Resampler(sr, 16000)(x)
    assert tiled.shape == plain.shape and torch.equal(tiled.view(torch.int32), plain.view(torch.int32))
    assert not torch.isfinite(tiled[0]).all() and not torch.isfinite(tiled[2]).all()
    ref = O.resample(x[1].numpy(), sr, 16000)
    assert np.abs(tiled[1].cpu().numpy() - ref).max() < 2e-6
