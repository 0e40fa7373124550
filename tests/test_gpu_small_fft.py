"""GPU tests of the 512- and 256-point STFT paths (ICBHI's 4 / 8 kHz rates, the 32 ms window at 16 kHz): the CUDA
kernel through the C ABI against the float64 oracle with torchaudio's filterbank and against torchaudio's CPU
MelSpectrogram -> AmplitudeToDB -> normalise, plus the bit-identity invariants the 1024 / 2048 paths keep.
Bars as in test_gpu_parity: dB 1e-3 absolute, mel power 1e-4 relative, normalised 2e-4, floor and frame counts exact."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import audio_classification_icbhi_b200 as A
from audio_classification_icbhi_b200 import wavio
from oracle import logmel_oracle as O
from tests.test_gpu_parity import rel_err, run_clips

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DB_ATOL = 1e-3
MEL_RTOL = 1e-4
NORM_ATOL = 2e-4

# (sample_rate, n_fft, hop, n_mels, target_length)
GEOMETRIES = [
    (16000, 512, 128, 128, 80000),   # 32 ms window at 16 kHz, 626 frames
    (16000, 512, 100, 64, 16000),    # a smaller even hop
    (8000, 512, 128, 64, 40000),     # 313 frames
    (8000, 256, 64, 40, 16000),
    (4000, 256, 64, 64, 20000),      # ICBHI's lowest rate, 313 frames
    (4000, 256, 50, 128, 12000),     # 128 mels on 129 bins: filters without support
    (4000, 512, 96, 40, 8000),
    (8000, 256, 64, 40, 129),        # target just above n_fft/2
    (16000, 512, 128, 64, 257),
]
GEO_IDS = [f"sr{g[0]}_n{g[1]}_h{g[2]}_m{g[3]}_T{g[4]}" for g in GEOMETRIES]

_plans = {}


def get_plan(sr, n_fft, hop, n_mels, T):
    key = (sr, n_fft, hop, n_mels, T)
    if key not in _plans:
        _plans[key] = A.LogMelPlan(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, target_length=T,
                                   device="cuda:0")
    return _plans[key]


def oracle_cfg(sr, n_fft, hop, n_mels, T):
    cfg = O.OracleConfig(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, duration=(T + 0.5) / sr)
    assert cfg.target_length == T
    return cfg


def torchaudio_fb(sr, n_fft, n_mels):
    return A.reference_filterbank(n_fft // 2 + 1, n_mels, sr).numpy()


def ragged_lengths(T, n_fft):
    return [T, 0, 1, n_fft // 2 + 1, T // 3 + 1, T - 1, T + 777, 2 * T + 1, n_fft + 3]


@pytest.mark.parametrize("geo", GEOMETRIES, ids=GEO_IDS)
def test_ragged_batch_matches_oracle(geo):
    """Padded, centre-cropped, empty and one-sample clips in one launch, against the float64 oracle: all three
    stages within the bars, the frame count exact, the -100 dB floor exact wherever the oracle's mel power is 0."""
    sr, n_fft, hop, n_mels, T = geo
    plan = get_plan(*geo)
    cfg = oracle_cfg(*geo)
    assert plan.frames == cfg.frames == 1 + T // hop
    fb = torchaudio_fb(sr, n_fft, n_mels)
    rs = np.random.RandomState(n_fft + hop + n_mels)
    clips = [(rs.standard_normal(n) * 0.1).astype(np.float32) for n in ragged_lengths(T, n_fft)]
    got = run_clips(plan, clips)
    assert got["out"].shape == (len(clips), n_mels, cfg.frames)
    for i, x in enumerate(clips):
        st = O.logmel(x, cfg, return_stages=True, fb=fb)
        assert rel_err(got["mel_power"][i], st["mel_power"]).max() < MEL_RTOL, (i, len(x))
        assert np.abs(got["db"][i] - st["db"]).max() < DB_ATOL, (i, len(x))
        assert np.abs(got["out"][i] - st["out"]).max() < NORM_ATOL, (i, len(x))
        # where the oracle's mel power is 0 the dB floor is exact; the power itself is below amin there but not
        # always 0: a silent frame packed with a sounding one into one complex FFT (a + i b) keeps the fp32 rounding
        # of the untangle (~1e-7 of its partner's amplitude), exactly as at n_fft = 1024
        silent = st["mel_power"] == 0.0
        assert (got["db"][i][silent] == -100.0).all() and (got["mel_power"][i][silent] < 1e-10).all(), (i, len(x))
    if n_mels == 128 and n_fft == 256:
        assert (fb.sum(axis=0) == 0.0).any()          # the case does contain filters without support
        empty = fb.sum(axis=0) == 0.0
        assert (got["db"][:, empty, :] == -100.0).all()


@pytest.mark.parametrize("geo", [GEOMETRIES[0], GEOMETRIES[2], GEOMETRIES[4], GEOMETRIES[5]], ids=lambda g: f"sr{g[0]}_n{g[1]}")
def test_matches_torchaudio_cpu_pipeline(geo):
    """T.MelSpectrogram -> T.AmplitudeToDB -> (x - mean) / (std + eps) on the CPU, on full-length and padded clips."""
    import torchaudio.transforms as TT
    sr, n_fft, hop, n_mels, T = geo
    plan = get_plan(*geo)
    rs = np.random.RandomState(7)
    clips = [(rs.standard_normal(n) * 0.1).astype(np.float32) for n in (T, T // 2 + 1, T)]
    clips[2] = (rs.uniform(-1, 1, T)).astype(np.float32)
    got = run_clips(plan, clips)
    mel = TT.MelSpectrogram(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels)
    to_db = TT.AmplitudeToDB()
    for i, x in enumerate(clips):
        w = torch.zeros(T)
        w[:len(x)] = torch.from_numpy(x)
        db = to_db(mel(w.unsqueeze(0)))[0]
        ref = ((db - db.mean()) / (db.std() + 1e-8)).numpy()
        assert db.shape == (n_mels, plan.frames)
        assert np.abs(got["db"][i] - db.numpy()).max() < DB_ATOL, i
        assert np.abs(got["out"][i] - ref).max() < NORM_ATOL, i


@pytest.mark.parametrize("geo", [GEOMETRIES[0], GEOMETRIES[4]], ids=lambda g: f"sr{g[0]}_n{g[1]}")
def test_seeded_augmentation_with_host_noise(geo):
    """draw_reference_augmentation (roll, host-drawn noise, SpecAugment) replayed on the GPU: the oracle matches and the
    masked rows / frames are exactly the drawn intervals."""
    sr, n_fft, hop, n_mels, T = geo
    plan = get_plan(*geo)
    cfg = oracle_cfg(*geo)
    fb = torchaudio_fb(sr, n_fft, n_mels)
    np.random.seed(42)
    torch.manual_seed(42)
    n = 8
    aug, noise = A.draw_reference_augmentation(n, T, n_mels, cfg.frames)
    noise = np.zeros((n, T), np.float32) if noise is None else noise.numpy()
    assert (aug["noise_scale"] != 0).any() and (aug["shift"] != 0).any()
    rs = np.random.RandomState(3)
    clips = [(rs.standard_normal(m) * 0.1).astype(np.float32) for m in (T, T // 2, T + 999, T, 17, T, T - 5, T)]
    got = run_clips(plan, clips, aug=aug, noise=noise)
    for c in range(n):
        a = aug[c]
        ref = O.logmel(clips[c], cfg, shift=int(a["shift"]), noise=noise[c], noise_scale=float(a["noise_scale"]),
                       masks=(int(a["f0"]), int(a["f1"]), int(a["t0"]), int(a["t1"])), fb=fb)
        assert np.abs(got["out"][c] - ref).max() < NORM_ATOL, c
        z = got["db"][c] == 0.0
        rows, cols = np.nonzero(z.all(axis=1))[0], np.nonzero(z.all(axis=0))[0]
        f0, f1 = (rows[0], rows[-1] + 1) if len(rows) else (0, 0)
        t0, t1 = (cols[0], cols[-1] + 1) if len(cols) else (0, 0)
        want_f = (int(a["f0"]), int(a["f1"])) if a["f1"] > a["f0"] else (0, 0)
        want_t = (int(a["t0"]), int(a["t1"])) if a["t1"] > a["t0"] else (0, 0)
        assert (f0, f1) == want_f and (t0, t1) == want_t, c


@pytest.mark.parametrize("geo", [GEOMETRIES[2], GEOMETRIES[4]], ids=lambda g: f"sr{g[0]}_n{g[1]}")
def test_gain_and_philox_noise(geo):
    """Gain with host noise against the oracle; on-device Philox noise gives finite features, masks inside their
    bounds, and the same features on a second launch."""
    sr, n_fft, hop, n_mels, T = geo
    plan = get_plan(*geo)
    cfg = oracle_cfg(*geo)
    fb = torchaudio_fb(sr, n_fft, n_mels)
    rs = np.random.RandomState(21)
    clips = [(rs.standard_normal(m) * 0.1).astype(np.float32) for m in (T, T - 3000, T + 901)]
    noise = rs.standard_normal((3, T)).astype(np.float32)
    aug = A.make_aug_array(3)
    aug["shift"] = [-(T // 5), T // 5, 1]
    aug["noise_scale"] = [0.005, 0.0, 0.01]
    aug["gain"] = [1.0, 0.5, 2.0]
    aug["f0"], aug["f1"], aug["t0"], aug["t1"] = [0, n_mels - 1, 5], [14, n_mels, 5], [0, 93, 10], [34, 94, 11]
    got = run_clips(plan, clips, aug=aug, noise=noise)
    for i in range(3):
        ref = O.logmel(clips[i], cfg, shift=int(aug[i]["shift"]), noise=noise[i], noise_scale=float(aug[i]["noise_scale"]),
                       gain=float(aug[i]["gain"]), masks=tuple(int(aug[i][k]) for k in ("f0", "f1", "t0", "t1")), fb=fb)
        assert np.abs(got["out"][i] - ref).max() < NORM_ATOL, i
    fast = A.draw_fast_augmentation(16, T, n_mels, cfg.frames, rng=np.random.default_rng(5), gain_db=3.0)
    fast["noise_scale"] = 0.01                                   # every clip draws Philox noise
    xs = [(rs.standard_normal(T) * 0.1).astype(np.float32) for _ in range(16)]
    r1 = run_clips(plan, xs, aug=fast)
    r2 = run_clips(plan, xs, aug=fast)
    assert np.isfinite(r1["out"]).all() and np.isfinite(r1["db"]).all()
    np.testing.assert_array_equal(r1["out"], r2["out"])
    for c in range(16):
        z = r1["db"][c] == 0.0
        rows, cols = np.nonzero(z.all(axis=1))[0], np.nonzero(z.all(axis=0))[0]
        if len(rows):
            assert rows[0] >= fast[c]["f0"] and rows[-1] < fast[c]["f1"]
        if len(cols):
            assert cols[0] >= fast[c]["t0"] and cols[-1] < fast[c]["t1"]


SMALL = [GEOMETRIES[0], GEOMETRIES[4]]


@pytest.mark.parametrize("geo", SMALL, ids=lambda g: f"n{g[1]}")
def test_tma_and_gather_staging_agree_bitwise(geo):
    plan = get_plan(*geo)
    T = geo[4]
    rs = np.random.RandomState(3)
    clips = [(rs.standard_normal(m) * 0.1).astype(np.float32) for m in (T, T, T // 2, T + 50, 3)]
    plan.set("tma", 1)
    a = run_clips(plan, clips, want_stages=False)["out"]
    plan.set("tma", 0)
    b = run_clips(plan, clips, want_stages=False)["out"]
    plan.set("tma", 1)
    np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("geo", SMALL, ids=lambda g: f"n{g[1]}")
def test_small_batch_split_and_batch_position(geo):
    """split 1 / automatic / 3 are bit-identical (masks, rolls, silent tiles, all three outputs); a clip's features do
    not depend on where it sits in the batch or on the grid size."""
    plan = get_plan(*geo)
    T = geo[4]
    rs = np.random.RandomState(21)
    for lens in ([T], [T, T // 3, T + 777], [int(rs.randint(200, 2 * T)) for _ in range(32)]):
        clips = [(rs.standard_normal(m) * 0.1).astype(np.float32) for m in lens]
        aug = A.make_aug_array(len(clips))
        aug["f0"], aug["f1"], aug["t0"], aug["t1"] = 10, 17, 100, 131
        aug["shift"][::2] = 1234
        plan.set("split", 1)
        ref = run_clips(plan, clips, aug=aug)
        plan.set("split", 0)
        got = run_clips(plan, clips, aug=aug)
        for key in ("out", "db", "mel_power"):
            np.testing.assert_array_equal(got[key], ref[key])
        plan.set("split", 3)
        got3 = run_clips(plan, clips, aug=aug, want_stages=False)
        plan.set("split", 0)
        np.testing.assert_array_equal(got3["out"], ref["out"])
    clips = [(rs.standard_normal(T) * 0.1).astype(np.float32) for _ in range(300)]
    full = run_clips(plan, clips, want_stages=False)["out"]
    np.testing.assert_array_equal(full[217], run_clips(plan, [clips[217]], want_stages=False)["out"][0])
    np.testing.assert_array_equal(full[5], run_clips(plan, clips[3:9], want_stages=False)["out"][2])
    plan.set("max_ctas", 1)
    one = run_clips(plan, clips[:3], want_stages=False)["out"]
    plan.set("max_ctas", 0)
    np.testing.assert_array_equal(full[:3], one)


@pytest.mark.parametrize("geo", SMALL, ids=lambda g: f"n{g[1]}")
def test_pcm16_kernel_and_host_paths_are_bit_identical(geo):
    """lm_forward_pcm16 == lm_pcm16_decode + lm_forward (8-sample aligned and odd starts, augmented clips, normalised and
    not); lm_forward_host (fp32 and int16) == the device path."""
    plan = get_plan(*geo)
    dev = plan.device
    T = geo[4]
    rs = np.random.RandomState(31)
    lens = [T, T, T // 7, T + 1, 0, T + T // 4, T, 7, T - 100, T, T, 300]
    starts, pos = [], 0
    for i, n in enumerate(lens):
        pos = (pos + 7) // 8 * 8 + (3 if i in (3, 6, 10) else 0)
        starts.append(pos)
        pos += n
    pcm = torch.from_numpy(rs.randint(-32768, 32768, size=pos + 8).astype(np.int16)).to(dev)
    offset = torch.tensor(starts, dtype=torch.int64, device=dev)
    length = torch.tensor(lens, dtype=torch.int32, device=dev)
    dec = plan.pcm16_decode(pcm)
    B = len(lens)
    aug = A.make_aug_array(B)
    aug["shift"][1], aug["gain"][1] = 4001, 0.5
    aug["noise_scale"][5], aug["seed"][5] = 0.01, 99
    aug["noise_scale"][9] = 0.005
    aug["f0"][2], aug["f1"][2], aug["t0"][2], aug["t1"][2] = 3, 17, 10, 40
    noise = torch.from_numpy(rs.standard_normal((B, T)).astype(np.float32)).to(dev)
    d_aug = plan.upload_aug(aug)
    for kw in (dict(), dict(normalize=False), dict(aug=d_aug, noise=noise), dict(aug=d_aug)):
        want = plan.forward(dec, offset, length, **kw)
        got = plan.forward_pcm16(pcm, offset, length, **kw)
        torch.cuda.synchronize()
        assert torch.equal(got, want), kw.keys()
    for i in (0, 3, 8):                                           # small batches: split over many groups
        want = plan.forward(dec, offset[i:i + 1], length[i:i + 1])
        got = plan.forward_pcm16(pcm, offset[i:i + 1], length[i:i + 1])
        torch.cuda.synchronize()
        assert torch.equal(got, want), i
    want = plan.forward(dec, offset, length)
    host_pcm = pcm.cpu().pin_memory()
    out_h16 = plan.forward_host(host_pcm, offset.cpu(), length.cpu())
    out_h32 = plan.forward_host(dec.cpu().pin_memory(), offset.cpu(), length.cpu())
    torch.cuda.synchronize()
    assert torch.equal(out_h16, want.cpu()) and torch.equal(out_h32, want.cpu())


@pytest.mark.parametrize("geo", SMALL, ids=lambda g: f"n{g[1]}")
def test_extra_outputs_are_consistent_with_the_features(geo):
    """out_db normalised in float64 gives out_norm; out_db is 10 log10(max(out_melpow, amin)) away from the masks."""
    plan = get_plan(*geo)
    T = geo[4]
    rs = np.random.RandomState(9)
    clips = [(rs.standard_normal(m) * 0.1).astype(np.float32) for m in (T, T // 3, T + 5)]
    aug = A.make_aug_array(3)
    aug["f0"][1], aug["f1"][1], aug["t0"][1], aug["t1"][1] = 2, 9, 30, 60
    got = run_clips(plan, clips, aug=aug)
    plain = run_clips(plan, clips, aug=aug, want_stages=False)["out"]
    np.testing.assert_allclose(got["out"], plain, rtol=0, atol=1e-6)
    for i in range(3):
        db = got["db"][i].astype(np.float64)
        assert np.abs((db - db.mean()) / (db.std(ddof=1) + 1e-8) - got["out"][i]).max() < 1e-4
        keep = db != 0.0
        ref = 10.0 * np.log10(np.maximum(got["mel_power"][i].astype(np.float64), 1e-10))
        assert np.abs(db - ref)[keep].max() < 1e-4


def test_forward_gather_stores_are_bit_identical():
    """lm_forward_gather's fused stores (here into two extra buffers on the same GPU standing in for peers) carry
    exactly lm_forward's features at a small n_fft."""
    plan = get_plan(*GEOMETRIES[4])
    dev = plan.device
    T, B = plan.target_length, 300
    g = torch.Generator(device=dev).manual_seed(4)
    lens = torch.randint(100, 2 * T, (B,), generator=g, device=dev, dtype=torch.int64)
    starts = torch.cumsum((lens + 7) // 8 * 8, 0) - (lens + 7) // 8 * 8
    wave = torch.randn(int(starts[-1] + lens[-1]) + 8, generator=g, device=dev) * 0.1
    offset, length = starts.contiguous(), lens.to(torch.int32)
    want = plan.forward(wave, offset, length)
    own = torch.full_like(want, float("nan"))
    peers = [torch.full_like(want, float("nan")) for _ in range(2)]
    plan.forward_gather(wave, offset, length, own.data_ptr(), [p.data_ptr() for p in peers])
    torch.cuda.synchronize()
    assert torch.equal(own, want) and all(torch.equal(p, want) for p in peers)


def test_forward_gather_checks_aug_and_noise():
    """forward_gather refuses aug / noise tensors that do not cover the batch, as forward does (the kernel would read
    past them)."""
    plan = get_plan(*GEOMETRIES[4])
    dev = plan.device
    T, B = plan.target_length, 4
    wave = torch.zeros(B * T, device=dev)
    offset = torch.arange(B, device=dev, dtype=torch.int64) * T
    length = torch.full((B,), T, device=dev, dtype=torch.int32)
    own = torch.empty(plan.out_shape(B), device=dev)
    short_aug = plan.upload_aug(A.make_aug_array(B - 1))
    with pytest.raises(ValueError, match="aug"):
        plan.forward_gather(wave, offset, length, own.data_ptr(), aug=short_aug)
    with pytest.raises(ValueError, match="noise"):
        plan.forward_gather(wave, offset, length, own.data_ptr(), noise=torch.zeros(B - 1, T, device=dev))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_fused_gather_across_gpus_small_fft():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29612", os.path.join(ROOT, "tests", "multi_gpu_small_fft_gather.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "SMALL_FFT_GATHER_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_icbhi_dataset_at_4khz_resamples_and_collates(tmp_path):
    """The drop-in at {sample_rate: 4000, n_fft: 256, hop_length: 64, n_mels: 64, duration: 5.0}: 10 kHz, 44.1 kHz and
    4 kHz PCM_16 recordings through raw() + GpuCollate, against the oracle applied to torchaudio's T.Resample output."""
    import torchaudio.transforms as TT
    d = tmp_path / "audio_and_txt_files"
    d.mkdir()
    rs = np.random.RandomState(6)
    rates = [10000, 44100, 4000, 44100, 10000, 4000]
    secs = [4, 6, 5, 3, 5, 2]
    sigs = []
    for i, (sr, s) in enumerate(zip(rates, secs)):
        x = (rs.standard_normal(sr * s) * 0.1).clip(-1, 1)
        sigs.append(x)
        wavio.write_wav_pcm16(str(d / f"{100 + i}_r.wav"), x, sr)
        (d / f"{100 + i}_r.txt").write_text(f"0.0\t1.0\t{i % 2}\t0\n")
    cfg = {"data": dict(sample_rate=4000, n_fft=256, hop_length=64, n_mels=64, duration=5.0)}
    ds = A.ICBHIDataset(tmp_path, "test", cfg)
    ds.data = [(str(d / f"{100 + i}_r.wav"), i % 2) for i in range(len(rates))]
    loader = torch.utils.data.DataLoader(ds.raw(), batch_size=3, shuffle=False, num_workers=0,
                                         collate_fn=A.GpuCollate(ds.preprocessor))
    feats, labels = [], []
    for f, y in loader:
        assert f.is_cuda and f.shape == (3, 1, 64, 313)
        feats.append(f)
        labels += y.tolist()
    assert labels == [i % 2 for i in range(len(rates))]
    feats = torch.cat(feats).cpu().numpy()
    ocfg = O.OracleConfig(sample_rate=4000, n_fft=256, hop_length=64, n_mels=64, duration=5.0)
    fb = torchaudio_fb(4000, 256, 64)
    for i, sr in enumerate(rates):
        xq = torch.from_numpy((np.rint(sigs[i] * 32767) / 32768.0).astype(np.float32))
        x4 = xq if sr == 4000 else TT.Resample(sr, 4000)(xq.unsqueeze(0))[0]
        ref = O.logmel(x4.numpy(), ocfg, fb=fb)
        # as for 16 kHz targets (test_gpu_dropin): the bands above the resampler's cut-off are nearly empty, where a
        # 1e-6 waveform difference between the fp32 resampler and torchaudio's moves a dB value visibly
        tol = NORM_ATOL if sr == 4000 else 5e-3
        assert np.abs(feats[i, 0] - ref).max() < tol, (i, sr)
