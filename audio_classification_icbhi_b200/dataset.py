"""Drop-in ICBHI datasets (reference: R/src/data/dataset.py:11-147, R/src/data/dataset_segmented.py:9-138).

Signatures, `CLASS_MAP`, `.data` (list of `(path, label)`), `.preprocessor`, split arithmetic and
error behaviour follow the reference.  `__getitem__` still returns `(mel_spec, label)` with
`mel_spec` a `[1, n_mels, frames]` float32 CPU tensor, so existing loops keep working -- but the
intended use on a B200 is the raw mode: workers (or the main process) hand back waveforms,
`GpuCollate` turns a whole batch into features with ONE kernel launch in the training process
(CUDA cannot be used in forked DataLoader workers; trainer_fixed.py:35-50 forks 4 of them).
"""
from __future__ import annotations

import random
from pathlib import Path
from typing import List, NamedTuple, Sequence, Tuple

import numpy as np
import torch
from torch.utils.data import Dataset

from .plan import clip_span
from .preprocessing import AudioPreprocessor
from .wavio import read_wav_span, wav_info

__all__ = ["ICBHIDataset", "ICBHISegmentedDataset", "GpuCollate", "GpuLoader", "raw_collate", "SpanItem"]


class SpanItem(NamedTuple):
    """A raw item that carries only the native samples its features read (`raw_span_item`)."""
    samples: np.ndarray   # int16 (mono 16-bit PCM files) or float32: native samples [first, first + len(samples))
    rate: int             # the file's sample rate
    length: int           # native samples of the whole recording
    first: int
    label: int


def _build_preprocessor(config, augment: bool) -> AudioPreprocessor:
    if config:
        d = config["data"]
        return AudioPreprocessor(sample_rate=d["sample_rate"], n_mels=d["n_mels"], n_fft=d["n_fft"],
                                 hop_length=d["hop_length"], duration=d["duration"], augment=augment)
    return AudioPreprocessor(augment=augment)


class _RawMixin:
    """Raw mode shared by both datasets."""

    def raw_item(self, idx) -> Tuple[torch.Tensor, int, int]:
        """(waveform `[1, len]` float32 mono at the FILE's sample rate, that rate, label): decode only.  No CUDA call
        -- raw ICBHI recordings are 4 / 10 / 44.1 kHz and resampling runs on the GPU, which a forked DataLoader
        worker must not touch; `GpuCollate` resamples in the process that owns the context."""
        audio_path, label = self.data[idx]
        waveform, sr = self.preprocessor.decode_audio(audio_path)
        return waveform, sr, label

    def raw_span_item(self, idx) -> SpanItem:
        """Like `raw_item`, but reads only the samples of the recording that the features use: the span that
        `clip_span` gives for the file's length and rate and the preprocessor's rate and target length (roll, noise,
        gain and masks act inside the crop, so augmentation does not widen it).  A mono 16-bit PCM file stays int16.
        Host only: reads the wav header and the span, touches no CUDA."""
        audio_path, label = self.data[idx]
        info = wav_info(audio_path)
        pre = self.preprocessor
        first, count = clip_span(info.rate, pre.sample_rate, pre.target_length, info.frames)
        return SpanItem(read_wav_span(audio_path, first, count), info.rate, info.frames, first, label)

    def raw(self, spans: bool = False) -> "RawView":
        """A Dataset view whose items are `raw_item`s, or `raw_span_item`s with `spans=True` (for DataLoader +
        GpuCollate)."""
        return RawView(self, spans)

    def __len__(self):
        return len(self.data)

    def __getitem__(self, idx):
        audio_path, label = self.data[idx]
        return self.preprocessor.preprocess(audio_path), label


class RawView(Dataset):
    def __init__(self, parent, spans: bool = False):
        self.parent = parent
        self.spans = spans

    def __len__(self):
        return len(self.parent)

    def __getitem__(self, idx):
        return self.parent.raw_span_item(idx) if self.spans else self.parent.raw_item(idx)


class GpuCollate:
    """collate_fn for raw items: list of (waveform, sample_rate, label) -- or (waveform, label) for waveforms already
    at the target rate -- -> (features [B,1,n_mels,frames] on the GPU, labels int64 on the GPU).  The batch is packed
    into one pinned buffer, uploaded with one copy and turned into features by ONE log-mel launch
    (`AudioPreprocessor.preprocess_batch`); recordings at other rates are resampled inside it (`lm_forward_resampled`).
    It must run in the process that owns the CUDA context.  A DataLoader calls its collate_fn INSIDE the worker
    processes, so with `num_workers > 0` give the loader `raw_collate` (workers hand back plain lists) and wrap it in
    `GpuLoader(loader, GpuCollate(...))`, which collates in the training process; with `num_workers=0` it can be
    the collate_fn itself.

    Items of `raw(spans=True)` (`SpanItem`s) carry only the native samples their features read.  They are packed the
    same way (int16 when every item is, else fp32 with int16 as x / 32768) and turned into features by
    `LogMelPlan.forward_spans` -- the same features as the whole recordings give.  A span item that misses samples this
    preprocessor's features read (cut for another rate or target length) raises ValueError before CUDA is touched.

    For either kind of item, a batch with more than LM_MAX_RESAMPLERS foreign rates makes one launch per group of at
    most that many rates, each filling its own rows of the output."""

    def __init__(self, preprocessor: AudioPreprocessor, fast_augment: bool = False):
        self.preprocessor = preprocessor
        self.fast_augment = fast_augment

    def __call__(self, batch: Sequence[tuple]):
        pre = self.preprocessor
        spans = [isinstance(item, SpanItem) for item in batch]
        if any(spans):
            if not all(spans):
                raise ValueError("a batch mixes SpanItems with whole-recording items")
            rate = int(pre.sample_rate)
            # An item cut for another rate or target length would come out of the kernel as a silent clip: refuse it
            # here, before anything touches CUDA.
            for it in batch:
                c = int(it.samples.shape[0])
                first, count = clip_span(int(it.rate), rate, pre.target_length, int(it.length))
                if count and not (it.first <= first and first + count <= it.first + c):
                    raise ValueError(f"span item [{it.first}, {it.first + c}) of a {it.length}-sample {it.rate} Hz "
                                     f"recording misses samples [{first}, {first + count}) that {rate} Hz features of "
                                     f"{pre.target_length} samples read")
            feats = pre._features([it.samples for it in batch], [it.rate for it in batch],
                                  first=[int(it.first) for it in batch], length=[int(it.length) for it in batch],
                                  fast_augment=self.fast_augment)
            labels = [int(it.label) for it in batch]
        else:
            waves, rates, labels = [], [], []
            for item in batch:
                w, sr, y = item if len(item) == 3 else (item[0], pre.sample_rate, item[1])
                waves.append(w)
                rates.append(int(sr))
                labels.append(int(y))
            feats = pre.preprocess_batch(waves, fast_augment=self.fast_augment, sample_rates=rates)
        return feats, torch.tensor(labels, dtype=torch.int64).to(feats.device, non_blocking=True)


def raw_collate(batch):
    """collate_fn for `DataLoader(dataset.raw(), num_workers > 0)`: keep the list of raw items as it is (decoded
    waveforms of different lengths and rates cannot be stacked, and the workers must not touch CUDA)."""
    return list(batch)


class GpuLoader:
    """Iterates a DataLoader of raw batches and turns each into (features, labels) on the GPU in THIS process:

        loader = DataLoader(ds.raw(), batch_size=32, shuffle=True, num_workers=4, collate_fn=raw_collate)
        for inputs, labels in GpuLoader(loader, GpuCollate(ds.preprocessor)): ...

    replaces R/src/training/trainer_fixed.py:35-50 + :146-147 (the workers decode, one kernel launch per batch
    extracts the features, `inputs.to(device)` becomes a no-op)."""

    def __init__(self, loader, collate: GpuCollate):
        self.loader, self.collate = loader, collate

    def __len__(self):
        return len(self.loader)

    def __iter__(self):
        for raw in self.loader:
            yield self.collate(raw)


class ICBHIDataset(_RawMixin, Dataset):
    """ICBHI respiratory sound database: <root>/audio_and_txt_files/{*.wav, *.txt}."""

    CLASS_MAP = {"normal": 0, "crackles": 1, "wheezes": 2, "both": 3}

    def __init__(self, root_dir, split="train", config=None, augment=False):
        self.root_dir = Path(root_dir)
        self.split = split
        self.augment = augment and (split == "train")
        self.preprocessor = _build_preprocessor(config, self.augment)
        self.data = self._load_data()

    def _load_data(self) -> List[Tuple[str, int]]:
        audio_dir = self.root_dir / "audio_and_txt_files"
        if not audio_dir.exists():
            raise ValueError(f"Audio directory not found: {audio_dir}")
        pairs = []
        for wav in sorted(audio_dir.glob("*.wav")):
            txt = wav.with_suffix(".txt")
            if txt.exists():
                pairs.append((str(wav), self._parse_annotation(txt)))
        n_train, n_val = int(0.7 * len(pairs)), int(0.15 * len(pairs))   # dataset.py:81-90
        if self.split == "train":
            pairs = pairs[:n_train]
        elif self.split == "val":
            pairs = pairs[n_train:n_train + n_val]
        else:
            pairs = pairs[n_train + n_val:]
        print(f"Loaded {len(pairs)} samples for {self.split} split")
        return pairs

    def _parse_annotation(self, txt_file) -> int:
        """Rows are `start<TAB>end<TAB>crackles<TAB>wheezes`; the recording's label is the union of
        its cycles (dataset.py:95-130)."""
        crackles = wheezes = False
        with open(txt_file, "r") as f:
            for line in f:
                cols = line.strip().split("\t")
                if len(cols) >= 4:
                    crackles |= int(cols[2]) == 1
                    wheezes |= int(cols[3]) == 1
        key = "both" if (crackles and wheezes) else "crackles" if crackles else "wheezes" if wheezes else "normal"
        return self.CLASS_MAP[key]


class ICBHISegmentedDataset(_RawMixin, Dataset):
    """Pre-segmented cycles: <root>/{normal,crackle,wheeze,both}/*.wav."""

    CLASS_MAP = {"normal": 0, "crackle": 1, "wheeze": 2, "both": 3}

    def __init__(self, root_dir, split="train", config=None, augment=False):
        self.root_dir = Path(root_dir)
        self.split = split
        self.augment = augment and (split == "train")
        self.preprocessor = _build_preprocessor(config, self.augment)
        self.data = self._load_data()
        self._split_data(config)

    def _load_data(self) -> List[Tuple[str, int]]:
        pairs = []
        for name, idx in self.CLASS_MAP.items():
            class_dir = self.root_dir / name
            if not class_dir.exists():
                print(f"Warning: Directory not found: {class_dir}")
                continue
            pairs.extend((str(w), idx) for w in class_dir.glob("*.wav"))
        if not pairs:
            raise ValueError(f"No audio files found in {self.root_dir}")
        random.seed(42)            # dataset_segmented.py:90-91: fixed shuffle for consistent splits
        random.shuffle(pairs)
        return pairs

    def _split_data(self, config) -> None:
        total = len(self.data)
        train_split = config["data"].get("train_split", 0.7) if config else 0.7
        val_split = config["data"].get("val_split", 0.15) if config else 0.15
        n_train, n_val = int(train_split * total), int(val_split * total)
        if self.split == "train":
            self.data = self.data[:n_train]
        elif self.split == "val":
            self.data = self.data[n_train:n_train + n_val]
        else:
            self.data = self.data[n_train + n_val:]
        print(f"Loaded {len(self.data)} samples for {self.split} split")
        names = {v: k for k, v in self.CLASS_MAP.items()}
        counts = {}
        for _, label in self.data:
            counts[names[label]] = counts.get(names[label], 0) + 1
        print(f"Class distribution for {self.split}:")
        for name, count in sorted(counts.items()):
            print(f"  {name}: {count} ({100 * count / max(len(self.data), 1):.1f}%)")
