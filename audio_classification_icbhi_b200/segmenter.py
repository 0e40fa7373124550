"""Drop-in `ICBHISegmenter` (reference: R/preprocess_icbhi.py:20-239): one-off offline slicing of
ICBHI recordings into per-cycle clips, class directories and a stats JSON.

This is file plumbing around the hot path (SURVEY.md section 8f "next"): decode, slice by
annotation row, drop cycles shorter than `min_duration`, write PCM_16 wavs.  Decoding uses the
stdlib reader in wavio.py (librosa / soundfile are not in the image); recordings whose rate
differs from `sample_rate` are resampled with the library's CUDA port of torchaudio's sinc resampler
(resample.py) -- librosa's soxr resampler is a different filter, so resampled segments are "parity unpinned".
`segments_to_features` is the new bit: the cycles of a recording go to the GPU as (offset, length)
pairs into the one uploaded recording, with no intermediate files.
"""
from __future__ import annotations

import json
from functools import partial
from pathlib import Path
from typing import List, Tuple

import numpy as np
import torch

from .wavio import read_wav, write_wav_pcm16

__all__ = ["ICBHISegmenter"]

CLASS_NAMES = ("normal", "crackle", "wheeze", "both")


class ICBHISegmenter:
    """Segment ICBHI audio files based on respiratory cycle annotations."""

    def __init__(self, input_dir, output_dir, sample_rate=16000, min_duration=0.5):
        self.input_dir = Path(input_dir)
        self.output_dir = Path(output_dir)
        self.sample_rate = sample_rate
        self.min_duration = min_duration
        self.create_output_dirs()
        self.stats = {name: 0 for name in CLASS_NAMES}
        self.stats.update(total_files=0, total_segments=0, skipped_segments=0)

    def create_output_dirs(self):
        self.output_dir.mkdir(parents=True, exist_ok=True)
        for name in CLASS_NAMES:
            (self.output_dir / name).mkdir(exist_ok=True)
        print(f"Created output directory: {self.output_dir}")

    def parse_annotation(self, txt_file) -> List[Tuple[float, float, int, int]]:
        """Rows `start<TAB>end<TAB>crackles<TAB>wheezes` -> [(start, end, crackle, wheeze)];
        unparsable rows are reported and skipped."""
        rows = []
        try:
            with open(txt_file, "r") as f:
                for line in f:
                    cols = line.strip().split("\t")
                    if len(cols) < 4:
                        continue
                    try:
                        rows.append((float(cols[0]), float(cols[1]), int(cols[2]), int(cols[3])))
                    except ValueError:
                        print(f"  Warning: Could not parse line in {Path(txt_file).name}: {line.strip()}")
        except OSError as e:
            print(f"  Error reading {txt_file}:  {e}")
        return rows

    def get_label(self, crackle, wheeze) -> str:
        if crackle == 1 and wheeze == 1:
            return "both"
        if crackle == 1:
            return "crackle"
        if wheeze == 1:
            return "wheeze"
        return "normal"

    def _load(self, audio_path) -> np.ndarray:
        data, sr = read_wav(str(audio_path))
        mono = data.mean(axis=0) if data.shape[0] > 1 else data[0]
        if sr != self.sample_rate:
            from .resample import get_resampler
            mono = get_resampler(int(sr), int(self.sample_rate))(torch.from_numpy(np.ascontiguousarray(mono, dtype=np.float32))).cpu().numpy()
        return np.ascontiguousarray(mono, dtype=np.float32)

    def cycle_table(self, n_samples: int, annotations) -> List[Tuple[int, int, int, str]]:
        """(row index, start sample, length, label) of the cycles that survive `min_duration`."""
        table = []
        for idx, (start, end, crackle, wheeze) in enumerate(annotations):
            s = int(start * self.sample_rate)
            e = int(end * self.sample_rate)
            s_c, e_c = min(max(s, 0), n_samples), min(max(e, 0), n_samples)   # python slice semantics
            length = max(e_c - s_c, 0)
            if length / self.sample_rate < self.min_duration:
                self.stats["skipped_segments"] += 1
                continue
            table.append((idx, s_c, length, self.get_label(crackle, wheeze)))
        return table

    def segment_audio(self, audio_path, txt_path) -> int:
        audio_path = Path(audio_path)
        try:
            audio = self._load(audio_path)
        except Exception as e:
            print(f"  Error loading {audio_path.name}: {e}")
            return 0
        annotations = self.parse_annotation(txt_path)
        if not annotations:
            print(f"  Warning: No valid annotations for {audio_path.name}")
            return 0
        made = 0
        for idx, start, length, label in self.cycle_table(len(audio), annotations):
            name = f"{audio_path.stem}_seg{idx:03d}_{label}.wav"
            try:
                write_wav_pcm16(str(self.output_dir / label / name), audio[start:start + length], self.sample_rate)
            except OSError as e:
                print(f"  Error saving segment {name}: {e}")
                continue
            made += 1
            self.stats[label] += 1
            self.stats["total_segments"] += 1
        return made

    def segments_to_features(self, audio_path, txt_path, preprocessor):
        """GPU shortcut: features of every surviving cycle of one recording, straight from the
        decoded recording (no wav files).  Returns (features [n,1,n_mels,frames], labels)."""
        audio = self._load(audio_path)
        table = self.cycle_table(len(audio), self.parse_annotation(txt_path))
        plan = preprocessor.plan
        if not table:
            return torch.empty(plan.out_shape(0), device=plan.device), []
        rec = torch.from_numpy(audio).to(plan.device)
        offset = torch.tensor([t[1] for t in table], dtype=torch.int64, device=plan.device)
        length = torch.tensor([t[2] for t in table], dtype=torch.int32, device=plan.device)
        feats = preprocessor._finish(plan, partial(plan.forward, rec, offset, length), None, None)
        return feats, [t[3] for t in table]

    def process_all(self):
        audio_files = list(self.input_dir.glob("*.wav"))
        if not audio_files:
            print(f"No .  wav files found in {self.input_dir}")
            return
        print(f"\nFound {len(audio_files)} audio files")
        print(f"Sample rate: {self.sample_rate} Hz")
        print(f"Minimum segment duration: {self.min_duration} seconds")
        for audio_path in audio_files:
            txt_path = audio_path.with_suffix(".txt")
            if not txt_path.exists():
                print(f"Warning: No annotation file for {audio_path.name}")
                continue
            self.segment_audio(audio_path, txt_path)
            self.stats["total_files"] += 1
        self.print_summary()
        self.save_stats()

    def print_summary(self):
        total = max(1, self.stats["total_segments"])
        print("\n" + "=" * 60 + "\nSEGMENTATION COMPLETE\n" + "=" * 60)
        print(f"Files processed: {self.stats['total_files']}")
        print(f"Total segments created: {self.stats['total_segments']}")
        print(f"Segments skipped (too short): {self.stats['skipped_segments']}")
        print("\nClass distribution:")
        for name in CLASS_NAMES:
            print(f"  {name.capitalize():8s} {self.stats[name]:4d} ({100 * self.stats[name] / total:.1f}%)")
        print("=" * 60 + f"\n\nSegmented files saved to: {self.output_dir}")

    def save_stats(self):
        stats_file = self.output_dir / "segmentation_stats.json"
        with open(stats_file, "w") as f:
            json.dump(self.stats, f, indent=2)
        print(f"Statistics saved to:  {stats_file}")


def main(argv=None):
    """CLI with the reference's flags (R/preprocess_icbhi.py:242-283)."""
    import argparse
    ap = argparse.ArgumentParser(description="Segment ICBHI dataset by respiratory cycles")
    ap.add_argument("--input-dir", type=str, default="data/ICBHI/audio_and_txt_files")
    ap.add_argument("--output-dir", type=str, default="data/ICBHI_segmented")
    ap.add_argument("--sample-rate", type=int, default=16000)
    ap.add_argument("--min-duration", type=float, default=0.5)
    a = ap.parse_args(argv)
    ICBHISegmenter(a.input_dir, a.output_dir, a.sample_rate, a.min_duration).process_all()


if __name__ == "__main__":
    main()
