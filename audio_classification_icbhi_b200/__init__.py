"""B200-native (sm_100a) log-mel front end for the ICBHI lung-sound classifier.

Drop-in for the preprocessing path of AkZuza/audio-classification-icbhi
(src/data/preprocessing.py, data/preprocessing_flexible.py and their dataset / analyzer /
segmenter callers).  All arithmetic of the path runs in hand-written CUDA behind a C ABI
(include/logmel_b200.h); there is no CPU fallback.  `compat/` at the repository root holds import
shims under the reference's own module paths.
"""
from .plan import LogMelPlan, clip_span, make_aug_array, reference_filterbank, reference_window
from .preprocessing import AudioPreprocessor
from .preprocessing_flexible import FlexibleAudioPreprocessor
from .dataset import GpuCollate, GpuLoader, ICBHIDataset, ICBHISegmentedDataset, SpanItem, raw_collate
from .analyzer import SlidingWindowLogMel, segment_offsets
from .segmenter import ICBHISegmenter
from .sharding import FusedGather, ShardedLogMel, shard_bounds, shard_size
from .augment import draw_fast_augmentation, draw_reference_augmentation
from .resample import Resampler, get_resampler

__all__ = [
    "LogMelPlan", "clip_span", "make_aug_array", "reference_filterbank", "reference_window",
    "AudioPreprocessor", "FlexibleAudioPreprocessor",
    "ICBHIDataset", "ICBHISegmentedDataset", "GpuCollate", "GpuLoader", "raw_collate", "SpanItem",
    "SlidingWindowLogMel", "segment_offsets", "ICBHISegmenter",
    "ShardedLogMel", "FusedGather", "shard_bounds", "shard_size",
    "draw_fast_augmentation", "draw_reference_augmentation",
    "Resampler", "get_resampler",
]
__version__ = "0.1.0"
