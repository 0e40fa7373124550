"""ctypes binding of liblogmel_b200.so (include/logmel_b200.h).

There is no CPU fallback: if the shared library is missing or a CUDA device is absent every
entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "liblogmel_b200.so")

LM_OK = 0
LM_MAX_RESAMPLERS = 8   # rate pairs of one lm_forward_resampled call


class LmConfig(C.Structure):
    _fields_ = [
        ("n_fft", C.c_int32), ("hop", C.c_int32), ("n_mels", C.c_int32), ("target_len", C.c_int32),
        ("window", C.POINTER(C.c_float)), ("fb", C.POINTER(C.c_float)),
        ("db_multiplier", C.c_float), ("amin", C.c_float), ("db_offset", C.c_float), ("norm_eps", C.c_float),
    ]


class LmAug(C.Structure):
    _fields_ = [
        ("shift", C.c_int32), ("noise_scale", C.c_float), ("gain", C.c_float),
        ("f0", C.c_int32), ("f1", C.c_int32), ("t0", C.c_int32), ("t1", C.c_int32),
        ("flags", C.c_int32), ("seed", C.c_uint64),
    ]


class LmInfo(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("frames", C.c_int32), ("n_freqs", C.c_int32), ("sm_count", C.c_int32),
        ("threads_per_cta", C.c_int32), ("smem_bytes", C.c_int32), ("fb_nnz", C.c_int32),
        ("tma_staging", C.c_int32), ("bytes_per_clip", C.c_int64),
    ]


assert C.sizeof(LmAug) == 40, "lm_aug layout drifted from include/logmel_b200.h"

# numpy dtype with the same layout as lm_aug (used to build [B] arrays on the host)
AUG_DTYPE = [("shift", "<i4"), ("noise_scale", "<f4"), ("gain", "<f4"), ("f0", "<i4"), ("f1", "<i4"),
             ("t0", "<i4"), ("t1", "<i4"), ("flags", "<i4"), ("seed", "<u8")]

EXPORTS = {
    "lm_abi_version": (C.c_int, []),
    "lm_strerror": (C.c_char_p, [C.c_int]),
    "lm_last_cuda_error": (C.c_char_p, []),
    "lm_plan_create": (C.c_int, [C.POINTER(LmConfig), C.c_int, C.POINTER(C.c_void_p)]),
    "lm_plan_destroy": (C.c_int, [C.c_void_p]),
    "lm_plan_frames": (C.c_int, [C.c_void_p]),
    "lm_plan_info": (C.c_int, [C.c_void_p, C.POINTER(LmInfo)]),
    "lm_plan_set": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "lm_plan_launch_count": (C.c_int64, [C.c_void_p]),
    "lm_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "lm_resize_finish": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_int32, C.c_float, C.c_void_p]),
    "lm_pcm16_roundtrip": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "lm_forward_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "lm_forward_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "lm_pcm16_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "lm_amplitude_to_db": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "lm_resampler_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int, C.POINTER(C.c_void_p)]),
    "lm_resampler_destroy": (C.c_int, [C.c_void_p]),
    "lm_resampler_out_len": (C.c_int64, [C.c_void_p, C.c_int64]),
    "lm_resample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "lm_resample_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int64,
                                   C.c_void_p]),
    "lm_forward_host_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "lm_forward_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "lm_forward_resampled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "lm_clip_span": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "lm_forward_spans": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int32, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the library once; raises RuntimeError (never falls back) when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is not built. Run `python -m audio_classification_icbhi_b200.build` "
            "(needs nvcc). The log-mel path has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.lm_abi_version() != 1:
        raise RuntimeError("liblogmel_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != LM_OK:
        lib = load()
        msg = lib.lm_strerror(status).decode()
        detail = lib.lm_last_cuda_error().decode()
        raise RuntimeError(f"liblogmel_b200: {msg}" + (f" [{detail}]" if detail and status == -4 else ""))
