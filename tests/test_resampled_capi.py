"""lm_forward_resampled refuses bad arguments with LM_ERR_INVALID_ARG before it touches the plan or a device (no GPU)."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from audio_classification_icbhi_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def test_max_resamplers_matches_the_header():
    import os
    import re
    from audio_classification_icbhi_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "logmel_b200.h")).read()
    assert int(re.search(r"#define LM_MAX_RESAMPLERS (\d+)", text).group(1)) == _lib.LM_MAX_RESAMPLERS == 8


def test_invalid_arguments_without_a_device(lib):
    # A stand-in plan handle: every check below must fail before the library dereferences it.
    fake_plan = C.create_string_buffer(64)
    buf = C.create_string_buffer(64)   # stand-in for device arrays; never read
    p = C.addressof(buf)
    one_null = (C.c_void_p * 1)(None)

    def call(plan=fake_plan, rs=None, n=0, wave=p, pcm16=0, offset=p, length=p, source=p, B=1, out=p):
        return lib.lm_forward_resampled(plan, rs, n, wave, pcm16, offset, length, source, B, None, None, out, 1, None)

    assert call(plan=None) == -1
    assert call(n=-1) == -1
    assert call(n=9) == -1                 # more than LM_MAX_RESAMPLERS
    assert call(n=1, rs=None) == -1        # NULL array
    assert call(n=1, rs=one_null) == -1    # NULL handle
    assert call(pcm16=2) == -1
    assert call(B=-1) == -1
    for name in ("wave", "offset", "length", "source", "out"):
        assert call(**{name: None}) == -1, name
    assert call(plan=None, B=0) == -1
    assert call(B=0) == 0                  # an empty batch is a no-op
