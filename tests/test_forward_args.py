"""lm_forward, lm_forward_pcm16, lm_forward_gather and the host-buffer entry points refuse bad arguments with
LM_ERR_INVALID_ARG, and accept an empty batch, before they touch a device (no GPU).  The statuses and the order of
the checks are part of the C ABI: a caller tells a bad argument from an empty batch by them."""
import ctypes as C

import numpy as np
import pytest

INVALID = -1


@pytest.fixture(scope="module")
def lib():
    from audio_classification_icbhi_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


# A stand-in plan handle, all zeros: the checks below either fail before the library dereferences it or, for the
# gather's alignment checks, read only its (zero) mel and frame counts.
FAKE_PLAN = C.create_string_buffer(4096)
BUF = C.create_string_buffer(64)   # stand-in for device arrays; never read
P = C.addressof(BUF)               # 16-byte aligned (ctypes buffers come from malloc)


@pytest.mark.parametrize("entry", ["lm_forward", "lm_forward_pcm16"])
def test_forward_refuses_bad_arguments(lib, entry):
    def call(plan=FAKE_PLAN, wave=P, offset=P, length=P, B=1, out=P):
        if entry == "lm_forward":
            return lib.lm_forward(plan, wave, offset, length, B, None, None, out, None, None, 1, None)
        return lib.lm_forward_pcm16(plan, wave, offset, length, B, None, None, out, 1, None)

    assert call(plan=None) == INVALID
    assert call(B=-1) == INVALID
    assert call(plan=None, B=0) == INVALID   # the plan is checked before the batch size
    for name in ("wave", "offset", "length", "out"):
        assert call(**{name: None}) == INVALID, name
        assert call(B=0, **{name: None}) == 0, name   # an empty batch needs no arrays
    assert call(B=0) == 0


def test_forward_gather_refuses_bad_arguments(lib):
    peers = (C.c_void_p * 7)(*([P] * 7))

    def call(plan=FAKE_PLAN, wave=P, offset=P, length=P, B=1, out=P, peer=None, n_peers=0, mc=None):
        return lib.lm_forward_gather(plan, wave, offset, length, B, None, None, out, peer, n_peers, mc, None)

    assert call(plan=None) == INVALID
    assert call(B=-1) == INVALID
    assert call(plan=None, B=0) == INVALID
    for n in (-1, 8):   # at most 7 peers; the count is checked before the batch size
        assert call(n_peers=n, peer=peers) == INVALID, n
        assert call(n_peers=n, peer=peers, B=0) == INVALID, n
    for name in ("wave", "offset", "length", "out"):
        assert call(**{name: None}) == INVALID, name
        assert call(B=0, **{name: None}) == 0, name
    assert call(n_peers=1, peer=None) == INVALID
    assert call(n_peers=1, peer=None, B=0) == 0
    assert call(B=0) == 0
    # the gather rides on 16-byte stores: every destination must be 16-byte aligned
    assert P % 16 == 0
    assert call(out=P + 4) == INVALID
    assert call(mc=P + 8) == INVALID
    assert call(n_peers=2, peer=(C.c_void_p * 2)(P, None)) == INVALID
    assert call(n_peers=2, peer=(C.c_void_p * 2)(P, P + 4)) == INVALID


@pytest.mark.parametrize("entry", ["lm_forward_host", "lm_forward_host_pcm16"])
def test_forward_host_refuses_bad_arguments(lib, entry):
    wave = np.zeros(64, dtype=np.float32)
    off = np.zeros(2, dtype=np.int64)
    ln = np.full(2, 16, dtype=np.int32)

    def call(plan=FAKE_PLAN, wave=wave.ctypes.data, total=64, offset=off, length=ln, B=2, out=P):
        o = offset.ctypes.data if isinstance(offset, np.ndarray) else offset
        n = length.ctypes.data if isinstance(length, np.ndarray) else length
        return getattr(lib, entry)(plan, wave, total, o, n, B, None, None, out, 1)

    assert call(plan=None) == INVALID
    assert call(B=-1) == INVALID
    assert call(total=-1) == INVALID
    assert call(plan=None, B=0) == INVALID
    assert call(total=-1, B=0) == INVALID
    for name in ("wave", "offset", "length", "out"):
        assert call(**{name: None}) == INVALID, name
        assert call(B=0, **{name: None}) == 0, name
    assert call(B=0) == 0
    # every clip must lie inside the buffer's total_samples
    assert call(total=31, offset=np.array([0, 16], dtype=np.int64)) == INVALID
    assert call(total=20, offset=np.array([0, 5], dtype=np.int64)) == INVALID
    assert call(offset=np.array([0, -1], dtype=np.int64)) == INVALID
    assert call(length=np.array([16, -1], dtype=np.int32)) == INVALID
