"""The second-stage networks of the 512- and 256-point FFTs (csrc/fft_gen.cuh: lm_fft16x2_soa, lm_fft8x4_soa and
the scalar lm_fft8) compiled with g++ through lm_f2.cuh, checked against numpy and against the scalar flavour."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "audio_classification_icbhi_b200", "csrc")

HARNESS = r"""
#include "fft_gen.cuh"
extern "C" void fft8(float* re, float* im){ float a[8], b[8]; for(int i=0;i<8;i++){a[i]=re[i];b[i]=im[i];} lm_fft8(a,b); for(int i=0;i<8;i++){re[i]=a[i];im[i]=b[i];} }
extern "C" void fft16(float* re, float* im){ float a[16], b[16]; for(int i=0;i<16;i++){a[i]=re[i];b[i]=im[i];} lm_fft16(a,b); for(int i=0;i<16;i++){re[i]=a[i];im[i]=b[i];} }
#define SOA(name, fn) extern "C" void name(float* re, float* im){ lm_f2 pr[16], pi[16]; for(int m=0;m<16;m++){ pr[m]=lm_pack(re[2*m],re[2*m+1]); pi[m]=lm_pack(im[2*m],im[2*m+1]); } float a[32], b[32]; fn(pr,pi,a,b); for(int i=0;i<32;i++){re[i]=a[i];im[i]=b[i];} }
SOA(fft16x2_soa, lm_fft16x2_soa)
SOA(fft8x4_soa, lm_fft8x4_soa)
"""

P = ctypes.POINTER(ctypes.c_float)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("fft_small")
    src = d / "h.cpp"
    src.write_text(HARNESS)
    so = d / "h.so"
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-I", CSRC, str(src), "-o", str(so)], check=True)
    return ctypes.CDLL(str(so))


def _inputs(n, count, seed):
    """Impulses at point 1 (every twiddle) and at point 0 of each transform, then random complex vectors."""
    total = n * count
    rs = np.random.RandomState(seed)
    for trial in range(20):
        if trial < 2:
            x = np.zeros(total, dtype=complex)
            x[1 - trial::n] = 1.0
        else:
            x = rs.standard_normal(total) + 1j * rs.standard_normal(total)
        yield x


@pytest.mark.parametrize("name,n,count", [("fft8", 8, 1), ("fft16", 16, 1), ("fft16x2_soa", 16, 2), ("fft8x4_soa", 8, 4)])
def test_fft_matches_numpy(harness, name, n, count):
    """Each of the `count` independent n-point transforms of a call matches numpy (relative error < 5e-7)."""
    f = getattr(harness, name)
    worst = 0.0
    for x in _inputs(n, count, 0):
        re, im = x.real.astype(np.float32), x.imag.astype(np.float32)
        ref = np.fft.fft((re.astype(np.float64) + 1j * im.astype(np.float64)).reshape(count, n), axis=1).reshape(-1)
        f(re.ctypes.data_as(P), im.ctypes.data_as(P))
        worst = max(worst, np.abs((re + 1j * im) - ref).max() / np.abs(ref).max())
    assert worst < 5e-7


@pytest.mark.parametrize("packed,scalar,n", [("fft16x2_soa", "fft16", 16), ("fft8x4_soa", "fft8", 8)])
def test_packed_and_scalar_flavours_agree(harness, packed, scalar, n):
    """Same butterfly network, same Linzer-Feig constants: the packed batch equals the scalar transform of each slice."""
    rs = np.random.RandomState(3)
    x = rs.standard_normal(32) + 1j * rs.standard_normal(32)
    re, im = x.real.astype(np.float32), x.imag.astype(np.float32)
    getattr(harness, packed)(re.ctypes.data_as(P), im.ctypes.data_as(P))
    for b in range(32 // n):
        sr = x.real[b * n:(b + 1) * n].astype(np.float32)
        si = x.imag[b * n:(b + 1) * n].astype(np.float32)
        getattr(harness, scalar)(sr.ctypes.data_as(P), si.ctypes.data_as(P))
        np.testing.assert_array_equal(re[b * n:(b + 1) * n], sr)
        np.testing.assert_array_equal(im[b * n:(b + 1) * n], si)
