"""CPU unit test of the register-resident DFTs of the mel kernel (csrc/mel_fft.cuh): the header is compiled as HOST code
into a scratch harness (tests/host/mel_fft_host.cu) and checked against numpy's FFT, including the lane-by-lane
emulation of the warp's 32 x 25 decomposition and the two-real-frames separation.  No GPU involved."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests._util import ROOT


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("host") / "libzeggs_mel_fft_host.so")
    src = os.path.join(ROOT, "tests", "host", "mel_fft_host.cu")
    r = subprocess.run(["/usr/local/cuda/bin/nvcc", "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-shared",
                        "-o", out, src], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("nvcc host harness build failed: " + r.stderr[-400:])
    return C.CDLL(out)


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("n,fn", [(25, "dft25_host"), (32, "dft32_host")])
def test_small_dfts_match_numpy(harness, n, fn):
    rs = np.random.RandomState(n)
    x = (rs.randn(n) + 1j * rs.randn(n)).astype(np.complex64)
    out = np.zeros(n, np.complex64)
    getattr(harness, fn)(P(x.view(np.float32)), P(out.view(np.float32)))
    ref = np.fft.fft(x.astype(np.complex128))
    assert np.abs(out - ref).max() <= 2e-5 * np.abs(ref).max()


def test_two_real_frames_through_one_800_point_fft(harness):
    rs = np.random.RandomState(7)
    fa, fb = rs.randn(800).astype(np.float32), (0.3 * rs.randn(800)).astype(np.float32)
    aa, ab = np.zeros(401, np.float32), np.zeros(401, np.float32)
    harness.two_frames_host(P(fa), P(fb), P(aa), P(ab))
    ra, rb = np.abs(np.fft.rfft(fa.astype(np.float64))), np.abs(np.fft.rfft(fb.astype(np.float64)))
    assert np.abs(aa - ra).max() <= 2e-5 * ra.max()
    assert np.abs(ab - rb).max() <= 2e-5 * ra.max()
