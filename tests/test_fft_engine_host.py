"""CPU check of csrc/fft_engine.cuh + csrc/fft_plan.hpp: the stage code is __host__ __device__, so the very same
index math, butterflies, digit-reversal tables and Bluestein driver that run in shared memory on the GPU are run
here by one host "thread" (tests/native/fft_host_test.cu) and compared with numpy.fft for every 1-D length the
pyramid's level-size rule produces at the benchmark resolutions (256^2, 1080p, 2048^2, 4K) plus every radix."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fusion-method-for-video-frame-interpolation_b200", "csrc")
SRC = os.path.join(ROOT, "tests", "native", "fft_host_test.cu")
SO = os.path.join(ROOT, "tests", "native", "fft_host_test.so")


@pytest.fixture(scope="module")
def lib():
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc not available")
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("fft_engine.cuh", "fft_plan.hpp", "fft_consts.cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["nvcc", "-O1", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-Wno-deprecated-gpu-targets",
                               "-I", CSRC, "-o", SO, SRC])
    L = ctypes.CDLL(SO)
    L.fft_host_run.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
    return L


def level_lengths(n, levels):
    out = []
    for _ in range(levels):
        out.append(n)
        n = int(np.ceil((n - 0.5) / np.sqrt(2) - 1e-9))
    return out


def run(L, n, mode, batch, rng, rader=True):
    x = (rng.standard_normal((batch, n)) + 1j * rng.standard_normal((batch, n))).astype(np.complex64)
    out = np.zeros((batch, n), np.complex64)
    info = np.zeros(16, np.int32)
    rc = L.fft_host_run(n, mode, batch, x.ctypes.data, out.ctypes.data, info.ctypes.data, int(rader))
    assert rc != -2, "n=%d mode=%d: the transform wrote outside its buffers (guard zone overwritten)" % (n, mode)
    assert rc == 0, "no plan for n=%d" % n
    ref = np.fft.fft(x.astype(np.complex128), axis=1)
    err = np.abs(out - ref).max() / np.abs(ref).max()
    return err, info


LENGTHS = sorted(set(
    list(range(2, 41)) + [45, 47, 49, 59, 64, 77, 81, 91, 94, 96, 100, 121, 128, 169, 171, 181, 191, 241, 256, 289, 361, 529, 1334]
    + level_lengths(256, 11) + level_lengths(1080, 16) + level_lengths(1920, 16) + level_lengths(2048, 17)
    + level_lengths(2160, 18) + level_lengths(3840, 18)))


@pytest.mark.parametrize("rader", [True, False], ids=["2", "0"])      # ids: 2 = the shipped plans, 0 = Bluestein only
@pytest.mark.parametrize("mode", [0, 1])
def test_all_lengths(lib, mode, rader):
    """rader = True: the shipped plans (Rader for n = r * p with p - 1 smooth; Bluestein for the rest); rader = False: Bluestein for
    every non-smooth length -- the Bluestein code runs on many more lengths."""
    rng = np.random.default_rng(mode)
    worst, kinds = 0.0, {0: 0, 1: 0, 2: 0}
    for n in LENGTHS:
        batch = 2 if n > 512 else 4
        err, info = run(lib, n, mode, batch, rng, rader)
        kinds[int(info[1])] += 1
        tol = 4e-6 if info[1] else 2e-6      # Bluestein: two FFTs of ~2n + chirps; Rader: two FFTs of p - 1 + the outer stages
        assert err < tol, "n=%d mode=%d rel err %.3g (M=%d kind=%d radices=%s)" % (
            n, mode, err, info[0], info[1], list(info[3:3 + info[2]]))
        worst = max(worst, err)
    print("worst relative error", worst, "plans direct/bluestein/rader:", kinds)
    assert (kinds[2] > 10) == rader


def test_plan_choices(lib):
    rng = np.random.default_rng(5)
    for n, stages in ((1080, 3), (1920, 3), (960, 3), (540, 3), (135, 2)):
        _, info = run(lib, n, 1, 1, rng)
        assert info[1] == 0 and info[2] == stages, (n, info[:8])
    for n in (764, 1358, 191, 241, 382, 679, 97, 61, 43, 31, 23):      # one large prime factor p with p - 1 smooth: Rader, no padding
        for mode in (0, 1):
            _, info = run(lib, n, mode, 1, rng)
            assert info[1] == 2 and info[0] == n, (n, info[:8])
    for n in (47, 59, 94, 529, 2 * 23 * 29):                           # p - 1 not smooth / two large primes / p^2: Bluestein
        _, info = run(lib, n, 0, 1, rng)
        assert info[1] == 1 and info[0] >= 2 * n - 1, (n, info[:8])
