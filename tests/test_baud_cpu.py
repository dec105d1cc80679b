"""CPU tier of baud-rate estimation: the numpy restatement the GPU tests compare against (tests/baud_ref.py), and the C++
facade members compiled and linked against the library."""
import os
import subprocess

import numpy as np
import pytest

import baud_ref
from habdec_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("m", [1, 2, 3, 32, 65])
def test_run_walk_equals_the_sample_by_sample_statement(m):
    rng = np.random.default_rng(m)
    for trial in range(20):
        n = int(rng.integers(1, 3000))
        # sign runs of random lengths around m, with exact zeros (they count as negative)
        lengths = rng.integers(1, 2 * m + 3, size=n)
        signs = np.resize([1.0, -1.0], n) * rng.choice([1.0, 0.0], size=n, p=[0.9, 0.1])
        d = np.repeat(signs, lengths).astype(np.float32)
        assert np.array_equal(baud_ref.edges(d, m), baud_ref.edges_literal(d, m))


def test_geometry_matches_the_stated_sizes():
    assert baud_ref.geometry(8000.0) == (1040, 3)           # 4 KB of histogram per channel
    assert baud_ref.geometry(78125.0) == (10157, 32)        # 40 KB
    assert baud_ref.geometry(1000.0) == (130, 1)


@pytest.mark.parametrize("fs", [8000.0, 78125.0])
@pytest.mark.parametrize("baud", [50.0, 75.0, 100.0, 150.0, 200.0, 300.0, 600.0, 297.0])
def test_clean_keying_gives_the_rate(fs, baud):
    """Noise-free keying, sampled at fs_dec: the estimator picks the candidate and fits the clock."""
    text = "".join(synth.make_sentence(3, k) for k in range(3)).encode()
    bits = synth.uart_bits(text, 8, 2, 4, 4)
    n = int(len(bits) * fs / baud)
    i = np.minimum((np.arange(n) * (baud / fs)).astype(np.int64), len(bits) - 1)
    d = np.where(bits[i] > 0, 1.0, -1.0).astype(np.float32)
    e = baud_ref.estimate(d, fs)
    assert e["nominal"] == (300.0 if baud == 297.0 else baud)
    assert e["confidence"] == 1.0 and e["runs"] > 100
    assert abs(e["baud"] - baud) / baud < 2e-3


def test_noise_and_silence():
    rng = np.random.default_rng(1)
    e = baud_ref.estimate(rng.standard_normal(80000).astype(np.float32), 8000.0)
    assert e["runs"] > 1000 and e["confidence"] < 0.5
    assert baud_ref.estimate(np.zeros(80000, np.float32), 8000.0) == {"baud": 0.0, "nominal": 0.0, "confidence": 0.0, "runs": 0,
                                                                      "long_runs": 0}


def test_cpp_facade_baud_members_build_and_link(tmp_path):
    """setBaudEstimation / getBaudEstimates / applyBaudEstimates compile as C++17 against the C ABI library.  Without a
    CUDA device the program fails loudly; with one, tests/test_gpu_baud.py runs it."""
    lib_dir = os.path.join(ROOT, "habdec_b200")
    exe = str(tmp_path / "baud_facade")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "baud_facade.cpp"),
                    "-L", lib_dir, "-lhabdec_b200", "-Wl,-rpath," + lib_dir, "-lpthread", "-o", exe], check=True)
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present: the run itself is covered by tests/test_gpu_baud.py")
    except ImportError:
        pass
    path = str(tmp_path / "z.cf32")
    np.zeros(2 * 65536, dtype=np.complex64).tofile(path)
    r = subprocess.run([exe, path, "2", "65536", "2048000"], capture_output=True)
    assert r.returncode != 0
    assert b"no usable CUDA device" in r.stderr and b"EST" not in r.stdout
