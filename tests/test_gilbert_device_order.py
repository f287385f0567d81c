"""csrc/nq_gilbert.h computes the Gilbert visiting order position by position (one GPU thread per position in
k_gilbert_order). Compiled here with g++ (NQ_HD is plain `inline` without nvcc), it must give the oracle's walk of
GilbertCurve.generate2d for every size, and the library's host entry nq_gilbert_order, built on the same function,
must too. No GPU involved."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "nquant_android_b200", "csrc", "nq_gilbert.h")

HARNESS = r"""
#include <stdint.h>
#include "nq_gilbert.h"
extern "C" void gilbert_bidx(int w, int h, uint32_t* out) {   // x + y*w, the layout of the oracle's walk
  const unsigned long long npix = (unsigned long long)w * (unsigned long long)h;
  for (unsigned long long n = 0; n < npix; ++n) {
    int x, y;
    nq::gilbert_xy(w, h, n, &x, &y);
    out[n] = (uint32_t)x + (uint32_t)y * (uint32_t)w;
  }
}
"""

LARGE = [(1, 65535), (65535, 1), (2, 4097), (4097, 3), (65535, 2), (495, 438), (1920, 1080), (1080, 1920), (3840, 2160)]


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("gilbert")
    src, so = d / "gilbert_harness.cpp", d / "libgilbert_harness.so"
    src.write_text(HARNESS)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", os.path.dirname(HEADER), "-o", str(so), str(src)])
    L = ctypes.CDLL(str(so))
    L.gilbert_bidx.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    L.gilbert_bidx.restype = None
    return L


def positional(L, w, h):
    out = np.empty(w * h, dtype=np.uint32)
    L.gilbert_bidx(w, h, out.ctypes.data)
    return out


def test_every_small_size_matches_the_oracle_walk(harness, oracle):
    for w in range(1, 49):
        for h in range(1, 49):
            assert np.array_equal(positional(harness, w, h), oracle.gilbert_order(w, h)), (w, h)


@pytest.mark.parametrize("w,h", LARGE, ids=[f"{w}x{h}" for w, h in LARGE])
def test_large_and_degenerate_sizes_match_the_oracle_walk(harness, oracle, w, h):
    assert np.array_equal(positional(harness, w, h), oracle.gilbert_order(w, h))


@pytest.mark.parametrize("w,h", [(5, 3), (48, 47), (495, 438), (1920, 1080), (1080, 1920), (65535, 2)])
def test_library_host_order_matches_the_oracle_walk(oracle, w, h):
    from nquant_android_b200 import _build
    from nquant_android_b200.quantizer import gilbert_order
    _build.build()
    assert np.array_equal(gilbert_order(w, h), oracle.gilbert_order(w, h))
