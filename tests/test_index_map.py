"""The index map's table (csrc/nq_index.h, built in shared memory by k_index_map) compiled with g++: built from a palette in
any insertion order, its lookup gives imageio.to_indices's index for every palette colour -- the lowest index of duplicate
colours -- and reports a colour the palette does not hold. And imageio.write_png8 writes what write_indexed_png writes. No GPU
involved."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from nquant_android_b200 import imageio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "nquant_android_b200", "csrc")

HARNESS = r"""
#include <stdint.h>
#include "nq_index.h"
// the table of pal[0..plen) with its entries inserted in the order `order` (as the device's threads may), then every pixel
// looked up; returns the number of pixels the palette does not hold (their index is -1)
extern "C" int index_map(const uint32_t* pal, int plen, const int* order, const uint32_t* px, long long n, int* out) {
  unsigned long long tab[NQ_IMAP_SLOTS];
  for (int k = 0; k < NQ_IMAP_SLOTS; ++k) tab[k] = NQ_IMAP_EMPTY;
  for (int k = 0; k < plen; ++k) nq::imap_insert(tab, pal, order[k]);
  int misses = 0;
  for (long long p = 0; p < n; ++p) { out[p] = nq::imap_lookup(tab, px[p]); misses += out[p] < 0; }
  return misses;
}
"""


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("index_map")
    src, so = d / "index_harness.cpp", d / "libindex_harness.so"
    src.write_text(HARNESS)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, "-o", str(so), str(src)])
    L = ctypes.CDLL(str(so))
    L.index_map.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
    L.index_map.restype = ctypes.c_int
    return L


def run(L, pal, px, order):
    pal = np.ascontiguousarray(pal, np.uint32)
    px = np.ascontiguousarray(px, np.uint32)
    order = np.ascontiguousarray(order, np.int32)
    out = np.empty(px.size, np.int32)
    misses = L.index_map(pal.ctypes.data, pal.size, order.ctypes.data, px.ctypes.data, px.size, out.ctypes.data)
    return out, misses


def palette(rng, n):
    """n colours with duplicates, colours that differ in alpha only, and the extremes 0 and 0xFFFFFFFF."""
    pal = rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32)
    if n >= 2:
        pal[-1] = pal[0]                                       # a duplicate: index 0 must win
    if n >= 17:
        pal[5] = (pal[3] & 0x00FFFFFF) | 0x80000000            # same RGB as entry 3, other alpha
        pal[6] = pal[3] & 0x00FFFFFF                           # ... and alpha 0
        pal[7], pal[8] = 0, 0xFFFFFFFF
        pal[9] = pal[4]                                        # another duplicate
        pal[-2] = pal[7]
    if n == 256:
        pal[100:140] = pal[60:100]                             # a run of duplicates
        pal[200:232] = rng.integers(0, 2**32, 8, dtype=np.uint64).astype(np.uint32).repeat(4)
    return pal


@pytest.mark.parametrize("n", [1, 2, 17, 256])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_lookup_matches_to_indices(harness, n, seed):
    rng = np.random.default_rng(1000 * n + seed)
    pal = palette(rng, n)
    px = np.concatenate([pal, pal[rng.integers(0, n, 50000)]])  # every palette colour, then a quantized-looking image
    want = imageio.to_indices(px, pal)
    assert np.array_equal(pal[want], px)
    for order in (np.arange(n), np.arange(n)[::-1], rng.permutation(n)):
        got, misses = run(harness, pal, px, order)
        assert misses == 0
        assert np.array_equal(got, want.astype(np.int32)), order[:8]


@pytest.mark.parametrize("n", [1, 2, 17, 256])
def test_a_colour_outside_the_palette_is_reported(harness, n):
    rng = np.random.default_rng(7 + n)
    pal = palette(rng, n)
    foreign = [c for c in (0x00000000, 0xFFFFFFFF, 0xFF000000, 0x12345678, int(pal[0]) ^ 0x01000000, int(pal[0]) ^ 1)
               if c not in set(pal.tolist())]
    px = np.concatenate([pal, np.array(foreign, np.uint32), pal])
    got, misses = run(harness, pal, px, rng.permutation(n))
    assert misses == len(foreign)
    assert (got[n:n + len(foreign)] == -1).all()
    assert np.array_equal(got[:n], imageio.to_indices(pal, pal).astype(np.int32))
    with pytest.raises(ValueError):
        imageio.to_indices(px, pal)


def test_a_full_table_of_colliding_colours(harness):
    """256 colours that all hash to one slot (the probe runs the whole chain and wraps around the end of the table)."""
    import itertools
    h = lambda c: ((c * 0x9E3779B1) & 0xFFFFFFFF) >> 22
    pal = np.array(list(itertools.islice((c for c in range(0, 2**31, 7) if h(c) == 1023), 256)), np.uint32)
    assert pal.size == 256
    px = np.concatenate([pal, pal[::-1]])
    got, misses = run(harness, pal, px, np.arange(256)[::-1])
    assert misses == 0 and np.array_equal(got, imageio.to_indices(px, pal).astype(np.int32))
    _, misses = run(harness, pal, np.array([pal.max() + 7], np.uint32), np.arange(256))
    assert misses == 1


@pytest.mark.parametrize("alpha", ["opaque", "semi"])
def test_write_png8_writes_what_write_indexed_png_writes(tmp_path, alpha):
    from nquant_android_b200.synth import make_image
    w, h = 37, 23
    rng = np.random.default_rng(3)
    pal = (rng.integers(0, 2**24, 40, dtype=np.uint64).astype(np.uint32) | np.uint32(0xFF000000))
    if alpha == "semi":
        pal[::3] &= np.uint32(0x7FFFFFFF)
    idx = (make_image(w, h, "noisy", "opaque", seed=5) % 40).astype(np.uint8)
    a, b = tmp_path / "a.png", tmp_path / "b.png"
    na = imageio.write_indexed_png(str(a), pal[idx], pal, w, h)
    nb = imageio.write_png8(str(b), idx, pal, w, h)
    assert na == nb and a.read_bytes() == b.read_bytes()
    with pytest.raises(ValueError):
        imageio.write_png8(str(b), np.full(w * h, 40, np.uint8), pal, w, h)
