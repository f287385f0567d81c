"""ctypes wrapper around tests/remap_oracle.cpp: the oracle's convert() with the caller's palette dithered to (test
infrastructure, built with g++ into build/ like the other host harnesses of the tests)."""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "build", "libnq_remap_oracle.so")
SRC = os.path.join(ROOT, "tests", "remap_oracle.cpp")
DEPS = [SRC] + [os.path.join(ROOT, *p) for p in (("oracle", "nq_oracle.cpp"), ("nquant_android_b200", "csrc", "nq_math.h"),
                                                 ("nquant_android_b200", "csrc", "nq_math_tables.h"),
                                                 ("nquant_android_b200", "csrc", "nq_bluenoise_table.h"))]
_lib = None


def lib():
    global _lib
    if _lib is None:
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(d) for d in DEPS):
            fma = ["-mfma"] if " fma " in open("/proc/cpuinfo").read() else []   # as oracle/Makefile
            tmp = f"{SO}.{os.getpid()}"
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-w"] + fma +
                                  ["-o", tmp, SRC])
            os.replace(tmp, SO)   # test workers may build it side by side
        L = ctypes.CDLL(SO)
        vp, ci = ctypes.c_void_p, ctypes.c_int
        L.nqo_create.restype = vp
        L.nqo_destroy.argtypes = [vp]
        L.nqo_error.restype = ctypes.c_char_p
        L.nqo_error.argtypes = [vp]
        L.nqo_get_scalars.argtypes = [vp, vp]
        L.nqr_remap.argtypes = [vp, ci, vp, ci, ci, ci, ci, ctypes.c_uint64, vp, ci, vp]
        _lib = L
    return _lib


class Result:
    pass


def remap(kind, argb, width, height, n_max_colors, dither, palette, seed=0):
    """The oracle's convert(n_max_colors, dither) with `palette` (1..256 colours) dithered to in place of its own palette
    (or of the fixed one of n_max_colors <= 2). kind: 0 PnnQuantizer, 1 PnnLABQuantizer. Returns a Result with .out,
    .palette and .scalars (oracle/pyoracle.py's Scalars)."""
    from oracle import pyoracle
    L = lib()
    argb = np.ascontiguousarray(argb, dtype=np.uint32).reshape(-1)
    pal = np.ascontiguousarray(palette, dtype=np.uint32).reshape(-1)
    assert argb.size == width * height and 1 <= pal.size <= 256
    h = L.nqo_create()
    try:
        out = np.empty(argb.size, dtype=np.uint32)
        if L.nqr_remap(h, kind, argb.ctypes.data, width, height, n_max_colors, int(bool(dither)), seed, pal.ctypes.data, pal.size,
                       out.ctypes.data) != 0:
            raise RuntimeError(L.nqo_error(h).decode())
        r = Result()
        r.out, r.palette = out, pal.copy()
        s = pyoracle.Scalars()
        L.nqo_get_scalars(h, ctypes.byref(s))
        r.scalars = s.as_dict()
        return r
    finally:
        L.nqo_destroy(h)
