"""ctypes wrapper around oracle/libnq_oracle.so. TEST INFRASTRUCTURE ONLY: imported by tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs, never by the product."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libnq_oracle.so")


def build(force=False):
    srcs = [os.path.join(_HERE, "nq_oracle.cpp")] + [os.path.join(_HERE, "..", "nquant_android_b200", "csrc", f)
                                                      for f in ("nq_math.h", "nq_math_tables.h", "nq_bluenoise_table.h")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE] + (["-B"] if force else []) + ["libnq_oracle.so"],
                              stdout=subprocess.DEVNULL)
    return _SO


class Scalars(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in
                ["hasSemiTransparency", "transparentPixelIndex", "maxbins", "quan_rt", "texicab", "isNano",
                 "transparentColor", "margin", "thresold", "DITHER_MAX", "ditherMax", "sortedByYDiff", "hasAlpha"]] + \
               [("beta", ctypes.c_float), ("bn_weight", ctypes.c_float)] + \
               [(n, ctypes.c_double) for n in ["weight", "weight_final", "ratio_init", "ratio_merge", "PR", "PG", "PB", "PA", "gweight"]] + \
               [(n, ctypes.c_longlong) for n in ["rng_draws", "pixelMapSize", "n_merges", "n_saliencies", "n_gweights", "n_bins", "n_init",
                                                    "n_rescans", "n_heap_pops"]]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()  # no-op unless the .so is missing or older than its source
        L = ctypes.CDLL(_SO)
        vp, ci, cd, cf = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_float
        L.nqo_create.restype = vp
        L.nqo_destroy.argtypes = [vp]
        L.nqo_error.restype = ctypes.c_char_p
        L.nqo_error.argtypes = [vp]
        L.nqo_convert.argtypes = [vp, ci, vp, ci, ci, ci, ci, ctypes.c_uint64, ci, vp, vp, vp]
        L.nqo_get_scalars.argtypes = [vp, vp]
        for n in ["nqo_get_bins", "nqo_get_merges", "nqo_get_saliencies", "nqo_get_gweights"]:
            getattr(L, n).argtypes = [vp, vp]
        L.nqo_get_init_nn.argtypes = [vp, vp, vp]
        L.nqo_gilbert_order.argtypes = [ci, ci, vp]
        L.nqo_gilbert_params.argtypes = [ci, cd, ci, ci] + [vp] * 6
        L.nqo_init_weights.argtypes = [ci, ci, vp]
        L.nqo_rgb2lab.argtypes = [ctypes.c_uint32, ci, vp]
        L.nqo_lab2rgb.argtypes = [cf] * 4 + [ci]
        L.nqo_lab2rgb.restype = ctypes.c_uint32
        L.nqo_ciede_parts.argtypes = [vp, vp, ci, vp]
        L.nqo_ciede_parts_batch.argtypes = [vp, vp, ci, ci, vp]
        L.nqo_java_random_next_int.argtypes = [ctypes.c_uint64, ci, ci, vp]
        L.nqo_hashmap_order.argtypes = [vp, ci, vp]
        L.nqo_math.argtypes = [ci, cd, cd, ci]
        L.nqo_math.restype = cd
        L.nqo_y_diff.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ci]
        L.nqo_y_diff.restype = cd
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class Result:
    pass


def convert(kind, argb, width, height, n_max_colors, dither, seed=0, math_mode=0, trace=True):
    """Runs the oracle's convert(). kind: 0 PnnQuantizer, 1 PnnLABQuantizer. Returns a Result with
    .out (uint32 ARGB, what the reference hands to Bitmap.createBitmap), .palette, .scalars and,
    with trace=True, the stage dumps (.bins, .init_err, .init_nn, .merges, .saliencies, .gweights)."""
    L = lib()
    argb = np.ascontiguousarray(argb, dtype=np.uint32)
    assert argb.size == width * height
    h = L.nqo_create()
    try:
        out = np.empty(argb.size, dtype=np.uint32)
        pal = np.zeros(65536, dtype=np.uint32)
        plen = ctypes.c_int(0)
        rc = L.nqo_convert(h, kind, _p(argb), width, height, n_max_colors, int(bool(dither)), seed, math_mode,
                           _p(out), _p(pal), ctypes.byref(plen))
        if rc != 0:
            raise RuntimeError(L.nqo_error(h).decode())
        r = Result()
        r.out = out
        r.palette = pal[:plen.value].copy()
        s = Scalars()
        L.nqo_get_scalars(h, ctypes.byref(s))
        r.scalars = s.as_dict()
        if trace:
            r.merges = np.zeros((s.n_merges, 2), dtype=np.int32)
            if s.n_merges:
                L.nqo_get_merges(h, _p(r.merges))
            r.bins = np.zeros((s.n_bins, 5), dtype=np.float64)
            if s.n_bins:
                L.nqo_get_bins(h, _p(r.bins))
            r.init_err = np.zeros(s.n_init, dtype=np.float32)
            r.init_nn = np.zeros(s.n_init, dtype=np.int32)
            if s.n_init:
                L.nqo_get_init_nn(h, _p(r.init_err), _p(r.init_nn))
            r.saliencies = np.zeros(s.n_saliencies, dtype=np.float32)
            if s.n_saliencies:
                L.nqo_get_saliencies(h, _p(r.saliencies))
            r.gweights = np.zeros(s.n_gweights, dtype=np.float32)
            if s.n_gweights:
                L.nqo_get_gweights(h, _p(r.gweights))
        return r
    finally:
        L.nqo_destroy(h)


def gilbert_order(w, h):
    out = np.empty(w * h, dtype=np.uint32)
    lib().nqo_gilbert_order(w, h, _p(out))
    return out


def gilbert_params(palette_len, weight, has_saliencies, math_mode=0):
    vals = [ctypes.c_int() for _ in range(5)]
    beta = ctypes.c_float()
    lib().nqo_gilbert_params(palette_len, weight, int(has_saliencies), math_mode,
                             *[ctypes.byref(v) for v in vals], ctypes.byref(beta))
    names = ["margin", "thresold", "DITHER_MAX", "ditherMax", "sorted"]
    d = {n: v.value for n, v in zip(names, vals)}
    d["beta"] = beta.value
    return d


def init_weights(size, math_mode=0):
    out = np.zeros(size, dtype=np.float32)
    lib().nqo_init_weights(size, math_mode, _p(out))
    return out


def rgb2lab(c, math_mode=0):
    out = np.zeros(4, dtype=np.float32)
    lib().nqo_rgb2lab(int(c) & 0xFFFFFFFF, math_mode, _p(out))
    return out


def lab2rgb(alpha, L_, A, B, math_mode=0):
    return lib().nqo_lab2rgb(alpha, L_, A, B, math_mode)


def ciede_parts(lab1, lab2, math_mode=0):
    a = np.asarray(lab1, dtype=np.float32)
    b = np.asarray(lab2, dtype=np.float32)
    out = np.zeros(4, dtype=np.float32)
    lib().nqo_ciede_parts(_p(a), _p(b), math_mode, _p(out))
    return out


def ciede_parts_batch(lab1, lab2, math_mode=0):
    """lab1, lab2: (n, 3) float32 arrays of (L, A, B). Returns (n, 4) float32: L', C', H', R_T terms."""
    a = np.ascontiguousarray(lab1, dtype=np.float32).reshape(-1, 3)
    b = np.ascontiguousarray(lab2, dtype=np.float32).reshape(-1, 3)
    out = np.zeros((a.shape[0], 4), dtype=np.float32)
    lib().nqo_ciede_parts_batch(_p(a), _p(b), a.shape[0], math_mode, _p(out))
    return out


def java_random_next_int(seed, bound, n):
    out = np.zeros(n, dtype=np.int32)
    lib().nqo_java_random_next_int(seed, bound, n, _p(out))
    return out


def hashmap_order(keys):
    k = np.asarray(keys, dtype=np.int32)
    out = np.zeros(len(k), dtype=np.int32)
    n = lib().nqo_hashmap_order(_p(k), len(k), _p(out))
    return out[:n]


def math_fn(name, x, y=0.0, math_mode=0):
    idx = ["pow", "exp", "tanh", "cbrt", "atan2", "sin", "cos"].index(name)
    return lib().nqo_math(idx, x, y, math_mode)


def y_diff(c1, c2, math_mode=0):
    return lib().nqo_y_diff(int(c1) & 0xFFFFFFFF, int(c2) & 0xFFFFFFFF, math_mode)
