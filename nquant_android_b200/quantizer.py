"""Host-side mirror of the reference's public surface over the C ABI (include/nquant_b200.h).

Reference (nQuant.master/src/main/java/com/android/nQuant/):
  PnnQuantizer(String fname)                      PnnQuantizer.java:35
  PnnLABQuantizer(String fname)                   PnnLABQuantizer.java:24
  Bitmap convert(int nMaxColors, boolean dither)  PnnQuantizer.java:409
  boolean hasAlpha()                              PnnQuantizer.java:458
Differences, all forced by the boundary: the constructor takes an ARGB int[] (uint32 numpy array)
plus width/height in place of a file name / Bitmap, and convert returns the ARGB int[] the reference
hands to Bitmap.createBitmap (PnnQuantizer.java:455). The protected overridables (getQuanFn, pnnquan,
nearestColorIndex, closestColorIndex, dither) do not cross the ABI. No JVM exists in the build image,
so this Python mirror is the host side that is exercised; java/ holds the FFM binding as source.
"""
import ctypes
import threading

import numpy as np

from . import _lib

_tls = threading.local()


class NQuantError(Exception):
    """convert() `throws Exception` in the reference (PnnQuantizer.java:409)."""

    def __init__(self, code, message):
        super().__init__(f"[{code}] {message}")
        self.code = code


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class Context:
    """One nq_ctx: a (thread, GPU) pair. Not re-entrant, like the reference's quantizer objects."""

    def __init__(self, device=0):
        self._L = _lib.load()
        self._h = self._L.nq_create(int(device))
        if not self._h:
            raise NQuantError(_lib.NQ_ERR_CUDA, self._L.nq_last_error().decode())
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._L.nq_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise NQuantError(rc, self._L.nq_last_error().decode())

    # -- the hot path ----------------------------------------------------------------------------
    def convert_batch(self, kind, argb, width, height, n_max_colors, dither, seeds=None):
        """argb: (n, height*width) uint32 host array. Returns (out, palettes, palette_lens, has_alpha)."""
        argb = np.ascontiguousarray(argb, dtype=np.uint32).reshape(-1, width * height)
        n = argb.shape[0]
        out = np.empty_like(argb)
        pal = np.zeros((n, 256), dtype=np.uint32)
        plen = np.zeros(n, dtype=np.int32)
        ha = np.zeros(n, dtype=np.int32)
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        self._check(self._L.nq_convert_batch(self._h, kind, _p(argb), n, width, height, int(n_max_colors), int(bool(dither)),
                                             _p(sd), _p(out), _p(pal), _p(plen), _p(ha)))
        return out, pal, plen, ha

    def convert_batch_ptr(self, kind, in_ptr, out_ptr, n, width, height, n_max_colors, dither, seeds=None, device=False,
                          palettes=None, palette_lens=None):
        """Raw-pointer variant (pinned host or device memory owned by the caller, e.g. torch tensors)."""
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        fn = self._L.nq_convert_batch_device if device else self._L.nq_convert_batch
        self._check(fn(self._h, kind, ctypes.c_void_p(in_ptr), n, width, height, int(n_max_colors), int(bool(dither)),
                       _p(sd), ctypes.c_void_p(out_ptr), _p(palettes), _p(palette_lens), None))

    def convert_ragged(self, kind, images, n_max_colors, dither, seeds=None):
        """nq_convert_ragged: images of different sizes in one call. images: list of (height, width) uint32 host arrays.
        Returns (list of (height, width) outputs, palettes (n, 256), palette_lens, has_alpha)."""
        R = _Ragged(images)
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        self._check(self._L.nq_convert_ragged(self._h, kind, R.in_ptrs, _p(R.widths), _p(R.heights), R.n, int(n_max_colors),
                                              int(bool(dither)), _p(sd), R.out_ptrs, _p(R.pal), _p(R.plen), _p(R.ha)))
        return R.outs, R.pal, R.plen, R.ha

    def convert_ragged_ptr(self, kind, in_ptr, out_ptr, widths, heights, n_max_colors, dither, seeds=None, palettes=None,
                           palette_lens=None, has_alpha=None):
        """nq_convert_ragged_device: device buffers (e.g. torch tensors) holding the images packed back to back, image i
        widths[i] x heights[i] pixels. palettes / palette_lens / has_alpha: optional host arrays that receive the results."""
        w = np.ascontiguousarray(widths, dtype=np.int32)
        h = np.ascontiguousarray(heights, dtype=np.int32)
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        self._check(self._L.nq_convert_ragged_device(self._h, kind, ctypes.c_void_p(in_ptr), _p(w), _p(h), len(w), int(n_max_colors),
                                                     int(bool(dither)), _p(sd), ctypes.c_void_p(out_ptr), _p(palettes), _p(palette_lens),
                                                     _p(has_alpha)))

    def convert_indexed(self, kind, images, n_max_colors, dither, seeds=None, with_argb=False):
        """nq_convert_ragged_indexed: the palette index of every output pixel, computed on the GPU (the lowest index of the
        pixel's colour, include/nquant_b200.h). images: list of (height, width) uint32 host arrays. Returns (list of
        (height, width) uint8 index maps, list of ARGB outputs or None unless with_argb, palettes (n, 256), palette_lens,
        has_alpha)."""
        R = _Ragged(images, argb_out=with_argb)
        idx = [np.empty(im.shape, dtype=np.uint8) for im in R.ins]
        idx_ptrs = (ctypes.c_void_p * R.n)(*[a.ctypes.data for a in idx])
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        self._check(self._L.nq_convert_ragged_indexed(self._h, kind, R.in_ptrs, _p(R.widths), _p(R.heights), R.n, int(n_max_colors),
                                                      int(bool(dither)), _p(sd), idx_ptrs, R.out_ptrs, _p(R.pal), _p(R.plen), _p(R.ha)))
        return idx, R.outs, R.pal, R.plen, R.ha

    def convert_indexed_ptr(self, kind, in_ptr, index_ptr, widths, heights, n_max_colors, dither, seeds=None, out_ptr=None,
                            palettes=None, palette_lens=None, has_alpha=None):
        """nq_convert_ragged_indexed_device: device buffers (e.g. torch tensors), images packed back to back; the index map
        of image i starts at byte sum_{j<i} widths[j]*heights[j] of index_ptr. out_ptr (optional) receives the ARGB output.
        Every pointer 16-byte aligned. palettes / palette_lens / has_alpha: optional host arrays that receive the results."""
        w = np.ascontiguousarray(widths, dtype=np.int32)
        h = np.ascontiguousarray(heights, dtype=np.int32)
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        self._check(self._L.nq_convert_ragged_indexed_device(self._h, kind, ctypes.c_void_p(in_ptr), _p(w), _p(h), len(w), int(n_max_colors),
                                                             int(bool(dither)), _p(sd), ctypes.c_void_p(index_ptr),
                                                             ctypes.c_void_p(out_ptr) if out_ptr else None, _p(palettes), _p(palette_lens),
                                                             _p(has_alpha)))

    def remap(self, kind, images, palettes, dither, n_max_colors=None, seeds=None, with_argb=True, with_indices=False):
        """nq_remap_ragged: dither each image to a palette the caller already has, as convert() would with its palette
        replaced, without the merge loop (include/nquant_b200.h). images: list of (height, width) uint32 host arrays.
        palettes: one 1-D array of 1..256 colours shared by every image, or a list with one such array per image.
        n_max_colors (the nMaxColors convert() would get) defaults to the longest palette, and at least 2. Returns (list of
        ARGB outputs or None unless with_argb, list of uint8 index maps or None unless with_indices, has_alpha)."""
        if not (with_argb or with_indices):
            raise NQuantError(_lib.NQ_ERR_ARG, "with_argb and with_indices are both False")
        R = _Ragged(images, argb_out=with_argb)
        pal, plen, npal = _palettes(palettes, R.n)
        nmax = max(2, int(plen.max())) if n_max_colors is None else int(n_max_colors)
        idx, idx_ptrs = None, None
        if with_indices:
            idx = [np.empty(im.shape, dtype=np.uint8) for im in R.ins]
            idx_ptrs = (ctypes.c_void_p * R.n)(*[a.ctypes.data for a in idx])
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        self._check(self._L.nq_remap_ragged(self._h, kind, R.in_ptrs, _p(R.widths), _p(R.heights), R.n, nmax, _p(pal), _p(plen),
                                            npal, int(bool(dither)), _p(sd), R.out_ptrs, idx_ptrs, _p(R.ha)))
        return R.outs, idx, R.ha

    def remap_ptr(self, kind, in_ptr, widths, heights, palettes, dither, n_max_colors=None, seeds=None, out_ptr=None, index_ptr=None,
                  has_alpha=None):
        """nq_remap_ragged_device: device buffers (e.g. torch tensors) packed as in convert_indexed_ptr, every pointer 16-byte
        aligned; out_ptr and index_ptr are each optional, but not both. palettes and n_max_colors as in remap()."""
        w = np.ascontiguousarray(widths, dtype=np.int32)
        h = np.ascontiguousarray(heights, dtype=np.int32)
        pal, plen, npal = _palettes(palettes, len(w))
        nmax = max(2, int(plen.max())) if n_max_colors is None else int(n_max_colors)
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        self._check(self._L.nq_remap_ragged_device(self._h, kind, ctypes.c_void_p(in_ptr), _p(w), _p(h), len(w), nmax, _p(pal), _p(plen),
                                                   npal, int(bool(dither)), _p(sd), ctypes.c_void_p(out_ptr) if out_ptr else None,
                                                   ctypes.c_void_p(index_ptr) if index_ptr else None, _p(has_alpha)))

    def dither_with_palette(self, kind, argb, width, height, n_max_colors, dither, palette, seed=0):
        argb = np.ascontiguousarray(argb, dtype=np.uint32)
        palette = np.ascontiguousarray(palette, dtype=np.uint32)
        out = np.empty_like(argb)
        self._check(self._L.nq_dither_with_palette(self._h, kind, _p(argb), width, height, int(n_max_colors), int(bool(dither)),
                                                   int(seed), _p(palette), len(palette), _p(out)))
        return out

    def histogram(self, kind, argb, width, height, n_max_colors):
        """Stage hook nq_histogram: alpha scan + histogram + initial find_nn sweep of one image.
        Returns (bins (n, 5) float64, init_err float32, init_nn int32); image_info(0) holds the scalars."""
        argb = np.ascontiguousarray(argb, dtype=np.uint32)
        nb = ctypes.c_int(0)
        self._check(self._L.nq_histogram(self._h, kind, _p(argb), width, height, int(n_max_colors), ctypes.byref(nb), None, None, None, 0))
        bins = np.zeros((nb.value, 5), dtype=np.float64)
        err = np.zeros(nb.value, dtype=np.float32)
        nn = np.zeros(nb.value, dtype=np.int32)
        self._check(self._L.nq_histogram(self._h, kind, _p(argb), width, height, int(n_max_colors), ctypes.byref(nb), _p(bins), _p(err), _p(nn), nb.value))
        return bins, err, nn

    def set_stream(self, cuda_stream):
        """Order the context's work with a caller-owned stream, e.g. torch.cuda.current_stream().cuda_stream. Handle 0
        is CUDA's legacy default stream (torch's default stream), NOT the context's own: use reset_stream() for that."""
        self._check(self._L.nq_set_stream(self._h, ctypes.c_void_p(int(cuda_stream or 0))))

    def reset_stream(self):
        """Back to the context's private non-blocking stream (the state after creation)."""
        self._check(self._L.nq_reset_stream(self._h))

    def set_chunk_images(self, images):
        """Images per pipeline chunk of a batch call (0 = automatic)."""
        self._check(self._L.nq_set_chunk_images(self._h, int(images)))

    def set_spec_dither(self, on, segment=8192, warmup=1024):
        """Speculative segment-parallel error diffusion for the images that qualify (include/nquant_b200.h); results are
        bit-identical either way."""
        self._check(self._L.nq_set_spec_dither(self._h, int(bool(on)), int(segment), int(warmup)))

    def spec_stats(self):
        images, rounds, fallbacks = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        self._check(self._L.nq_get_spec_stats(self._h, ctypes.byref(images), ctypes.byref(rounds), ctypes.byref(fallbacks)))
        return {"images": images.value, "rounds": rounds.value, "fallbacks": fallbacks.value}

    # -- introspection ------------------------------------------------------------------------------
    def set_debug(self, flag):
        self._check(self._L.nq_set_debug(self._h, int(bool(flag))))

    def image_info(self, image=0):
        info = _lib.ImageInfo()
        self._check(self._L.nq_get_image_info(self._h, image, ctypes.byref(info)))
        return info.as_dict()

    def debug_bins(self, image=0):
        mb = self.image_info(image)["maxbins"]
        bins = np.zeros((mb, 5), dtype=np.float64)
        err = np.zeros(mb, dtype=np.float32)
        nn = np.zeros(mb, dtype=np.int32)
        self._check(self._L.nq_debug_get_bins(self._h, image, _p(bins), _p(err), _p(nn)))
        return bins, err, nn

    def debug_merges(self, image=0):
        m = self.image_info(image)["merges"]
        pairs = np.zeros((m, 2), dtype=np.int32)
        if m:
            self._check(self._L.nq_debug_get_merges(self._h, image, _p(pairs)))
        return pairs

    def debug_saliencies(self, npix, image=0):
        out = np.zeros(npix, dtype=np.float32)
        self._check(self._L.nq_debug_get_saliencies(self._h, image, _p(out)))
        return out

    def kernel_launches(self):
        return int(self._L.nq_kernel_launches(self._h))

    STAGES = ["alpha_scan", "histogram", "find_nn_sweep", "merge", "dither_setup", "dither"]

    def stage_times(self, reset=False):
        """{stage: (device ms, launches)} accumulated since the last reset (CUDA events on the stream)."""
        ms = np.zeros(6, dtype=np.float64)
        ln = np.zeros(6, dtype=np.uint64)
        self._check(self._L.nq_get_stage_times(self._h, _p(ms), _p(ln), int(bool(reset))))
        return {s: (float(ms[i]), int(ln[i])) for i, s in enumerate(self.STAGES)}

    KERNELS = ["k_spec_run", "k_dither_fifo", "k_dither_sorted", "k_merge"]

    def kernel_times(self, reset=False):
        """{kernel: (device ms, launches)} of the kernels that are timed on their own (CUDA events around each launch)."""
        ms = np.zeros(4, dtype=np.float64)
        ln = np.zeros(4, dtype=np.uint64)
        self._check(self._L.nq_get_kernel_times(self._h, _p(ms), _p(ln), int(bool(reset))))
        return {s: (float(ms[i]), int(ln[i])) for i, s in enumerate(self.KERNELS)}

    def math(self, fn, x, y=None):
        names = ["pow", "exp", "tanh", "cbrt", "atan2", "sin", "cos"]
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = None if y is None else np.ascontiguousarray(y, dtype=np.float64)
        out = np.empty_like(x)
        self._check(self._L.nq_debug_math(self._h, names.index(fn), _p(x), _p(y), _p(out), x.size))
        return out

    def ciede(self, lab1, lab2):
        """(n, 3) float32 (L, A, B) pairs -> ((n, 4) float32 L', C', H', R_T terms, pairs that took the exact path)."""
        a = np.ascontiguousarray(lab1, dtype=np.float32).reshape(-1, 3)
        b = np.ascontiguousarray(lab2, dtype=np.float32).reshape(-1, 3)
        out = np.zeros((a.shape[0], 4), dtype=np.float32)
        cnt = ctypes.c_int(0)
        self._check(self._L.nq_debug_ciede(self._h, _p(a), _p(b), _p(out), ctypes.byref(cnt), a.shape[0]))
        return out, cnt.value

    def synth_device(self, out_ptr, n, width, height, cls, alpha_mode, seed0):
        self._check(self._L.nq_synth_device(self._h, ctypes.c_void_p(out_ptr), n, width, height, cls, alpha_mode, seed0))


def convert_batch_multi(contexts, kind, argb, width, height, n_max_colors, dither, seeds=None, queue_images=0):
    """nq_convert_batch_multi: one batch over several contexts (one per GPU of the node, normally), pieces of
    `queue_images` images handed out dynamically (0 = one piece per context). Returns (out, palettes, palette_lens, has_alpha)."""
    L = _lib.load()
    argb = np.ascontiguousarray(argb, dtype=np.uint32).reshape(-1, width * height)
    n = argb.shape[0]
    out = np.empty_like(argb)
    pal = np.zeros((n, 256), dtype=np.uint32)
    plen = np.zeros(n, dtype=np.int32)
    ha = np.zeros(n, dtype=np.int32)
    sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
    handles = (ctypes.c_void_p * len(contexts))(*[c._h for c in contexts])
    rc = L.nq_convert_batch_multi(handles, len(contexts), kind, _p(argb), n, width, height, int(n_max_colors), int(bool(dither)),
                                  _p(sd), _p(out), _p(pal), _p(plen), _p(ha), int(queue_images))
    if rc != 0:
        raise NQuantError(rc, L.nq_last_error().decode())
    return out, pal, plen, ha


def _palettes(palettes, n):
    """One shared palette (a 1-D array) or one per image (a list of n of them) -> the (n_palettes, 256) uint32 array, the
    lengths and n_palettes of the remap calls."""
    shared = isinstance(palettes, np.ndarray) and palettes.ndim == 1
    pals = [palettes] if shared else list(palettes)
    if not shared and len(pals) != n:
        raise NQuantError(_lib.NQ_ERR_ARG, "palettes: one array shared by every image, or one per image")
    out = np.zeros((len(pals), 256), dtype=np.uint32)
    lens = np.zeros(len(pals), dtype=np.int32)
    for i, p in enumerate(pals):
        p = np.asarray(p, dtype=np.uint32).reshape(-1)
        if not 1 <= p.size <= 256:
            raise NQuantError(_lib.NQ_ERR_ARG, f"palette {i}: length must be 1..256")
        out[i, :p.size] = p
        lens[i] = p.size
    return out, lens, len(pals)


class _Ragged:
    """Host arguments of the ragged entry points: sides, per-image pointer arrays, result arrays."""

    def __init__(self, images, argb_out=True):
        self.ins = [np.ascontiguousarray(im, dtype=np.uint32) for im in images]
        if any(im.ndim != 2 for im in self.ins):
            raise NQuantError(_lib.NQ_ERR_ARG, "every image must be a (height, width) array")
        self.n = len(self.ins)
        self.heights = np.array([im.shape[0] for im in self.ins], dtype=np.int32)
        self.widths = np.array([im.shape[1] for im in self.ins], dtype=np.int32)
        self.in_ptrs = (ctypes.c_void_p * self.n)(*[im.ctypes.data for im in self.ins])
        self.outs, self.out_ptrs = None, None
        if argb_out:
            self.outs = [np.empty_like(im) for im in self.ins]
            self.out_ptrs = (ctypes.c_void_p * self.n)(*[o.ctypes.data for o in self.outs])
        self.pal = np.zeros((self.n, 256), dtype=np.uint32)
        self.plen = np.zeros(self.n, dtype=np.int32)
        self.ha = np.zeros(self.n, dtype=np.int32)


def convert_ragged_multi(contexts, kind, images, n_max_colors, dither, seeds=None, queue_images=0):
    """nq_convert_ragged_multi: images of different sizes over several contexts, pieces of `queue_images` images handed out
    dynamically (0 = one piece per context). Returns (list of outputs, palettes, palette_lens, has_alpha)."""
    L = _lib.load()
    R = _Ragged(images)
    sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
    handles = (ctypes.c_void_p * len(contexts))(*[c._h for c in contexts])
    rc = L.nq_convert_ragged_multi(handles, len(contexts), kind, R.in_ptrs, _p(R.widths), _p(R.heights), R.n, int(n_max_colors),
                                   int(bool(dither)), _p(sd), R.out_ptrs, _p(R.pal), _p(R.plen), _p(R.ha), int(queue_images))
    if rc != 0:
        raise NQuantError(rc, L.nq_last_error().decode())
    return R.outs, R.pal, R.plen, R.ha


def default_context(device=0):
    """Per-thread, per-device context cache (one nq_ctx per (thread, GPU))."""
    cache = getattr(_tls, "ctx", None)
    if cache is None:
        cache = _tls.ctx = {}
    if device not in cache:
        cache[device] = Context(device)
    return cache[device]


def gilbert_order(width, height):
    out = np.empty(width * height, dtype=np.uint32)
    L = _lib.load()
    if L.nq_gilbert_order(width, height, _p(out)) != 0:
        raise NQuantError(_lib.NQ_ERR_ARG, L.nq_last_error().decode())
    return out


class PnnQuantizer:
    """com.android.nQuant.PnnQuantizer (PnnQuantizer.java:16)."""
    KIND = _lib.NQ_KIND_PNN

    def __init__(self, argb, width, height, device=0, rng_seed=0):
        argb = np.ascontiguousarray(argb, dtype=np.uint32).reshape(-1)
        if argb.size != width * height:
            raise NQuantError(_lib.NQ_ERR_ARG, "argb must hold width*height pixels")
        self.pixels = argb.copy()          # the reference keeps a private copy (PnnQuantizer.java:42-43)
        self.width, self.height = width, height
        self.device = device
        self.rng_seed = rng_seed
        self.palette = None
        self._has_alpha = False

    def convert(self, nMaxColors, dither):
        """Bitmap convert(int nMaxColors, boolean dither) -> ARGB uint32 array (PnnQuantizer.java:409)."""
        ctx = default_context(self.device)
        out, pal, plen, ha = ctx.convert_batch(self.KIND, self.pixels[None, :], self.width, self.height, nMaxColors, dither,
                                               seeds=[self.rng_seed])
        self.palette = pal[0, :plen[0]].copy()
        self._has_alpha = bool(ha[0])
        self.info = ctx.image_info(0)
        return out[0]

    def convert_indexed(self, nMaxColors, dither):
        """convert() as palette indices: one uint8 per pixel, palette[index] is the colour convert() returns (the lowest
        index of that colour). Sets palette, hasAlpha() and info like convert()."""
        ctx = default_context(self.device)
        idx, _, pal, plen, ha = ctx.convert_indexed(self.KIND, [self.pixels.reshape(self.height, self.width)], nMaxColors, dither,
                                                    seeds=[self.rng_seed])
        self.palette = pal[0, :plen[0]].copy()
        self._has_alpha = bool(ha[0])
        self.info = ctx.image_info(0)
        return idx[0].reshape(-1)

    def hasAlpha(self):
        """boolean hasAlpha() (PnnQuantizer.java:458)."""
        return self._has_alpha


class PnnLABQuantizer(PnnQuantizer):
    """com.android.nQuant.PnnLABQuantizer (PnnLABQuantizer.java:17)."""
    KIND = _lib.NQ_KIND_PNNLAB
