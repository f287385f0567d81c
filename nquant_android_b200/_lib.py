"""ctypes binding of include/nquant_b200.h. There is no fallback: if the CUDA library is missing or
cannot be loaded, importing callers get an ImportError."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libnquant_b200.so")

# every symbol include/nquant_b200.h declares
SYMBOLS = [
    "nq_device_count", "nq_create", "nq_destroy", "nq_last_error", "nq_convert", "nq_convert_batch",
    "nq_convert_batch_device", "nq_dither_with_palette", "nq_gilbert_order", "nq_get_image_info", "nq_set_debug",
    "nq_debug_get_bins", "nq_debug_get_merges", "nq_debug_get_saliencies", "nq_kernel_launches", "nq_debug_math",
    "nq_synth_device", "nq_get_stage_times", "nq_set_stream", "nq_debug_ciede", "nq_sizeof_image_info",
    "nq_set_spec_dither", "nq_get_spec_stats", "nq_reset_stream", "nq_set_chunk_images", "nq_get_kernel_times", "nq_convert_batch_multi", "nq_histogram",
]

NQ_KIND_PNN, NQ_KIND_PNNLAB = 0, 1
NQ_OK, NQ_ERR_CUDA, NQ_ERR_ARG, NQ_ERR_COLOR, NQ_ERR_UNSUPPORTED, NQ_ERR_NOMEM = 0, -1, -2, -3, -4, -5


class ImageInfo(ctypes.Structure):
    _fields_ = [
        ("has_semi_transparency", ctypes.c_int), ("transparent_pixel_index", ctypes.c_int),
        ("transparent_color", ctypes.c_uint32),
        ("maxbins", ctypes.c_int), ("quan_rt", ctypes.c_int), ("texicab", ctypes.c_int), ("is_nano", ctypes.c_int),
        ("weight", ctypes.c_double), ("ratio_init", ctypes.c_double), ("ratio_merge", ctypes.c_double),
        ("pr", ctypes.c_double), ("pg", ctypes.c_double), ("pb", ctypes.c_double), ("pa", ctypes.c_double),
        ("g_margin", ctypes.c_int), ("g_thresold", ctypes.c_int), ("g_dither_max_q", ctypes.c_int),
        ("g_dither_max", ctypes.c_int), ("g_sorted", ctypes.c_int), ("g_has_alpha", ctypes.c_int),
        ("g_use_saliency", ctypes.c_int),
        ("g_beta", ctypes.c_float), ("bn_weight", ctypes.c_float), ("palette_len", ctypes.c_int),
        ("merges", ctypes.c_ulonglong), ("rescans", ctypes.c_ulonglong), ("pair_tests", ctypes.c_ulonglong),
        ("rng_draws", ctypes.c_ulonglong), ("heap_pops", ctypes.c_ulonglong),
        ("error", ctypes.c_int),
        ("full_evals", ctypes.c_ulonglong),
        ("merge_cycles", ctypes.c_ulonglong * 6), ("live_blocks", ctypes.c_ulonglong), ("screened", ctypes.c_ulonglong),
        ("dither_cycles", ctypes.c_ulonglong * 3),
        ("merge_rounds", ctypes.c_ulonglong), ("rescans_discarded", ctypes.c_ulonglong),
        ("merge_ctas_per_sm", ctypes.c_int),
    ]

    def as_dict(self):
        return {n: (list(getattr(self, n)) if n in ("merge_cycles", "dither_cycles") else getattr(self, n)) for n, _ in self._fields_}


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        raise ImportError(f"{SO} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). This package has no CPU fallback.")
    L = ctypes.CDLL(SO)
    vp, ci, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64
    L.nq_device_count.restype = ci
    L.nq_create.restype = vp
    L.nq_create.argtypes = [ci]
    L.nq_destroy.argtypes = [vp]
    L.nq_destroy.restype = None
    L.nq_last_error.restype = ctypes.c_char_p
    L.nq_convert.argtypes = [vp, ci, vp, ci, ci, ci, ci, u64, vp, vp, vp, vp]
    L.nq_convert_batch.argtypes = [vp, ci, vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp]
    L.nq_convert_batch_device.argtypes = [vp, ci, vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp]
    L.nq_convert_batch_multi.argtypes = [vp, ci, ci, vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp, ci]
    L.nq_dither_with_palette.argtypes = [vp, ci, vp, ci, ci, ci, ci, u64, vp, ci, vp]
    L.nq_gilbert_order.argtypes = [ci, ci, vp]
    L.nq_histogram.argtypes = [vp, ci, vp, ci, ci, ci, vp, vp, vp, vp, ci]
    L.nq_get_image_info.argtypes = [vp, ci, vp]
    L.nq_set_debug.argtypes = [vp, ci]
    L.nq_debug_get_bins.argtypes = [vp, ci, vp, vp, vp]
    L.nq_debug_get_merges.argtypes = [vp, ci, vp]
    L.nq_debug_get_saliencies.argtypes = [vp, ci, vp]
    L.nq_kernel_launches.argtypes = [vp]
    L.nq_kernel_launches.restype = ctypes.c_ulonglong
    L.nq_debug_math.argtypes = [vp, ci, vp, vp, vp, ci]
    L.nq_set_stream.argtypes = [vp, vp]
    L.nq_reset_stream.argtypes = [vp]
    L.nq_set_chunk_images.argtypes = [vp, ci]
    L.nq_get_kernel_times.argtypes = [vp, vp, vp, ci]
    L.nq_debug_ciede.argtypes = [vp, vp, vp, vp, vp, ci]
    L.nq_get_stage_times.argtypes = [vp, vp, vp, ci]
    L.nq_synth_device.argtypes = [vp, vp, ci, ci, ci, ci, ci, u64]
    L.nq_set_spec_dither.argtypes = [vp, ci, ci, ci]
    L.nq_get_spec_stats.argtypes = [vp, vp, vp, vp]
    for s in SYMBOLS:
        getattr(L, s)
    if L.nq_sizeof_image_info() != ctypes.sizeof(ImageInfo):
        raise ImportError("nq_image_info: the ctypes mirror in _lib.py does not match include/nquant_b200.h")
    _lib = L
    return L
