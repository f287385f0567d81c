"""The dither across its parameter space. Its behaviour is a decision tree over the Gilbert weight
(weight = min(.9, nMaxColors / maxbins)), the palette length and the alpha situation, restated on the GPU in k_dither_setup,
in ditherPixel (nq_dither.cuh twice, nq_dither_spec.cuh once) and in the CIELAB quan_rt of nq_hist.cuh. The tests here put
images exactly on those decisions instead of meeting them by accident:

- a case table whose images have an exact number of histogram keys n, so that K / n lies just below, exactly on or just
  above every weight threshold of the GilbertCurve constructor, of ditherPixel and of the CIELAB quan_rt, at the palette
  length boundaries, with a dither-off subset for the BlueNoise second pass (k_bn_rgb_*, the CIELAB bn_weight at
  delta = .023). On the CPU the oracle must land every case where its name says; on the GPU every case must match the
  oracle's constants, palette, draw count and output bit for bit;
- one image for each of the six instantiations of the speculative stage 6 (k_spec_run<DITHER_MAX, ., NCH>), then all six
  with an image for k_dither_fifo and one for k_dither_sorted in one call, once more through three reused work-array slots;
- the alpha classes the synthetic images never produce (near-opaque: alpha in 0xE0..0xFE and none below; faint: alpha
  1..15 and no transparent pixel; each with and without alpha-0 pixels; the edges 0xDF / 0xE0 and 15 / 16) through every
  dither kernel and the index-map call;
- near-opaque images and a batch mixing instantiations through the speculative pipeline on the CPU
  (tests/spec_host_harness.cpp)."""
import ctypes
import multiprocessing
import os
import subprocess
import sys
import zlib
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_merge_limits import image_with_bins, scheme_for  # noqa: E402


def _pool():
    return ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn"))


def _side(q, t, side):
    return {"below": q < t, "on": q == t, "above": q > t}[side]


def _size(n):
    """The smallest of a few image sizes that holds n keys with repeats to spare."""
    for w, h in ((64, 64), (96, 96), (128, 128), (256, 128), (256, 256)):
        if 3 * n <= 2 * w * h:
            return w, h
    return 256, 256


# ---------------------------------------------------------------------------------------------------------------------
# the case table

# (label, threshold, K, n on the threshold, quantizers where it is live, what it decides). weight = K / n is correctly
# rounded, so K / n_on is the double of the threshold; n_on + 1 lies below it and n_on - 1 above.
WEIGHT_THRESHOLDS = [
    ("w0015", .0015, 6, 4000, (0, 1)),              # beta += .1 (plen 5..16); ditherPixel keeps the pixel (c1)
    ("w002", .002, 8, 4000, (0, 1)),                # sign of the ditherMax deviation
    ("w0025", .0025, 10, 4000, (0, 1)),             # margin 12 / 8, DITHER_MAX 16 / 25; ditherPixel .55 / .5, 1.82 / 2
    ("w003", .003, 24, 8000, (0, 1)),               # beta += .075 (plen 17..32)
    ("w004", .004, 16, 4000, (0, 1)),               # margin 8 / 6; ditherPixel (plen <= 32, weight >= .004)
    ("wbnd", .005 - .0000625 * 30, 30, 9600, (0, 1)),   # beta .25 above .005 - .0000625 plen (.003125 at 30 colours)
    ("w005", .005, 20, 4000, (0, 1)),               # beta (plen 17..32, weight <= .005); ditherPixel twice
    ("w01", .01, 60, 6000, (0, 1)),                 # ditherMax (5 + edge)^2: weight > .01, plen < 64, plen / weight > 5000
    ("w012", .012, 75, 6250, (0, 1)),               # beta += .05 (plen >= 64, .012 < weight < .0125)
    ("w0125", .0125, 75, 6000, (0, 1)),
    ("w015", .015, 48, 3200, (0, 1)),               # DITHER_MAX 25 / 9, isNano, beta .55 (plen 33..63)
    ("w02", .02, 160, 8000, (0, 1)),                # sortedByYDiff, beta * .4 or .18
    ("w025", .025, 40, 1600, (0, 1)),               # beta += .05 (.025 < weight < .03)
    ("w03", .03, 48, 1600, (0, 1)),                 # ... and ditherMax (5 + edge)^2 below .03 with plen / weight < 3200
    ("w045", .045, 243, 5400, (0, 1)),              # ditherMax (5 + edge)^2: weight > .045, plen / weight > 5000
    ("dp0008", .0008, 8, 10000, (1,)),              # ditherPixel normalDistribution peak 2.5 / 1.75
    ("dp007", .007, 28, 4000, (1,)),                # ditherPixel gamma = 1 - beta (plen <= 32, .007 < weight < .01)
    ("dp01", .01, 32, 3200, (1,)),
    ("qr001", .001, 16, 16000, (1,)),               # CIELAB quan_rt 2 below .001
    ("qr0015", .0015, 33, 22000, (1,)),             # ... 2 strictly between .0015 and .0022
    ("qr0022", .0022, 33, 15000, (1,)),
    ("qr0075", .0075, 15, 2000, (1,)),              # ... 2 below .0075 with fewer than 16 colours
]
# plen / weight against 5000 (with weight > .01 and plen < 64, or weight > .045) and against the density 3200 / 1500
# (weight < .03, 16 <= plen < 256; 3200 above 16 colours): plen / weight = n exactly here, so n_on - 1 is below
RATIO_THRESHOLDS = [("pw5000", 5000, 60, 5000, (0, 1)), ("pw5000_045", 5000, 243, 5000, (0, 1)),
                    ("pw3200", 3200, 64, 3200, (0, 1)), ("pw1500", 1500, 16, 1500, (0, 1))]
# the palette length boundaries, each at weight .02 (n = 50 K)
PLENS = (4, 5, 16, 17, 32, 33, 63, 64, 65, 128, 129, 255, 256)
# thresholds whose dither-off cases run the BlueNoise second pass (more than 32 colours)
OFF_LABELS = ("w015", "w02", "w045", "pw5000")
# (name, distinct colours, side): CIELAB bn_weight = 37.013 delta + .906 unless delta = plen^2 / pixelMap.size() > .023. The size
# counts every colour getLab has seen, the diffused ones of the Gilbert pass included, so the images come from a search:
# 46 colours and these distinct-colour counts put delta at .02305 (above) and .022996 (below)
BN_CASES = [("bn023_above", 29600, "above"), ("bn023_below", 30200, "below")]
BN_K = 46


def _cases():
    """(name, kind, K, n, alpha, dither, quantity, threshold, side)"""
    out = []
    for label, t, K, n_on, kinds in WEIGHT_THRESHOLDS:
        for side, n in (("below", n_on + 1), ("on", n_on), ("above", n_on - 1)):
            for kind in kinds:
                out.append((f"{label}_{side}_{'lab' if kind else 'rgb'}", kind, K, n, "opaque", True, "weight", t, side))
                if label in OFF_LABELS:
                    out.append((f"{label}_{side}_{'lab' if kind else 'rgb'}_off", kind, K, n, "opaque", False, "weight", t, side))
    for label, t, K, n_on, kinds in RATIO_THRESHOLDS:
        for side, n in (("below", n_on - 1), ("on", n_on), ("above", n_on + 1)):
            for kind in kinds:
                out.append((f"{label}_{side}_{'lab' if kind else 'rgb'}", kind, K, n, "opaque", True, "plen/weight", t, side))
                if label in OFF_LABELS:
                    out.append((f"{label}_{side}_{'lab' if kind else 'rgb'}_off", kind, K, n, "opaque", False, "plen/weight", t, side))
    for K in PLENS:
        for kind in (0, 1):
            out.append((f"plen{K}_{'lab' if kind else 'rgb'}", kind, K, 50 * K, "opaque", True, "weight", .02, "on"))
            if K in (32, 33, 255, 256):
                out.append((f"plen{K}_{'lab' if kind else 'rgb'}_off", kind, K, 50 * K, "opaque", False, "weight", .02, "on"))
    # 256 colours inside [.0125, .02), the regime of the headline images that no other test reaches: DITHER_MAX 25 -> 9
    # and isNano at .015, sortedByYDiff at .02
    for n, t, side in ((17067, .015, "below"), (17066, .015, "above"), (12801, .02, "below")):
        for kind in (0, 1):
            out.append((f"k256_{n}_{'lab' if kind else 'rgb'}", kind, 256, n, "opaque", True, "weight", t, side))
    # semi-transparent images (the weight reaches the GilbertCurve constructor negative): sortedByYDiff's `weight < .18`
    # and PnnQuantizer's isNano (nq_dither.cuh: !(weight > .015) on the signed weight)
    for label, t, K, n_on in (("a018", .18, 180, 1000), ("anano", .015, 48, 3200)):
        for side, n in (("below", n_on + 1), ("on", n_on), ("above", n_on - 1)):
            for kind in (0, 1):
                out.append((f"{label}_{side}_{'lab' if kind else 'rgb'}", kind, K, n, "semi", True, "weight", t, side))
    for name, d, side in BN_CASES:
        out.append((name, 1, BN_K, d, "opaque", False, "delta", .023, side))
    return out


CASES = _cases()
CASE_IDS = [c[0] for c in CASES]
assert len(set(CASE_IDS)) == len(CASE_IDS)


def _seed(name):
    return zlib.crc32(name.encode())


def image_with_colours(d, n_keys, w, h, seed):
    """w x h opaque pixels holding exactly d distinct colours, spread over n_keys 1-5-5-5 histogram keys (512 colours a key)."""
    rng = np.random.default_rng(seed)
    keys = rng.choice(32768, n_keys, replace=False).astype(np.int64)
    combo = rng.choice(n_keys * 512, d, replace=False).astype(np.int64)
    k, low = keys[combo // 512], combo % 512
    r, g, b = ((k >> 10) & 31) << 3 | (low >> 6), ((k >> 5) & 31) << 3 | ((low >> 3) & 7), (k & 31) << 3 | (low & 7)
    px = (255 << 24) | (r << 16) | (g << 8) | b
    px = np.concatenate([px, rng.choice(px, w * h - d)])
    return px[rng.permutation(w * h)].astype(np.uint32)


def case_image(case):
    name, kind, K, n, alpha, dither, q, t, side = case
    if q == "delta":
        return image_with_colours(n, 256, 256, 256, n), 256, 256
    w, h = _size(n)
    return image_with_bins(n, w, h, scheme_for(K, alpha), _seed(name)), w, h


def _oracle_case(case):
    from oracle import pyoracle
    img, w, h = case_image(case)
    return pyoracle.convert(case[1], img, w, h, case[2], case[5], seed=_seed(case[0]), trace=False)


@pytest.fixture(scope="module")
def table_refs(oracle):
    """The oracle's result of every case of the table, computed in a pool of host processes while the GPU runs."""
    ex = _pool()
    yield {c[0]: ex.submit(_oracle_case, c) for c in CASES}
    ex.shutdown(cancel_futures=True)


def expected_nano(kind, weight, semi):
    """isNano: PnnLABQuantizer latches weight <= .015 in pnnquan; PnnQuantizer's nearestColorIndex reads the field after
    the sign flip of a semi-transparent image, i.e. !(-weight > .015)."""
    return weight <= .015 if kind else not ((-weight if semi else weight) > .015)


def expected_lab_quan_rt(K, weight):
    """PL:130-190 for an image without transparent or semi-transparent pixels."""
    q = 1
    if (K < 16 and weight < .0075) or weight < .001 or (.0015 < weight < .0022):
        q = 2
    if weight < .04 and K >= 64:
        q = 0
    if 16 < K < 64 and abs(K / 8000.0 - weight) < .001:
        q = 2
    return q


def test_every_case_lands_on_its_side(table_refs):
    """The oracle's scalars of every case: exactly n histogram keys and a palette of K colours, weight = K / n, the quantity
    the case is named for on the named side of its threshold, and the decisions that hang on it -- margin, DITHER_MAX,
    sortedByYDiff, isNano, CIELAB quan_rt -- as the reference's rules give them for that weight."""
    bad = []
    for case in CASES:
        name, kind, K, n, alpha, dither, q, t, side = case
        r = table_refs[name].result()
        s = r.scalars
        semi = alpha == "semi"
        try:
            assert len(r.palette) == K, ("palette", len(r.palette))
            assert s["hasSemiTransparency"] == semi and s["transparentPixelIndex"] < 0
            if q == "delta":
                assert _side(K * K / s["pixelMapSize"], t, side), ("delta", K * K / s["pixelMapSize"])
                want = 1.0 if K * K / s["pixelMapSize"] > .023 else np.float32(37.013 * (K * K / s["pixelMapSize"]) + .906)
                assert np.float32(s["bn_weight"]) == np.float32(want) and (side == "above") == (s["bn_weight"] == 1.0)
                continue
            w = K / n
            assert s["maxbins"] == n, ("maxbins", s["maxbins"])
            assert s["weight"] == w, ("weight", s["weight"])
            assert _side(w if q == "weight" else len(r.palette) / w, t, side), (q, w)
            sw = -w if semi else w                       # what the GilbertCurve constructor reads
            assert s["hasAlpha"] == semi
            assert s["margin"] == (12 if sw < .0025 else 8 if sw < .004 else 6), ("margin", s["margin"])
            assert s["DITHER_MAX"] == (9 if sw >= .015 else 25 if sw > .0025 else 16), ("DITHER_MAX", s["DITHER_MAX"])
            assert s["sortedByYDiff"] == (K > 128 and sw >= .02 and (not semi or sw < .18)), ("sorted", s["sortedByYDiff"])
            if kind:
                assert s["isNano"] == expected_nano(1, w, semi), ("isNano", s["isNano"])
                if not semi:
                    assert s["quan_rt"] == expected_lab_quan_rt(K, w), ("quan_rt", s["quan_rt"])
        except AssertionError as e:
            bad.append((name, str(e)))
    assert not bad, bad


def test_table_covers_every_threshold_side_and_quantizer():
    have = {(c[0].rsplit("_", 2 if c[0].endswith("_off") else 1)[0], c[1], c[5]) for c in CASES}
    for label, t, K, n_on, kinds in WEIGHT_THRESHOLDS + RATIO_THRESHOLDS:
        for side in ("below", "on", "above"):
            for kind in kinds:
                assert (f"{label}_{side}", kind, True) in have, (label, side, kind)
                if label in OFF_LABELS:
                    assert (f"{label}_{side}", kind, False) in have
    # the semi-transparent thresholds, both quantizers
    for label in ("a018", "anano"):
        for side in ("below", "on", "above"):
            assert {(f"{label}_{side}", k, True) for k in (0, 1)} <= have


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_table_case_matches_oracle(gpu_ctx, table_refs, case):
    name, kind, K, n, alpha, dither, q, t, side = case
    img, w, h = case_image(case)
    out, pal, plen, _ = gpu_ctx.convert_batch(kind, img[None, :], w, h, K, dither, seeds=[_seed(name)])
    info = gpu_ctx.image_info(0)
    r = table_refs[name].result()
    s = r.scalars
    assert info["maxbins"] == s["maxbins"] and info["weight"] == s["weight"] and info["quan_rt"] == s["quan_rt"]
    for g, o in [("g_margin", "margin"), ("g_thresold", "thresold"), ("g_dither_max_q", "DITHER_MAX"),
                 ("g_dither_max", "ditherMax"), ("g_sorted", "sortedByYDiff"), ("g_has_alpha", "hasAlpha")]:
        assert info[g] == s[o], (g, info[g], s[o])
    assert np.float32(info["g_beta"]) == np.float32(s["beta"]), (info["g_beta"], s["beta"])
    assert info["is_nano"] == (s["isNano"] if kind else expected_nano(0, s["weight"], alpha == "semi"))
    if not dither and plen[0] > 32 and kind == 1:
        assert np.float32(info["bn_weight"]) == np.float32(s["bn_weight"]), (info["bn_weight"], s["bn_weight"])
    assert np.array_equal(pal[0, :plen[0]], r.palette), "palette differs"
    assert info["rng_draws"] == s["rng_draws"]
    assert np.array_equal(out[0], r.out), f"{int((out[0] != r.out).sum())} of {w * h} output pixels differ"


# ---------------------------------------------------------------------------------------------------------------------
# alpha classes

def with_alpha(img, cls, seed):
    """Replaces the alpha of an opaque image. near_opaque: every alpha in 0xE0..0xFE, both ends present; faint: one pixel in
    eight alpha 1..15 (15 present), the rest opaque; '_alpha0': one pixel in sixteen fully transparent; near_opaque_df and
    faint_16: one pixel in 64 at 0xDF or 16, the first semi-transparent alpha below each class."""
    rng = np.random.default_rng(seed)
    rgb = img.astype(np.int64) & 0xFFFFFF
    npix = rgb.size
    free = np.arange(npix) >= 2                     # pixels 0 and 1 keep the class's extreme alphas
    a = np.full(npix, 255, np.int64)
    if cls.startswith("near_opaque"):
        a = rng.integers(0xE0, 0xFF, npix)
        a[:2] = (0xE0, 0xFE)
    if cls.startswith("faint"):
        m = (rng.random(npix) < 1 / 8) & free
        a[m] = rng.integers(1, 16, int(m.sum()))
        a[0] = 15
    if cls.endswith("_alpha0"):
        a[(rng.random(npix) < 1 / 16) & free] = 0
    if cls.endswith("_df") or cls.endswith("_16"):
        a[(rng.random(npix) < 1 / 64) & free] = 0xDF if cls.endswith("_df") else 16
    return ((a << 24) | rgb)[rng.permutation(npix)].astype(np.uint32)


ALPHA_CLASSES = ("near_opaque", "near_opaque_alpha0", "faint", "faint_alpha0", "near_opaque_df", "faint_16")
SEMI_CLASSES = ("near_opaque_df", "faint_16")


def _alpha_configs(cls):
    """(n, kind, K, dither): 20 000 keys give 256 colours a weight of .0128 (DITHER_MAX 25, ArrayDeque queue:
    k_spec_run or k_dither_fifo), 6000 keys .043 (PriorityQueue: k_dither_sorted for CIELAB). PnnQuantizer without dither
    runs k_bn_rgb_*; PnnLABQuantizer without dither its BlueNoise pass (32 colours for semi-transparent images, which it
    does not take above 32). 16 colours meet the `plen <= 32 && a_pix > 0xF0` branch of diffusePixel."""
    lab_off = (20000, 1, 32 if cls in SEMI_CLASSES else 256, False)
    return [(20000, 1, 256, True), (20000, 0, 256, True), (20000, 0, 256, False), lab_off, (20000, 1, 16, True),
            (20000, 0, 16, True), (6000, 1, 256, True)]


ALPHA_CASES = [(f"{cls}_n{n}_{'lab' if kind else 'rgb'}{K}_{'on' if d else 'off'}", cls, n, kind, K, d)
               for cls in ALPHA_CLASSES for n, kind, K, d in _alpha_configs(cls)]


def alpha_image(cls, n):
    return with_alpha(image_with_bins(n, 256, 256, "565", 7000 + n), cls, zlib.crc32(cls.encode()) + n)


def _oracle_alpha(case):
    from oracle import pyoracle
    name, cls, n, kind, K, d = case
    return pyoracle.convert(kind, alpha_image(cls, n), 256, 256, K, d, seed=_seed(name), trace=False)


@pytest.fixture(scope="module")
def alpha_refs(oracle):
    ex = _pool()
    yield {c[0]: ex.submit(_oracle_alpha, c) for c in ALPHA_CASES}
    ex.shutdown(cancel_futures=True)


def test_alpha_images_are_in_their_class():
    for cls in ALPHA_CLASSES:
        a = alpha_image(cls, 20000) >> 24
        semi = ((a > 15) & (a < 0xE0)).any()
        assert semi == (cls in SEMI_CLASSES), cls
        assert (a == 0).any() == cls.endswith("_alpha0"), cls
        assert ((a >= 1) & (a <= 15)).any() == cls.startswith("faint"), cls
        if cls.startswith("near_opaque"):
            assert a.min() in (0, 0xDF, 0xE0) and a.max() == 0xFE and (a == 0xE0).any()
        else:
            assert a.max() == 255 and (a == 15).any()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ALPHA_CASES, ids=[c[0] for c in ALPHA_CASES])
def test_alpha_class_matches_oracle(gpu_ctx, alpha_refs, case):
    name, cls, n, kind, K, dither = case
    img = alpha_image(cls, n)
    out, pal, plen, ha = gpu_ctx.convert_batch(kind, img[None, :], 256, 256, K, dither, seeds=[_seed(name)])
    info = gpu_ctx.image_info(0)
    r = alpha_refs[name].result()
    s = r.scalars
    assert info["has_semi_transparency"] == s["hasSemiTransparency"] == (cls in SEMI_CLASSES)
    assert info["transparent_pixel_index"] == s["transparentPixelIndex"] and bool(ha[0]) == (s["transparentPixelIndex"] >= 0)
    assert info["maxbins"] == s["maxbins"] and info["quan_rt"] == s["quan_rt"]
    for g, o in [("g_margin", "margin"), ("g_dither_max_q", "DITHER_MAX"), ("g_dither_max", "ditherMax"),
                 ("g_sorted", "sortedByYDiff"), ("g_has_alpha", "hasAlpha")]:
        assert info[g] == s[o], (g, info[g], s[o])
    assert np.float32(info["g_beta"]) == np.float32(s["beta"])
    if kind == 1 and not dither and plen[0] > 32:
        assert np.float32(info["bn_weight"]) == np.float32(s["bn_weight"])
    assert np.array_equal(pal[0, :plen[0]], r.palette), "palette differs"
    assert info["rng_draws"] == s["rng_draws"]
    assert np.array_equal(out[0], r.out), f"{int((out[0] != r.out).sum())} of {256 * 256} output pixels differ"
    if n == 20000 and K == 256 and kind == 1 and dither and cls == "near_opaque":
        assert s["DITHER_MAX"] == 25 and not s["sortedByYDiff"]   # the speculative path's 4-channel image of this table


INDEXED = [c for c in ALPHA_CASES if c[4] == 256 and c[2] == 20000 and (c[3], c[5]) in ((1, True), (0, False))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", INDEXED, ids=[c[0] for c in INDEXED])
def test_alpha_class_index_map(gpu_ctx, alpha_refs, case):
    """Palettes of these images hold colours that differ only in alpha: the index map must still be the lowest index of
    each output colour, and palette[index] the oracle's output."""
    from nquant_android_b200.imageio import to_indices
    name, cls, n, kind, K, dither = case
    img = alpha_image(cls, n).reshape(256, 256)
    idx, _, pal, plen, _ = gpu_ctx.convert_indexed(kind, [img], K, dither, seeds=[_seed(name)])
    r = alpha_refs[name].result()
    assert np.array_equal(pal[0, :plen[0]], r.palette)
    assert np.array_equal(idx[0].reshape(-1), to_indices(r.out, r.palette).reshape(-1))
    assert np.array_equal(r.palette[idx[0].reshape(-1)], r.out)


# ---------------------------------------------------------------------------------------------------------------------
# the six instantiations of k_spec_run

# One palette size for the whole mixed call: the PriorityQueue needs more than 128 colours, and at 130 DITHER_MAX 9 without
# it lies in [.015, .02) (n 6501..8666), DITHER_MAX 25 in (.0025, .015) and DITHER_MAX 16 at weight .0025 (n = 52 000).
SPEC_K = 130
SPEC_IMAGES = [  # (name, n, alpha, DITHER_MAX or the serial kernel)
    ("dm9_opaque", 8000, "opaque", 9), ("dm9_near", 8000, "near_opaque", 9),
    ("dm16_opaque", 52000, "opaque", 16), ("dm16_near", 52000, "near_opaque", 16),
    ("dm25_opaque", 20000, "opaque", 25), ("dm25_near", 20000, "near_opaque", 25),
    ("fifo", 20000, "transparent", "fifo"), ("sorted", 4000, "opaque", "sorted"),
]
SPEC_SEG, SPEC_WARM = 2048, 512


def spec_image(name, n, alpha):
    if alpha == "transparent":
        return image_with_bins(n, 256, 256, "1555", 9100 + n, transparent=True)
    img = image_with_bins(n, 256, 256, "565", 9000 + n)
    return with_alpha(img, "near_opaque", n) if alpha == "near_opaque" else img


def _oracle_spec(item):
    from oracle import pyoracle
    name, n, alpha, _ = item
    return pyoracle.convert(1, spec_image(name, n, alpha), 256, 256, SPEC_K, True, seed=_seed(name), trace=False)


@pytest.fixture(scope="module")
def spec_refs(oracle):
    ex = _pool()
    yield {it[0]: ex.submit(_oracle_spec, it) for it in sorted(SPEC_IMAGES, key=lambda it: -it[1])}
    ex.shutdown(cancel_futures=True)


@pytest.fixture(scope="module")
def spec_ctx():
    from nquant_android_b200 import _build
    from nquant_android_b200.quantizer import Context
    _build.build()
    ctx = Context(0)
    ctx.set_spec_dither(True, SPEC_SEG, SPEC_WARM)
    yield ctx
    ctx.close()


def four_channels(img, palette):
    """k_spec_setup's choice: stage 6 keeps the alpha errors (NCH 4) unless every pixel is opaque and every palette alpha
    is 254 or 255."""
    return bool(((img >> 24) != 255).any() or ((palette >> 24) < 254).any())


def _check_spec_result(name, img, out, pal, plen, info, r):
    assert np.array_equal(pal[:plen], r.palette), (name, "palette")
    assert info["rng_draws"] == r.scalars["rng_draws"], name
    assert np.array_equal(out, r.out), (name, f"{int((out != r.out).sum())} output pixels differ")


SIX = [it for it in SPEC_IMAGES if isinstance(it[3], int)]


@pytest.mark.gpu
@pytest.mark.parametrize("item", SIX, ids=[it[0] for it in SIX])
def test_each_spec_instantiation(spec_ctx, spec_refs, item):
    name, n, alpha, dm = item
    img = spec_image(name, n, alpha)
    r = spec_refs[name].result()
    assert r.scalars["DITHER_MAX"] == dm and not r.scalars["sortedByYDiff"] and r.scalars["transparentPixelIndex"] < 0
    assert four_channels(img, r.palette) == (alpha == "near_opaque")
    before = spec_ctx.spec_stats()
    out, pal, plen, _ = spec_ctx.convert_batch(1, img[None, :], 256, 256, SPEC_K, True, seeds=[_seed(name)])
    info = spec_ctx.image_info(0)
    assert info["g_dither_max_q"] == dm
    _check_spec_result(name, img, out[0], pal[0], plen[0], info, r)
    st = spec_ctx.spec_stats()
    assert st["images"] == before["images"] + 1 and st["fallbacks"] == 0, (before, st)


def _mixed_call(ctx, spec_refs):
    imgs = np.stack([spec_image(name, n, alpha) for name, n, alpha, _ in SPEC_IMAGES])
    before = ctx.spec_stats()
    out, pal, plen, _ = ctx.convert_batch(1, imgs, 256, 256, SPEC_K, True, seeds=[_seed(it[0]) for it in SPEC_IMAGES])
    for i, (name, n, alpha, dm) in enumerate(SPEC_IMAGES):
        info = ctx.image_info(i)
        r = spec_refs[name].result()
        if dm == "sorted":
            assert info["g_sorted"] == 1
        elif dm == "fifo":
            assert info["g_sorted"] == 0 and info["transparent_pixel_index"] >= 0
        else:
            assert info["g_dither_max_q"] == dm and info["g_sorted"] == 0
        _check_spec_result(name, imgs[i], out[i], pal[i], plen[i], info, r)
    st = ctx.spec_stats()
    assert st["images"] == before["images"] + len(SIX) and st["fallbacks"] == 0, (before, st)


@pytest.mark.gpu
def test_all_six_instantiations_in_one_call(spec_ctx, spec_refs):
    """Six speculative groups (one per instantiation) with k_dither_fifo and k_dither_sorted beside them, in one call."""
    _mixed_call(spec_ctx, spec_refs)


@pytest.mark.gpu
def test_all_six_instantiations_through_three_slots(spec_refs, monkeypatch):
    """The same call through three work-array slots in chunks of three images: images of different instantiations are
    admitted into slots other images have left."""
    from nquant_android_b200.quantizer import Context
    monkeypatch.setenv("NQ_SPEC_SLOTS", "3")
    ctx = Context(0)
    try:
        ctx.set_spec_dither(True, SPEC_SEG, SPEC_WARM)
        ctx.set_chunk_images(3)
        _mixed_call(ctx, spec_refs)
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# the speculative pipeline on the CPU (tests/spec_host_harness.cpp) with near-opaque images and mixed instantiations

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_SO = os.path.join(ROOT, "build", "libnq_spec_host.so")
HOST_SRC = os.path.join(ROOT, "tests", "spec_host_harness.cpp")
HOST_DEPS = [HOST_SRC] + [os.path.join(ROOT, *p) for p in (("oracle", "nq_oracle.cpp"), ("nquant_android_b200", "csrc", "nq_dither_spec.cuh"),
                                                            ("nquant_android_b200", "csrc", "nq_color.h"), ("nquant_android_b200", "csrc", "nq_math.h"))]
HOST_KEYS = ["eligible", "exact", "rounds", "anomaly", "nseg", "segRuns", "slowPixels", "notes", "mismatches", "rejected", "patches", "redos"]


@pytest.fixture(scope="module")
def host_lib():
    os.makedirs(os.path.dirname(HOST_SO), exist_ok=True)
    if not os.path.exists(HOST_SO) or os.path.getmtime(HOST_SO) < max(os.path.getmtime(d) for d in HOST_DEPS):
        fma = ["-mfma"] if " fma " in open("/proc/cpuinfo").read() else []
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-w"] + fma +
                              ["-o", HOST_SO, HOST_SRC])
    L = ctypes.CDLL(HOST_SO)
    vp, ci = ctypes.c_void_p, ctypes.c_int
    L.nqs_spec_host.argtypes = [vp, ci, ci, ci, ci, ctypes.c_uint64, ci, ci, ci, vp]
    L.nqs_spec_batch_add.argtypes = [vp, ci, ci, ci, ctypes.c_uint64, ci, ci]
    L.nqs_spec_batch_run.argtypes = [ci, ci, ci, vp]
    return L


# the images of the GPU tests above: the CPU pipeline must be exact on the near-opaque ones, and the emulated batch of all
# six needs every instantiation. (Near-opaque DITHER_MAX 16 images of 65 to 70 colours are handed back to the serial kernel:
# below 128 colours their lookups read the diffused colour, and an exact run of one segment creates more than NQS_NOTES memo
# entries. Their result stays exact, but they do not run stage 6 to the end, hence 130 colours here.)
NEAR = [it for it in SIX if it[2] == "near_opaque"]


@pytest.mark.parametrize("item", NEAR, ids=[it[0] for it in NEAR])
def test_host_pipeline_near_opaque(host_lib, item):
    name, n, alpha, dm = item
    img = np.ascontiguousarray(spec_image(name, n, alpha))
    out = np.zeros(12, np.int64)
    assert host_lib.nqs_spec_host(img.ctypes.data, 256, 256, SPEC_K, 1, _seed(name), SPEC_SEG, SPEC_WARM, 1, out.ctypes.data) == 0
    r = dict(zip(HOST_KEYS, [int(v) for v in out]))
    assert r["eligible"] == 1 and r["anomaly"] == 0 and r["rejected"] == 0, r
    assert r["mismatches"] == 0 and r["exact"] == 1, r


def test_host_batch_mixes_instantiations(host_lib):
    """k_spec_setup, spec_drive and the k_spec_run instantiations run thread by thread on a batch of the six images, one per
    instantiation, through wave slots of two: every image completed by the path and equal to the oracle."""
    host_lib.nqs_spec_batch_begin()
    for name, n, alpha, _ in SIX:
        img = np.ascontiguousarray(spec_image(name, n, alpha))
        assert host_lib.nqs_spec_batch_add(img.ctypes.data, 256, 256, SPEC_K, _seed(name), SPEC_SEG, SPEC_WARM) == 0
    out = np.zeros(9, np.int64)
    assert host_lib.nqs_spec_batch_run(SPEC_SEG, SPEC_WARM, 2, out.ctypes.data) == 0
    r = dict(zip(["images", "eligible", "completed", "handed_back", "rounds", "patches", "redos", "wrong", "launches"], [int(v) for v in out]))
    assert r["images"] == 6 and r["eligible"] == 6 and r["completed"] == 6 and r["handed_back"] == 0, r
    assert r["wrong"] == 0, r
