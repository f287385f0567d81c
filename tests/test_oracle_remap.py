"""The remap oracle (tests/remap_oracle.cpp): the oracle's convert() with the caller's palette dithered to in place of its
own. The round trip is the invariant the GPU's remap is checked against: remapping an image to the palette
its own convert() produced, with the same n_max_colors and seed, must return convert()'s output and RNG draws exactly --
over both quantizers, palette sizes on both sides of the 32 and 64 thresholds, dither on and off, every synthetic class and
alpha mode, and the few-colours images of PnnLABQuantizer's early return. The oracle covers every branch, including the one
the GPU leaves unsupported (PnnLABQuantizer, dither off, semi-transparent pixels, more than 32 colours)."""
import os
import sys

import numpy as np
import pytest

from nquant_android_b200.synth import make_image

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import remap_oracle  # noqa: E402

W, H = 48, 40
KS = [2, 16, 32, 33, 64, 65, 256]
IMAGES = [(cls, alpha) for cls in ("smooth", "noisy", "rand") for alpha in ("opaque", "transparent", "semi")] + [("few", "opaque")]


@pytest.mark.parametrize("dither", [True, False], ids=["on", "off"])
@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_remap_to_the_convert_palette_is_convert(oracle, kind, K, dither):
    for i, (cls, alpha) in enumerate(IMAGES):
        img = make_image(W, H, cls, alpha, seed=0x5EED0700 + i)
        seed = 40 + i
        ref = oracle.convert(kind, img, W, H, K, dither, seed=seed, trace=False)
        got = remap_oracle.remap(kind, img, W, H, K, dither, ref.palette, seed=seed)
        what = f"{cls}_{alpha}"
        assert np.array_equal(got.out, ref.out), what
        assert got.scalars["rng_draws"] == ref.scalars["rng_draws"], what
        for k in ("weight", "weight_final", "ratio_merge", "isNano", "maxbins", "bn_weight", "pixelMapSize"):
            assert got.scalars[k] == ref.scalars[k], (what, k)


@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_the_callers_palette_wins_over_the_fixed_one(oracle, kind):
    """n_max_colors <= 2 takes the fixed-palette branch of convert (black and white here); a remap dithers to the caller's
    two colours instead, as a two-colour e-ink panel needs."""
    img = make_image(W, H, "noisy", "opaque", seed=0x5EED0777)
    pal = np.array([0xFFFF0000, 0xFF0000FF], dtype=np.uint32)
    got = remap_oracle.remap(kind, img, W, H, 2, True, pal, seed=3)
    assert set(np.unique(got.out)) == {0xFFFF0000, 0xFF0000FF}
    fixed = oracle.convert(kind, img, W, H, 2, True, seed=3, trace=False)
    assert list(fixed.palette) == [0xFF000000, 0xFFFFFFFF]
    assert np.array_equal(remap_oracle.remap(kind, img, W, H, 2, True, fixed.palette, seed=3).out, fixed.out)
