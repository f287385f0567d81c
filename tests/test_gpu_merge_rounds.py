"""The CIELAB merge loop rescans stale heap entries in rounds of several bins and replays the reference's heap
loop with their results (nq_pnn.cuh, k_merge_lab). The merge sequence must stay the oracle's, the rescans applied
must stay the reference's own count, and the rounds must actually batch them: fewer rounds than rescans, and more
rounds than merges (some merge intervals hold more stale entries than one round takes, so a round starts after
another round's results were applied)."""
import numpy as np
import pytest

from nquant_android_b200.synth import make_image

pytestmark = pytest.mark.gpu


def _merge_and_rounds(gpu_ctx, oracle, W, H, cls, K, dither, seed):
    img = make_image(W, H, cls, "opaque")
    ref = oracle.convert(1, img, W, H, K, dither, seed=seed)
    gpu_ctx.set_debug(True)
    try:
        out, pal, plen, _ = gpu_ctx.convert_batch(1, img[None, :], W, H, K, dither, seeds=[seed])
        info = gpu_ctx.image_info(0)
        assert np.array_equal(gpu_ctx.debug_merges(0), ref.merges), "merge sequence differs"
    finally:
        gpu_ctx.set_debug(False)
    assert np.array_equal(pal[0, :plen[0]], ref.palette) and np.array_equal(out[0], ref.out)
    assert info["merges"] == len(ref.merges)
    return info


def test_rounds_headline_class_512(gpu_ctx, oracle):
    info = _merge_and_rounds(gpu_ctx, oracle, 512, 512, "noisy", 256, True, 0xC0FFEE)
    assert info["rescans"] == 58016                        # the reference's rescans, one at a time
    assert info["merges"] < info["merge_rounds"] < info["rescans"], info


def test_rounds_noisy_1080p(gpu_ctx, oracle):
    info = _merge_and_rounds(gpu_ctx, oracle, 1920, 1080, "noisy", 256, False, 7)
    assert info["merges"] < info["merge_rounds"] < info["rescans"], info


def test_rounds_smooth_few_bins_16_colours(gpu_ctx, oracle):
    """Few bins, so the whole heap sits in shared memory and the rounds run into its last levels; 16 colours run
    the merge loop almost to the end of the heap."""
    info = _merge_and_rounds(gpu_ctx, oracle, 320, 240, "smooth", 16, True, 5)
    assert 0 < info["merge_rounds"] <= info["rescans"], info
