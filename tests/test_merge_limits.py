"""The merge loops at the limits of their fixed-size tables. A heap slot l sits in shared memory when l < HS and in the
global spill (S.heap) otherwise: HS is 2048 for k_merge_lab<8>, 5632 for k_merge_lab<4> and 6144 for k_merge_rgb. The
heap build, HeapView::set/err/idnn and sift_down switch sides at HS, and sift_down reads two children with one 16-byte
load past it. With all 65 536 histogram keys occupied every table of the merge loops is exactly full: the 11-bit block
field of sBat, sBits/sPre, the 16-bit position of sPos, bin ids and nn of 65 535 in pack_idnn, k_merge_rgb's sBlk and
block planes of 2048, and heap slot 65 536 (its child load reaches slot 65 537 of an NQ_NBINS + 2 allocation).

image_with_bins() builds images with an exact number of histogram keys (getColorIndex, BU:8-15), so each case lands on
the limit it is named for, and the oracle's counters of rescans and heap pops check the replay beyond its merge order."""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

# keys a scheme can hold besides the one key of the transparent colour (every pixel of alpha <= 15 becomes that colour)
KEY_SPACE = {"565": 65536, "1555": 32768, "4444": 15 * 4096}
# the largest 4-4-4-4 alpha nibble that is semi-transparent (alpha < 0xE0)
SEMI_NIBBLES = 13


def scheme_for(n_max_colors, alpha="opaque"):
    """The key scheme getColorIndex uses: 4-4-4-4 with semi-transparent pixels, 1-5-5-5 with a transparent pixel or
    fewer than 64 colours, 5-6-5 otherwise."""
    if alpha == "semi":
        return "4444"
    return "1555" if alpha == "transparent" or n_max_colors < 64 else "565"


def image_with_bins(n, w, h, scheme, seed, transparent=False):
    """w x h ARGB pixels whose histogram keys under `scheme` are exactly n distinct values. Every key is used at least
    once, the remaining pixels repeat keys at random, and the bits below each key are random. With transparent=True one
    of the n keys is that of a transparent colour (alpha 0). 1-5-5-5 holds at most 32 768 opaque keys and 4-4-4-4 at most
    61 440 keys of alpha >= 16; at least one 4-4-4-4 key is semi-transparent."""
    rng = np.random.default_rng(seed)
    m = n - int(transparent)
    npix = w * h
    assert 0 < m <= KEY_SPACE[scheme] and n <= npix, (n, w, h, scheme)
    keys = rng.choice(KEY_SPACE[scheme], m, replace=False).astype(np.int64)
    if scheme == "4444" and not (keys < SEMI_NIBBLES * 4096).any():
        keys[0] = rng.integers(SEMI_NIBBLES * 4096)
    t = min(max(1, npix // 64), npix - m) if transparent else 0
    k = np.concatenate([keys, rng.choice(keys, npix - m - t)])

    def low(bits):
        return rng.integers(0, 1 << bits, k.size)

    if scheme == "565":
        a, r, g, b = np.full(k.size, 255), (k >> 11) << 3 | low(3), ((k >> 5) & 63) << 2 | low(2), (k & 31) << 3 | low(3)
    elif scheme == "1555":
        a, r, g, b = np.full(k.size, 255), ((k >> 10) & 31) << 3 | low(3), ((k >> 5) & 31) << 3 | low(3), (k & 31) << 3 | low(3)
    else:
        a, r, g, b = (1 + (k >> 12)) << 4 | low(4), ((k >> 8) & 15) << 4 | low(4), ((k >> 4) & 15) << 4 | low(4), (k & 15) << 4 | low(4)
    px = a << 24 | r << 16 | g << 8 | b
    if t:
        px = np.concatenate([px, np.full(t, int(rng.integers(0, 1 << 24)))])
    return px[rng.permutation(npix)].astype(np.uint32)


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------
# heap slots in shared memory (the split) of the instance a single image runs on: k_merge_lab<4> and k_merge_rgb
HEAP_SPLIT = {1: 5632, 0: 6144}
# CTAs per SM of k_merge_lab<4>: __launch_bounds__(128, 4) caps it at 128 registers a thread, so four CTAs take all 64 K
# registers of an SM; k_merge_lab<8> holds 8 (64 registers)
LAB4_CTAS = 4

# the cases: (name, kind, n, w, h, K, alpha, image seed, rng seed)
SPLIT_CASES = [(f"{'lab' if kind else 'rgb'}_{HEAP_SPLIT[kind] + d}_k{K}", kind, HEAP_SPLIT[kind] + d, 96, 96, K, "opaque",
                1000 + HEAP_SPLIT[kind] + d + K, 77 + HEAP_SPLIT[kind] + d)
               for kind in (1, 0) for d in (-1, 0, 1) for K in (256, 16)]
FULL_CASES = [("rgb_65536", 0, 65536, 256, 256, 256, "opaque", 11, 5), ("lab_65536", 1, 65536, 256, 256, 256, "opaque", 12, 6),
              ("rgb_semi_61441", 0, 61441, 256, 256, 256, "semi", 13, 7)]


def _case_image(kind, n, w, h, K, alpha, img_seed):
    return image_with_bins(n, w, h, scheme_for(K, alpha), img_seed, transparent=alpha == "semi" and n > KEY_SPACE["4444"])


# palette sizes of the eight-per-SM batch: 256 colours (5-6-5 keys) and 16 (1-5-5-5 keys, the merge loop runs the heap
# almost empty through the 2048 split); a call takes one palette size, so each is a batch of its own
BATCH_KS = (256, 16)


def _batch_cases(n_images):
    """(bins, image seed, rng seed) of n_images 96 x 96 images: bin counts spread from 1900 to 6000, exact at 2047-2049
    and 5631-5633 and dense around both splits, distinct rng seeds."""
    exact = [2047, 2048, 2049, 5631, 5632, 5633]
    dense = list(range(2030, 2070)) + list(range(5610, 5650))
    rest = max(0, n_images - len(exact) - len(dense))
    ns = (exact + dense + list(np.linspace(1900, 6000, rest).astype(int)))[:n_images]
    return [(int(n), 5000 + i, 900 + 7 * i) for i, n in enumerate(ns)]


def _oracle_job(kind, img, w, h, K, seed):
    from oracle import pyoracle
    r = pyoracle.convert(kind, img, w, h, K, True, seed=seed)
    del r.saliencies, r.gweights
    return r


@pytest.fixture(scope="module")
def refs(oracle):
    """The oracle's results of every case of this file, computed in a pool of host processes while the GPU runs."""
    ex = ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn"))
    futs = {}
    for name, kind, n, w, h, K, alpha, img_seed, seed in FULL_CASES + SPLIT_CASES:
        futs[name] = ex.submit(_oracle_job, kind, _case_image(kind, n, w, h, K, alpha, img_seed), w, h, K, seed)
    for K in BATCH_KS:
        for i, (n, img_seed, seed) in enumerate(_batch_cases(4 * _sms() + 1)):
            futs[("batch", K, i)] = ex.submit(_oracle_job, 1, image_with_bins(n, 96, 96, scheme_for(K), img_seed), 96, 96, K,
                                              seed)
    yield futs
    ex.shutdown(cancel_futures=True)


def _check_single(gpu_ctx, ref, kind, n, w, h, K, alpha, img_seed, seed):
    img = _case_image(kind, n, w, h, K, alpha, img_seed)
    gpu_ctx.set_debug(True)
    try:
        out, pal, plen, _ = gpu_ctx.convert_batch(kind, img[None, :], w, h, K, True, seeds=[seed])
        info = gpu_ctx.image_info(0)
        bins, ierr, inn = gpu_ctx.debug_bins(0)
        merges = gpu_ctx.debug_merges(0)
    finally:
        gpu_ctx.set_debug(False)
    r = ref.result()
    s = r.scalars
    assert info["maxbins"] == n and s["maxbins"] == n
    assert np.array_equal(bins, r.bins), "histogram bins (means, counts) differ"
    assert np.array_equal(ierr.view(np.uint32), r.init_err.view(np.uint32)) and np.array_equal(inn, r.init_nn)
    assert np.array_equal(merges, r.merges), "merge sequence differs"
    assert info["rescans"] == s["n_rescans"] and info["heap_pops"] == s["n_heap_pops"], (info, s)
    assert np.array_equal(pal[0, :plen[0]], r.palette), "palette differs"
    assert info["rng_draws"] == s["rng_draws"]
    assert np.array_equal(out[0], r.out), f"{int((out[0] != r.out).sum())} of {w * h} output pixels differ"
    return info


# ---------------------------------------------------------------------------------------------------------------------
# host: the helper's key counts and the oracle's counters

def _keys(img, scheme):
    """getColorIndex (BU:8-15) of every pixel after the reference's alpha handling (alpha <= 15 -> transparent colour)."""
    p = img.astype(np.int64)
    a, r, g, b = p >> 24 & 255, p >> 16 & 255, p >> 8 & 255, p & 255
    if scheme == "4444":
        k = (a & 0xF0) << 8 | (r & 0xF0) << 4 | (g & 0xF0) | b >> 4
    elif scheme == "1555":
        k = (a & 0x80) << 8 | (r & 0xF8) << 7 | (g & 0xF8) << 2 | b >> 3
    else:
        k = (r & 0xF8) << 8 | (g & 0xFC) << 3 | b >> 3
    return np.where(a <= 15, -1, k)


HELPER_CASES = [("565", 256, n, False) for n in (65536, 6145, 2049)] + \
               [("1555", 16, n, False) for n in (32768, 6145, 2049)] + [("1555", 256, 32769, True)] + \
               [("4444", 256, n, n > 61440) for n in (61441, 6145, 2049)]


@pytest.mark.parametrize("scheme,K,n,transparent", HELPER_CASES)
def test_image_with_bins_has_exactly_n_keys(scheme, K, n, transparent):
    w = h = 256 if n > 9216 else 96
    img = image_with_bins(n, w, h, scheme, seed=n + K, transparent=transparent)
    alpha = img >> 24
    assert scheme_for(K, "semi" if ((alpha > 15) & (alpha < 0xE0)).any() else "transparent" if (alpha == 0).any() else "opaque") == scheme
    assert len(np.unique(_keys(img, scheme))) == n


def _oracle_maxbins(args):
    kind, scheme, K, n, transparent = args
    from oracle import pyoracle
    w = h = 256 if n > 9216 else 96
    img = image_with_bins(n, w, h, scheme, seed=n + K, transparent=transparent)
    return pyoracle.convert(kind, img, w, h, K, True, seed=1, trace=False).scalars["maxbins"]


def test_oracle_maxbins_is_n_for_every_key_scheme(oracle):
    """The oracle's own histogram has exactly n bins, at the largest n of each scheme and two smaller ones (PnnQuantizer,
    whose find_nn is the cheaper; the histogram is the same code in both quantizers)."""
    jobs = [(0, scheme, K, n, tr) for scheme, K, n, tr in HELPER_CASES]
    with ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn")) as ex:
        got = list(ex.map(_oracle_maxbins, jobs))
    assert got == [n for _, _, _, n, _ in jobs]


def test_oracle_rescans_headline_512(oracle):
    """The oracle counts the reference's rescans: 58 016 on the 512x512 headline image, the number the GPU's rescan
    rounds must apply (test_gpu_merge_rounds.py)."""
    from nquant_android_b200.synth import make_image
    img = make_image(512, 512, "noisy", "opaque")
    s = oracle.convert(1, img, 512, 512, 256, True, seed=0xC0FFEE, trace=False).scalars
    assert s["n_rescans"] == 58016
    assert 0 < s["n_heap_pops"] < s["maxbins"] - 256 + 1


# ---------------------------------------------------------------------------------------------------------------------
# GPU: single images at the heap splits of k_merge_lab<4> (5632) and k_merge_rgb (6144)

@pytest.mark.gpu
@pytest.mark.parametrize("case", SPLIT_CASES, ids=[c[0] for c in SPLIT_CASES])
def test_single_image_at_heap_split(gpu_ctx, refs, case):
    name, kind, n, w, h, K, alpha, img_seed, seed = case
    info = _check_single(gpu_ctx, refs[name], kind, n, w, h, K, alpha, img_seed, seed)
    assert abs(info["maxbins"] - HEAP_SPLIT[kind]) <= 1, info["maxbins"]   # the GPU's histogram sits on the split
    if kind == 1:
        assert info["merge_ctas_per_sm"] == LAB4_CTAS        # k_merge_lab<4>, whose split is 5632
    elif K == 256:
        # k_merge_rgb's unpruned redo (err reached U = 4 err32, the reference's break fall-through) runs here: about
        # 2000 redos per image on a B200, so the oracle comparison above covers that path
        assert info["full_evals"] > 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every image of a batch that runs k_merge_lab<8> (heap split 2048), and the same batch in chunks on k_merge_lab<4>

@pytest.mark.gpu
@pytest.mark.parametrize("K", BATCH_KS)
def test_every_image_of_an_eight_per_sm_batch(gpu_ctx, refs, K):
    """4 x SMs + 1 images in one call. With debug on the call is one chunk on k_merge_lab<8>, and every image's merge
    sequence, palette, output, rescans and heap pops are the oracle's. In chunks of SMs images the same batch runs on
    k_merge_lab<4>, and every image's result and counters stay the same."""
    cases = _batch_cases(4 * _sms() + 1)
    n_img, w, h = len(cases), 96, 96
    imgs = np.stack([image_with_bins(n, w, h, scheme_for(K), s) for n, s, _ in cases])
    seeds = [seed for _, _, seed in cases]
    gpu_ctx.set_debug(True)
    try:
        out, pal, plen, _ = gpu_ctx.convert_batch(1, imgs, w, h, K, True, seeds=seeds)
        infos = [gpu_ctx.image_info(i) for i in range(n_img)]
        merges = [gpu_ctx.debug_merges(i) for i in range(n_img)]
    finally:
        gpu_ctx.set_debug(False)
    assert all(info["merge_ctas_per_sm"] >= 7 for info in infos), infos[0]["merge_ctas_per_sm"]   # k_merge_lab<8>
    assert [info["maxbins"] for info in infos] == [c[0] for c in cases]
    assert {c[0] for c in cases} >= {2047, 2048, 2049, 5631, 5632, 5633}
    print(f"\nmerge_ctas_per_sm: {infos[0]['merge_ctas_per_sm']} in one chunk", end="")
    for i in range(n_img):
        r = refs[("batch", K, i)].result()
        assert np.array_equal(merges[i], r.merges), f"image {i} ({cases[i]}): merge sequence differs"
        assert np.array_equal(pal[i, :plen[i]], r.palette) and np.array_equal(out[i], r.out), (i, cases[i])
        assert infos[i]["rescans"] == r.scalars["n_rescans"], (i, cases[i])
        assert infos[i]["heap_pops"] == r.scalars["n_heap_pops"], (i, cases[i])

    sms = _sms()
    gpu_ctx.set_chunk_images(sms)
    try:
        out4, pal4, plen4, _ = gpu_ctx.convert_batch(1, imgs, w, h, K, True, seeds=seeds)
        infos4 = [gpu_ctx.image_info(i) for i in range(n_img)]
    finally:
        gpu_ctx.set_chunk_images(0)
    print(f", {infos4[0]['merge_ctas_per_sm']} in chunks of {sms}", end="")
    assert all(info["merge_ctas_per_sm"] == LAB4_CTAS for info in infos4), infos4[0]["merge_ctas_per_sm"]   # k_merge_lab<4>
    assert np.array_equal(plen4, plen) and np.array_equal(pal4, pal) and np.array_equal(out4, out)
    for key in ("maxbins", "rescans", "merge_rounds", "rescans_discarded", "heap_pops"):
        assert [info[key] for info in infos4] == [info[key] for info in infos], key


# ---------------------------------------------------------------------------------------------------------------------
# GPU: all 65 536 keys occupied (5-6-5), and the largest 4-4-4-4 histogram (61 441 keys, the transparent one included)

@pytest.mark.gpu
@pytest.mark.parametrize("case", FULL_CASES, ids=[c[0] for c in FULL_CASES])
def test_full_histogram(gpu_ctx, refs, case):
    name, kind, n, w, h, K, alpha, img_seed, seed = case
    info = _check_single(gpu_ctx, refs[name], kind, n, w, h, K, alpha, img_seed, seed)
    # every key of the scheme occupied on the GPU: all 65 536 of 5-6-5; all 61 440 of 4-4-4-4 with alpha >= 16 and the
    # transparent colour's
    assert info["maxbins"] == (KEY_SPACE["4444"] + 1 if alpha == "semi" else 65536), info["maxbins"]
