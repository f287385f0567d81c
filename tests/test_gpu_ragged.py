"""Mixed-size calls (nq_convert_ragged, nq_convert_ragged_device, nq_convert_ragged_multi): every image of one call must get
exactly what it gets alone -- against the oracle's frozen outputs at the benchmarked sizes, against the oracle itself on
small and degenerate sizes, and against the equal-size entry points and every other way of cutting the same call."""
import ctypes
import hashlib
import json
import multiprocessing
import os
import sys
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

from nquant_android_b200.synth import make_image

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "tools"))
BIG = {c["name"]: c for c in json.load(open(os.path.join(HERE, "golden", "oracle_big_cases.json")))}
COUNTERS = ("maxbins", "merges", "rescans", "heap_pops", "rng_draws", "palette_len", "error")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).astype("<u4").tobytes()).hexdigest()


def _big_image(c):
    import make_golden_big
    img = make_golden_big.build_image(c)
    assert sha(img) == c["input_sha"]
    return img.reshape(c["h"], c["w"])


@pytest.mark.parametrize("kind,names", [
    (1, ["config1_1080p_lab_noisy", "config3_4k_lab_img0", "config3_4k_lab_img591", "config3_4k_lab_img1023", "config4_8192_lab_256_on"]),
    (0, ["config0_512_noisy", "config0_512_smooth", "config0_512_rand", "config4_8192_rgb_256_on", "q3_8192_rgb_256_on"]),
], ids=["lab", "rgb"])
def test_benchmarked_sizes_in_one_call_match_frozen_oracle_output(kind, names):
    from nquant_android_b200.quantizer import Context
    cases = [BIG[n] for n in names]
    assert all(c["kind"] == kind and c["k"] == 256 and c["dither"] == 1 for c in cases)
    ctx = Context(0)
    try:
        before = ctx.spec_stats()["images"]
        outs, pal, plen, _ = ctx.convert_ragged(kind, [_big_image(c) for c in cases], 256, True, seeds=[c["seed"] for c in cases])
        for i, c in enumerate(cases):
            info = ctx.image_info(i)
            assert [int(v) for v in pal[i, :plen[i]]] == c["palette"], c["name"]
            assert sha(outs[i]) == c["output_sha"], c["name"]
            assert info["maxbins"] == c["maxbins"] and info["rng_draws"] == c["rng_draws"], c["name"]
        if kind == 1:   # the 1080p, 4K and 8192x8192 images share the speculative pool instead of the serial kernel
            assert ctx.spec_stats()["images"] - before == len(cases)
    finally:
        ctx.close()


def _sample():
    from nquant_android_b200.imageio import load_argb
    argb, w, h = load_argb(os.path.join(HERE, "golden", "sample_495x438.png"))
    return argb.reshape(h, w)


def _small_images():
    imgs = []
    for i, (w, h, cls, alpha) in enumerate([(1, 1, "noisy", "opaque"), (1, 777, "noisy", "opaque"), (777, 1, "rand", "opaque"),
                                            (2, 3, "rand", "opaque"), (63, 65, "noisy", "transparent"), (96, 80, "few", "opaque"),
                                            (256, 256, "smooth", "opaque"), (640, 480, "noisy", "transparent"),
                                            (640, 480, "noisy", "semi")]):
        imgs.append((f"{w}x{h}_{cls}_{alpha}", make_image(w, h, cls, alpha, seed=0x5EED0000 + i).reshape(h, w)))
    imgs.insert(6, ("sample_495x438", _sample()))
    return imgs


SMALL_SETTINGS = [(256, True), (16, True), (64, False), (2, True)]


def _oracle_job(kind, img, K, dither, seed):
    from oracle import pyoracle
    r = pyoracle.convert(kind, img.reshape(-1), img.shape[1], img.shape[0], K, dither, seed=seed)
    del r.saliencies, r.gweights, r.bins, r.init_err, r.init_nn
    return r


def _semi_lab_unsupported(kind, name, K, dither):
    return kind == 1 and not dither and K > 32 and name.endswith("_semi")


@pytest.fixture(scope="module")
def small_refs(oracle):
    """The oracle's result of every small image at every setting, computed in a pool of host processes while the GPU runs."""
    ex = ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn"))
    futs = {}
    for kind in (0, 1):
        for K, dither in SMALL_SETTINGS:
            for i, (name, img) in enumerate(_small_images()):
                if not _semi_lab_unsupported(kind, name, K, dither):
                    futs[(kind, K, dither, name)] = ex.submit(_oracle_job, kind, img, K, dither, 1000 + i)
    yield futs
    ex.shutdown(cancel_futures=True)


@pytest.mark.parametrize("K,dither", SMALL_SETTINGS, ids=[f"k{K}_{'on' if d else 'off'}" for K, d in SMALL_SETTINGS])
@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_small_mixed_sizes_match_the_oracle(gpu_ctx, small_refs, kind, K, dither):
    from nquant_android_b200.quantizer import NQuantError
    items = [(name, img, 1000 + i) for i, (name, img) in enumerate(_small_images())]
    if any(_semi_lab_unsupported(kind, n, K, dither) for n, _, _ in items):
        with pytest.raises(NQuantError) as e:   # the branch the batch calls leave uncovered too (test_error_codes)
            gpu_ctx.convert_ragged(kind, [im for _, im, _ in items], K, dither, seeds=[s for _, _, s in items])
        assert e.value.code == -4
        items = [it for it in items if not _semi_lab_unsupported(kind, it[0], K, dither)]
    gpu_ctx.set_debug(True)
    try:
        outs, pal, plen, ha = gpu_ctx.convert_ragged(kind, [im for _, im, _ in items], K, dither, seeds=[s for _, _, s in items])
        merges = [gpu_ctx.debug_merges(i) for i in range(len(items))]
    finally:
        gpu_ctx.set_debug(False)
    for i, (name, img, _) in enumerate(items):
        ref = small_refs[(kind, K, dither, name)].result()
        assert np.array_equal(pal[i, :plen[i]], ref.palette), name
        assert np.array_equal(outs[i].reshape(-1), ref.out), name
        assert bool(ha[i]) == (ref.scalars["transparentPixelIndex"] > -1), name
        assert gpu_ctx.image_info(i)["rng_draws"] == ref.scalars["rng_draws"], name
        assert np.array_equal(merges[i], ref.merges), name


def _infos(ctx, n):
    return [{k: ctx.image_info(i)[k] for k in COUNTERS} for i in range(n)]


@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_equal_sizes_through_the_ragged_entry_match_the_batch_entry(gpu_ctx, kind):
    w, h, n = 320, 240, 6
    imgs = np.stack([make_image(w, h, "noisy" if i % 2 else "rand", "opaque", seed=0x5EED0100 + i) for i in range(n)])
    seeds = [77 + i for i in range(n)]
    out, pal, plen, ha = gpu_ctx.convert_batch(kind, imgs, w, h, 256, True, seeds=seeds)
    want = _infos(gpu_ctx, n)
    routs, rpal, rplen, rha = gpu_ctx.convert_ragged(kind, [im.reshape(h, w) for im in imgs], 256, True, seeds=seeds)
    assert _infos(gpu_ctx, n) == want
    assert np.array_equal(np.stack([o.reshape(-1) for o in routs]), out)
    assert np.array_equal(rpal, pal) and np.array_equal(rplen, plen) and np.array_equal(rha, ha)


def _mixed_ten():
    sizes = [(640, 480), (495, 438), (1280, 720), (33, 17), (640, 480), (1080, 1920), (256, 256), (1920, 1080), (97, 1), (800, 600)]
    return [make_image(w, h, "noisy", "opaque" if i != 3 else "transparent", seed=0x5EED0200 + i).reshape(h, w)
            for i, (w, h) in enumerate(sizes)]


def test_same_results_whichever_way_the_call_is_cut(gpu_ctx):
    import torch
    from nquant_android_b200.quantizer import Context, convert_ragged_multi
    imgs = _mixed_ten()
    n = len(imgs)
    seeds = [500 + i for i in range(n)]
    outs, pal, plen, ha = gpu_ctx.convert_ragged(1, imgs, 256, True, seeds=seeds)
    want = _infos(gpu_ctx, n)
    spec = gpu_ctx.spec_stats()["images"]

    def same(o, p, pl, a, infos=None, what=""):
        for i in range(n):
            assert np.array_equal(o[i], outs[i]), (what, i)
        assert np.array_equal(p, pal) and np.array_equal(pl, plen) and np.array_equal(a, ha), what
        if infos is not None:
            assert infos == want, what

    # every image alone
    for i, im in enumerate(imgs):
        o, p, pl, a = gpu_ctx.convert_batch(1, im.reshape(1, -1), im.shape[1], im.shape[0], 256, True, seeds=[seeds[i]])
        assert np.array_equal(o[0], outs[i].reshape(-1)) and np.array_equal(p[0], pal[i]), i
        assert _infos(gpu_ctx, 1)[0] == want[i], i
    # device buffers, packed back to back
    d_in = torch.cat([torch.from_numpy(im.reshape(-1).view(np.int32)) for im in imgs]).cuda()
    d_out = torch.empty_like(d_in)
    p, pl, a = np.zeros((n, 256), np.uint32), np.zeros(n, np.int32), np.zeros(n, np.int32)
    gpu_ctx.convert_ragged_ptr(1, d_in.data_ptr(), d_out.data_ptr(), [im.shape[1] for im in imgs], [im.shape[0] for im in imgs], 256, True,
                               seeds=seeds, palettes=p, palette_lens=pl, has_alpha=a)
    flat = d_out.cpu().numpy().view(np.uint32)
    offs = np.cumsum([0] + [im.size for im in imgs])
    same([flat[offs[i]:offs[i + 1]].reshape(imgs[i].shape) for i in range(n)], p, pl, a, _infos(gpu_ctx, n), "device")
    # chunks of three images
    gpu_ctx.set_chunk_images(3)
    try:
        o, p, pl, a = gpu_ctx.convert_ragged(1, imgs, 256, True, seeds=seeds)
        same(o, p, pl, a, _infos(gpu_ctx, n), "chunks of 3")
    finally:
        gpu_ctx.set_chunk_images(0)
    assert gpu_ctx.spec_stats()["images"] > spec
    # three contexts on device 0, dynamic queue
    ctxs = [Context(0) for _ in range(3)]
    try:
        for q in (0, 1, 3):
            o, p, pl, a = convert_ragged_multi(ctxs, 1, imgs, 256, True, seeds=seeds, queue_images=q)
            same(o, p, pl, a, what=f"multi queue {q}")
    finally:
        for c in ctxs:
            c.close()


def test_argument_errors_leave_the_context_usable(gpu_ctx):
    L = gpu_ctx._L
    imgs = [make_image(8, 8, seed=1).reshape(8, 8), make_image(16, 4, seed=2).reshape(4, 16)]
    outs = [np.empty_like(im) for im in imgs]
    ins_p = (ctypes.c_void_p * 2)(*[im.ctypes.data for im in imgs])
    outs_p = (ctypes.c_void_p * 2)(*[o.ctypes.data for o in outs])

    def call(ws, hs, ip=ins_p):
        w = np.array(ws, np.int32)
        h = np.array(hs, np.int32)
        return L.nq_convert_ragged(gpu_ctx._h, 0, ip, w.ctypes.data, h.ctypes.data, 2, 16, 1, None, outs_p, None, None, None)

    assert call([8, 0], [8, 4]) == -2                 # a zero width
    assert call([8, 70000], [8, 1]) == -2             # a side the order tables cannot hold
    assert call([8, 16], [8, 4], (ctypes.c_void_p * 2)(imgs[0].ctypes.data, None)) == -2   # a null image pointer
    assert L.nq_convert_ragged(gpu_ctx._h, 0, ins_p, None, None, 2, 16, 1, None, outs_p, None, None, None) == -2
    assert call([8, 16], [8, 4]) == 0
    for i, im in enumerate(imgs):
        o, _, _, _ = gpu_ctx.convert_batch(0, im.reshape(1, -1), im.shape[1], im.shape[0], 16, True)
        assert np.array_equal(o[0], outs[i].reshape(-1))
