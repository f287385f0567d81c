"""Remap calls (nq_remap_ragged, nq_remap_ragged_device): images dithered to palettes the caller supplies, as convert() would
with its palette replaced, without the merge loop. Checked against the remap oracle (tests/remap_oracle.cpp) on small mixed-size images with
foreign palettes (another image's, web-safe, transparent entries, duplicates, palette lengths on the other side of 32 and 64
from n_max_colors); by the round trip at the benchmarked sizes (remapping an image to the palette its convert produced
returns the frozen oracle output); by every way of making the call; and by what the call launches and rejects."""
import ctypes
import os
import sys
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from nquant_android_b200.imageio import to_indices
from nquant_android_b200.synth import make_image

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import remap_oracle  # noqa: E402
from test_gpu_ragged import BIG, _big_image, sha  # noqa: E402

SMALL = [(1, 1, "noisy", "opaque"), (37, 29, "smooth", "opaque"), (64, 48, "noisy", "opaque"), (50, 61, "rand", "opaque"),
         (63, 65, "smooth", "transparent"), (80, 40, "noisy", "transparent"), (45, 45, "rand", "transparent"),
         (70, 52, "smooth", "semi"), (96, 80, "noisy", "semi"), (33, 90, "rand", "semi"), (96, 80, "few", "opaque")]


def _small_images():
    return [(f"{w}x{h}_{cls}_{a}", make_image(w, h, cls, a, seed=0x5EED0900 + i).reshape(h, w)) for i, (w, h, cls, a) in enumerate(SMALL)]


def _websafe():
    v = [0, 51, 102, 153, 204, 255]
    return np.array([0xFF000000 | r << 16 | g << 8 | b for r in v for g in v for b in v], dtype=np.uint32)


def _palettes():
    from oracle import pyoracle
    other = make_image(64, 48, "rand", "semi", seed=0x5EED0999)
    rng = np.random.default_rng(7)
    p16 = rng.integers(0, 1 << 24, 16).astype(np.uint32) | np.uint32(0xFF000000)
    p16t = p16.copy()
    p16t[5] = 0x00FFFFFF                                        # a fully transparent entry
    dup = np.concatenate([p16[:8], p16[:4], p16[:6] & np.uint32(0x80FFFFFF), p16[6:10] & np.uint32(0x20FFFFFF)])
    p40 = rng.integers(0, 1 << 32, 40, dtype=np.uint64).astype(np.uint32) | np.uint32(0x30000000)
    return {   # name: (palette, n_max_colors)
        "other_image": (pyoracle.convert(0, other, 64, 48, 64, True, seed=1, trace=False).palette, 64),
        "websafe216": (_websafe(), 216),
        "16_transparent": (p16t, 16),
        "duplicates_alpha": (dup, 22),
        "two_colours_k2": (np.array([0xFFFF0000, 0xFF0000FF], np.uint32), 2),
        "16_colours_k64": (p16, 64),
        "40_colours_k16": (p40, 16),
    }


PALETTES = ["other_image", "websafe216", "16_transparent", "duplicates_alpha", "two_colours_k2", "16_colours_k64", "40_colours_k16"]


def _unsupported(kind, name, plen, dither):
    return kind == 1 and not dither and plen > 32 and name.endswith("_semi")


@pytest.mark.parametrize("dither", [True, False], ids=["on", "off"])
@pytest.mark.parametrize("pal_name", PALETTES)
@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_foreign_palettes_match_the_oracle(gpu_ctx, kind, pal_name, dither):
    from nquant_android_b200.quantizer import NQuantError
    pal, K = _palettes()[pal_name]
    items = [(name, img, 300 + i) for i, (name, img) in enumerate(_small_images())]
    if any(_unsupported(kind, n, pal.size, dither) for n, _, _ in items):
        with pytest.raises(NQuantError) as e:   # the branch convert leaves uncovered, keyed on the palette length
            gpu_ctx.remap(kind, [im for _, im, _ in items], pal, dither, n_max_colors=K, seeds=[s for _, _, s in items])
        assert e.value.code == -4
        items = [it for it in items if not _unsupported(kind, it[0], pal.size, dither)]
    imgs, seeds = [im for _, im, _ in items], [s for _, _, s in items]
    outs, idx, ha = gpu_ctx.remap(kind, imgs, pal, dither, n_max_colors=K, seeds=seeds, with_indices=True)
    for i, (name, img, seed) in enumerate(items):
        ref = remap_oracle.remap(kind, img.reshape(-1), img.shape[1], img.shape[0], K, dither, pal, seed=seed)
        info = gpu_ctx.image_info(i)
        assert np.array_equal(outs[i].reshape(-1), ref.out), name
        assert np.array_equal(idx[i], to_indices(outs[i], pal).reshape(img.shape)), name
        assert info["rng_draws"] == ref.scalars["rng_draws"], name
        assert info["merges"] == 0 and info["palette_len"] == pal.size, name
        assert ha[i] == (ref.scalars["transparentPixelIndex"] >= 0), name


# the cases test_gpu_golden_big.py leaves opt-in (NQ_BIG_GOLDEN=all): minutes of GPU time on the serial dither chain each
from test_gpu_golden_big import SLOW  # noqa: E402
ROUND_TRIP = [c for c in BIG.values() if c.get("palette") and (c["name"] not in SLOW or os.environ.get("NQ_BIG_GOLDEN") == "all")]
_SYNTH = threading.Lock()   # one 8192x8192 synthetic image at a time: its generator holds a few GB of intermediates


def _round_trip(c):
    from nquant_android_b200.quantizer import Context
    with _SYNTH:
        img = _big_image(c)
    ctx = Context(0)
    try:
        outs, _, _ = ctx.remap(c["kind"], [img], np.array(c["palette"], np.uint32), bool(c["dither"]), n_max_colors=c["k"], seeds=[c["seed"]])
        info = ctx.image_info(0)
        return sha(outs[0]), info["rng_draws"], info["merges"], ctx.stage_times()
    finally:
        ctx.close()


def test_round_trip_at_the_benchmarked_sizes():
    """Every frozen case with a palette (4K CIELAB images on the speculative path, the semi-transparent 4K RGB case, the
    8192x8192 images; with NQ_BIG_GOLDEN=all also the 8192x8192 BlueNoise passes of both kinds and the K = 2 fixed palettes),
    remapped to the palette its convert produced with its k, dither and seed: the frozen output and draw count, no merge.
    The serial dither chains of the 8192x8192 images take tens of seconds or more each, so the cases run side by side, one
    context each."""
    assert "q3_8192_lab_256_on" not in {c["name"] for c in ROUND_TRIP}
    with ThreadPoolExecutor(max_workers=8) as ex:
        results = list(ex.map(_round_trip, ROUND_TRIP))
    bad = []
    for c, (digest, draws, merges, st) in zip(ROUND_TRIP, results):
        if digest != c["output_sha"] or draws != c["rng_draws"] or merges != 0 or st["merge"][1] or st["find_nn_sweep"][1]:
            bad.append((c["name"], digest == c["output_sha"], draws, c["rng_draws"], merges))
    assert not bad, bad


def _mixed():
    return [make_image(w, h, cls, "opaque", seed=0x5EED0A00 + i).reshape(h, w)
            for i, (w, h, cls) in enumerate([(512, 512, "noisy"), (640, 480, "noisy"), (300, 700, "noisy"), (512, 512, "smooth"),
                                             (256, 256, "rand"), (1, 1, "noisy"), (777, 3, "noisy")])]


@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_same_result_whichever_way_the_call_is_made(gpu_ctx, kind):
    import torch
    imgs = _mixed()
    n = len(imgs)
    seeds = [700 + i for i in range(n)]
    donor = make_image(512, 512, "noisy", "opaque", seed=0x5EED0AFF)
    _, dpal, dplen, _ = gpu_ctx.convert_batch(kind, donor[None, :], 512, 512, 256, True)
    pal = dpal[0, :dplen[0]].copy()                  # another image's palette: 256 colours, the speculative dither's case
    spec0 = gpu_ctx.spec_stats()
    outs, idx, ha = gpu_ctx.remap(kind, imgs, pal, True, seeds=seeds, with_indices=True)
    spec1 = gpu_ctx.spec_stats()
    if kind == 1:   # images the speculative path took, finished or handed back, are counted there
        assert spec1["images"] - spec0["images"] + spec1["fallbacks"] - spec0["fallbacks"] > 0
    infos = [gpu_ctx.image_info(i)["rng_draws"] for i in range(n)]
    for i in range(n):
        assert np.array_equal(idx[i], to_indices(outs[i], pal).reshape(imgs[i].shape)), i
        assert pal[idx[i]].tolist() == outs[i].tolist(), i

    def same(o, x, what):
        for i in range(n):
            if o is not None:
                assert np.array_equal(o[i].reshape(imgs[i].shape), outs[i]), (what, i)
            if x is not None:
                assert np.array_equal(x[i].reshape(imgs[i].shape), idx[i]), (what, i)
        assert [gpu_ctx.image_info(i)["rng_draws"] for i in range(n)] == infos, what

    o, x, a = gpu_ctx.remap(kind, imgs, [pal] * n, True, seeds=seeds, with_indices=True)
    same(o, x, "one palette per image")
    assert np.array_equal(a, ha)
    o, x, _ = gpu_ctx.remap(kind, imgs, pal, True, seeds=seeds, with_argb=False, with_indices=True)
    assert o is None
    same(o, x, "indices only")
    o, x, _ = gpu_ctx.remap(kind, imgs, pal, True, seeds=seeds)
    assert x is None
    same(o, x, "colours only")
    d_in = torch.cat([torch.from_numpy(im.reshape(-1).view(np.int32)) for im in imgs]).cuda()
    offs = np.cumsum([0] + [im.size for im in imgs])
    ws, hs = [im.shape[1] for im in imgs], [im.shape[0] for im in imgs]
    for with_out, with_idx in ((True, True), (False, True), (True, False)):
        d_out = torch.empty_like(d_in) if with_out else None
        d_idx = torch.full((d_in.numel(),), 0xAB, dtype=torch.uint8, device="cuda") if with_idx else None
        dha = np.zeros(n, np.int32)
        gpu_ctx.remap_ptr(kind, d_in.data_ptr(), ws, hs, pal, True, seeds=seeds, out_ptr=d_out.data_ptr() if with_out else None,
                          index_ptr=d_idx.data_ptr() if with_idx else None, has_alpha=dha)
        fo = d_out.cpu().numpy().view(np.uint32) if with_out else None
        fx = d_idx.cpu().numpy() if with_idx else None
        same(None if fo is None else [fo[offs[i]:offs[i + 1]] for i in range(n)],
             None if fx is None else [fx[offs[i]:offs[i + 1]] for i in range(n)], f"device, colours {with_out}, indices {with_idx}")
        assert np.array_equal(dha, ha)
    gpu_ctx.set_chunk_images(1)
    try:
        o, x, _ = gpu_ctx.remap(kind, imgs, pal, True, seeds=seeds, with_indices=True)
        same(o, x, "chunks of one image")
    finally:
        gpu_ctx.set_chunk_images(0)
    gpu_ctx.set_spec_dither(False)
    try:
        o, x, _ = gpu_ctx.remap(kind, imgs, pal, True, seeds=seeds, with_indices=True)
        same(o, x, "speculative dither off")
    finally:
        gpu_ctx.set_spec_dither(True, 0, 1024)
    for i in range(n):   # one call per image
        o, x, _ = gpu_ctx.remap(kind, imgs[i:i + 1], pal, True, seeds=seeds[i:i + 1], with_indices=True)
        assert np.array_equal(o[0], outs[i]) and np.array_equal(x[0], idx[i]), ("alone", i)
        assert gpu_ctx.image_info(0)["rng_draws"] == infos[i], ("alone", i)


@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_remap_skips_the_find_nn_sweep_and_the_merge_loop(gpu_ctx, kind):
    imgs = [make_image(256, 256, "noisy", "opaque", seed=0x5EED0B00 + i).reshape(256, 256) for i in range(4)]
    outs, pal, plen, _ = gpu_ctx.convert_ragged(kind, imgs, 256, True, seeds=[1, 2, 3, 4])
    gpu_ctx.stage_times(reset=True)
    l0 = gpu_ctx.kernel_launches()
    gpu_ctx.convert_ragged(kind, imgs, 256, True, seeds=[1, 2, 3, 4])
    l1 = gpu_ctx.kernel_launches()
    conv = gpu_ctx.stage_times(reset=True)
    assert conv["merge"][1] > 0 and conv["find_nn_sweep"][1] > 0
    got, _, _ = gpu_ctx.remap(kind, imgs, [pal[i, :plen[i]] for i in range(4)], True, n_max_colors=256, seeds=[1, 2, 3, 4])
    l2 = gpu_ctx.kernel_launches()
    st = gpu_ctx.stage_times(reset=True)
    assert st["merge"][1] == 0 and st["find_nn_sweep"][1] == 0, st
    assert st["histogram"][1] > 0 and st["dither"][1] > 0, st
    if kind == 1:   # no radix passes or bin sums either
        assert l2 - l1 < l1 - l0, (l2 - l1, l1 - l0)
    assert all(np.array_equal(got[i], outs[i]) for i in range(4))


def test_argument_errors(gpu_ctx):
    from nquant_android_b200.quantizer import NQuantError
    L = gpu_ctx._L
    imgs = [make_image(8, 8, seed=1).reshape(8, 8), make_image(16, 4, seed=2).reshape(4, 16)]
    outs = [np.empty_like(im) for im in imgs]
    ins_p = (ctypes.c_void_p * 2)(*[im.ctypes.data for im in imgs])
    out_p = (ctypes.c_void_p * 2)(*[o.ctypes.data for o in outs])
    w, h = np.array([8, 16], np.int32), np.array([8, 4], np.int32)
    pal = np.zeros((2, 256), np.uint32)
    pal[:, 1] = 0xFFFFFFFF
    pal[:, 0] = 0xFF000000

    def host(pp=pal.ctypes.data, lens=(2, 2), npal=1, op=out_p, ip=None):
        ln = np.array(lens, np.int32)
        return L.nq_remap_ragged(gpu_ctx._h, 0, ins_p, w.ctypes.data, h.ctypes.data, 2, 16, pp, ln.ctypes.data, npal, 1, None, op, ip, None)

    assert host(pp=None) == -2                      # null palette
    assert host(npal=3, lens=(2, 2, 2)) == -2       # n_palettes neither 1 nor n_images
    assert host(npal=0) == -2
    assert host(lens=(0,)) == -2                    # palette length 0
    assert host(lens=(257,)) == -2                  # palette length 257
    assert host(npal=2, lens=(2, 257)) == -2
    assert host(op=None) == -2                      # neither colours nor indices
    assert L.nq_remap_ragged_device(gpu_ctx._h, 0, None, w.ctypes.data, h.ctypes.data, 2, 16, pal.ctypes.data,
                                    np.array([2], np.int32).ctypes.data, 1, 1, None, None, None, None) == -2
    assert host() == 0 and host(npal=2, lens=(2, 1)) == 0
    assert set(np.unique(outs[1])) <= {0xFF000000}
    # PnnLABQuantizer, dither off, semi-transparent pixels, a palette of more than 32 entries: as convert
    semi = make_image(64, 48, "noisy", "semi", seed=3).reshape(48, 64)
    with pytest.raises(NQuantError) as e:
        gpu_ctx.remap(1, [semi], _websafe()[:33], False, n_max_colors=16)
    assert e.value.code == -4
    o, _, _ = gpu_ctx.remap(1, [semi], _websafe()[:32], False, n_max_colors=64)   # keyed on the palette length
    assert np.isin(o[0], _websafe()[:32]).all()
