"""Index-map calls (nq_convert_ragged_indexed, nq_convert_ragged_indexed_device): the palette index of every output pixel,
computed on the GPU by k_index_map. The indices must be imageio.to_indices of the same call's ARGB output, with the palettes
and counters of nq_convert_ragged; palette[index] must reproduce the oracle's frozen outputs; and every way of making the
call -- host or device buffers, with or without the colours, in chunks, with the speculative dither on or off, with the
progressive copy-out of a large CIELAB host call -- must give the same indices."""
import ctypes
import os
import sys

import numpy as np
import pytest

from nquant_android_b200.imageio import to_indices
from nquant_android_b200.synth import make_image

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_ragged import BIG, SMALL_SETTINGS, _big_image, _mixed_ten, _semi_lab_unsupported, _small_images, sha  # noqa: E402

COUNTERS = ("maxbins", "merges", "rescans", "heap_pops", "rng_draws", "palette_len", "error")


def _infos(ctx, n):
    return [{k: ctx.image_info(i)[k] for k in COUNTERS} for i in range(n)]


def _expected(outs, pal, plen):
    return [to_indices(o, pal[i, :plen[i]]).reshape(o.shape) for i, o in enumerate(outs)]


@pytest.mark.parametrize("K,dither", SMALL_SETTINGS, ids=[f"k{K}_{'on' if d else 'off'}" for K, d in SMALL_SETTINGS])
@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_small_mixed_sizes_match_to_indices_of_the_ragged_call(gpu_ctx, kind, K, dither):
    from nquant_android_b200.quantizer import NQuantError
    items = [(name, img, 1000 + i) for i, (name, img) in enumerate(_small_images())]
    if any(_semi_lab_unsupported(kind, n, K, dither) for n, _, _ in items):
        with pytest.raises(NQuantError) as e:   # the branch nq_convert_ragged leaves uncovered: the same error here
            gpu_ctx.convert_indexed(kind, [im for _, im, _ in items], K, dither, seeds=[s for _, _, s in items])
        assert e.value.code == -4
        items = [it for it in items if not _semi_lab_unsupported(kind, it[0], K, dither)]
    imgs, seeds = [im for _, im, _ in items], [s for _, _, s in items]
    outs, pal, plen, ha = gpu_ctx.convert_ragged(kind, imgs, K, dither, seeds=seeds)
    want = _infos(gpu_ctx, len(items))
    idx, argb, ipal, iplen, iha = gpu_ctx.convert_indexed(kind, imgs, K, dither, seeds=seeds, with_argb=True)
    assert _infos(gpu_ctx, len(items)) == want
    assert np.array_equal(ipal, pal) and np.array_equal(iplen, plen) and np.array_equal(iha, ha)
    for i, (name, _, _) in enumerate(items):
        assert idx[i].dtype == np.uint8 and idx[i].shape == outs[i].shape, name
        assert np.array_equal(idx[i], _expected(outs, pal, plen)[i]), name
        assert np.array_equal(argb[i], outs[i]), name


FROZEN = [
    ("lab_256_on", ["config1_1080p_lab_noisy", "config3_4k_lab_img0"]),
    ("rgb_256_on", ["config0_512_noisy", "config0_512_smooth", "config0_512_rand", "q3_8192_rgb_256_on"]),
    ("rgb_16_on_semi", ["config2_4k_rgb16_semi"]),
    ("rgb_256_off", ["config4_8192_rgb_256_off"]),   # BlueNoise second pass on the aux stream (k_bn_rgb_*)
]


@pytest.mark.parametrize("names", [n for _, n in FROZEN], ids=[g for g, _ in FROZEN])
def test_palette_at_index_is_the_frozen_oracle_output(gpu_ctx, names):
    import torch
    cases = [BIG[n] for n in names]
    kind, K, dither = cases[0]["kind"], cases[0]["k"], cases[0]["dither"]
    assert all((c["kind"], c["k"], c["dither"]) == (kind, K, dither) for c in cases)
    imgs, seeds = [_big_image(c) for c in cases], [c["seed"] for c in cases]

    def check(idx, pal, plen, what):
        for i, c in enumerate(cases):
            p = pal[i, :plen[i]]
            assert [int(v) for v in p] == c["palette"], (what, c["name"])
            assert sha(p[idx[i].reshape(-1)]) == c["output_sha"], (what, c["name"])

    idx, argb, pal, plen, _ = gpu_ctx.convert_indexed(kind, imgs, K, bool(dither), seeds=seeds)
    assert argb is None
    check(idx, pal, plen, "host")
    if K == 256 and dither:   # the device entry, the colours left in the context's scratch
        d_in = torch.cat([torch.from_numpy(im.reshape(-1).view(np.int32)) for im in imgs]).cuda()
        d_idx = torch.empty(d_in.numel(), dtype=torch.uint8, device="cuda")
        pal, plen = np.zeros((len(cases), 256), np.uint32), np.zeros(len(cases), np.int32)
        gpu_ctx.convert_indexed_ptr(kind, d_in.data_ptr(), d_idx.data_ptr(), [im.shape[1] for im in imgs], [im.shape[0] for im in imgs],
                                    K, True, seeds=seeds, palettes=pal, palette_lens=plen)
        flat = d_idx.cpu().numpy()
        offs = np.cumsum([0] + [im.size for im in imgs])
        check([flat[offs[i]:offs[i + 1]] for i in range(len(cases))], pal, plen, "device")


@pytest.mark.parametrize("kind", [0, 1], ids=["rgb", "lab"])
def test_same_indices_whichever_way_the_call_is_made(gpu_ctx, kind):
    import torch
    imgs = _mixed_ten()
    n = len(imgs)
    seeds = [500 + i for i in range(n)]
    outs, pal, plen, ha = gpu_ctx.convert_ragged(kind, imgs, 256, True, seeds=seeds)
    want = _expected(outs, pal, plen)
    infos = _infos(gpu_ctx, n)

    def same(idx, p, pl, what):
        for i in range(n):
            assert np.array_equal(idx[i].reshape(imgs[i].shape), want[i]), (what, i)
        assert np.array_equal(p, pal) and np.array_equal(pl, plen), what
        assert _infos(gpu_ctx, n) == infos, what

    idx, argb, p, pl, a = gpu_ctx.convert_indexed(kind, imgs, 256, True, seeds=seeds, with_argb=True)
    same(idx, p, pl, "host, with colours")
    assert all(np.array_equal(argb[i], outs[i]) for i in range(n)) and np.array_equal(a, ha)
    idx, argb, p, pl, _ = gpu_ctx.convert_indexed(kind, imgs, 256, True, seeds=seeds)
    same(idx, p, pl, "host, indices only")
    # device buffers, packed back to back, with and without the colours
    d_in = torch.cat([torch.from_numpy(im.reshape(-1).view(np.int32)) for im in imgs]).cuda()
    offs = np.cumsum([0] + [im.size for im in imgs])
    ws, hs = [im.shape[1] for im in imgs], [im.shape[0] for im in imgs]
    for with_out in (True, False):
        d_idx = torch.full((d_in.numel(),), 0xAB, dtype=torch.uint8, device="cuda")
        d_out = torch.empty_like(d_in) if with_out else None
        p, pl = np.zeros((n, 256), np.uint32), np.zeros(n, np.int32)
        gpu_ctx.convert_indexed_ptr(kind, d_in.data_ptr(), d_idx.data_ptr(), ws, hs, 256, True, seeds=seeds,
                                    out_ptr=d_out.data_ptr() if with_out else None, palettes=p, palette_lens=pl)
        flat = d_idx.cpu().numpy()
        same([flat[offs[i]:offs[i + 1]] for i in range(n)], p, pl, f"device, colours {with_out}")
        if with_out:
            o = d_out.cpu().numpy().view(np.uint32)
            assert all(np.array_equal(o[offs[i]:offs[i + 1]].reshape(imgs[i].shape), outs[i]) for i in range(n))
    # chunks of three images
    gpu_ctx.set_chunk_images(3)
    try:
        idx, _, p, pl, _ = gpu_ctx.convert_indexed(kind, imgs, 256, True, seeds=seeds)
        same(idx, p, pl, "chunks of 3")
    finally:
        gpu_ctx.set_chunk_images(0)
    # every image to the serial dither kernels
    gpu_ctx.set_spec_dither(False)
    try:
        idx, _, p, pl, _ = gpu_ctx.convert_indexed(kind, imgs, 256, True, seeds=seeds)
        same(idx, p, pl, "speculative dither off")
    finally:
        gpu_ctx.set_spec_dither(True, 0, 1024)


def test_progressive_copy_out_of_a_large_lab_host_call(gpu_ctx):
    """64 noisy 512x512 CIELAB images from host buffers: two chunks of 32, every image on the speculative dither, which hands
    each complete prefix of 16 images or more to the copy-out (SpecCudaBackend::done_prefix) -- at the latest the whole
    chunk once its last image is done. The indices of such a prefix are computed inside that hand-over, before the copy is
    enqueued, so at least one k_index_map launch per chunk."""
    w, h, n = 512, 512, 64
    imgs = [make_image(w, h, "noisy", "opaque", seed=0x5EED0300 + i).reshape(h, w) for i in range(n)]
    seeds = [900 + i for i in range(n)]
    gpu_ctx.convert_ragged(1, imgs[:1], 256, True, seeds=seeds[:1])   # the size's visiting order, built once
    spec = gpu_ctx.spec_stats()["images"]
    l0 = gpu_ctx.kernel_launches()
    outs, pal, plen, ha = gpu_ctx.convert_ragged(1, imgs, 256, True, seeds=seeds)
    l1 = gpu_ctx.kernel_launches()
    assert gpu_ctx.spec_stats()["images"] - spec == n
    want = _expected(outs, pal, plen)
    infos = _infos(gpu_ctx, n)
    for with_argb in (False, True):
        l2 = gpu_ctx.kernel_launches()
        idx, argb, p, pl, a = gpu_ctx.convert_indexed(1, imgs, 256, True, seeds=seeds, with_argb=with_argb)
        extra = gpu_ctx.kernel_launches() - l2 - (l1 - l0)
        assert extra >= 2, f"{extra} k_index_map launches for two chunks"
        assert all(np.array_equal(idx[i], want[i]) for i in range(n)), with_argb
        assert np.array_equal(p, pal) and np.array_equal(pl, plen) and np.array_equal(a, ha)
        assert _infos(gpu_ctx, n) == infos
        if with_argb:
            assert all(np.array_equal(argb[i], outs[i]) for i in range(n))


def test_argument_errors_leave_the_context_usable(gpu_ctx):
    import torch
    L = gpu_ctx._L
    imgs = [make_image(8, 8, seed=1).reshape(8, 8), make_image(16, 4, seed=2).reshape(4, 16)]
    idx = [np.empty(im.shape, np.uint8) for im in imgs]
    ins_p = (ctypes.c_void_p * 2)(*[im.ctypes.data for im in imgs])
    idx_p = (ctypes.c_void_p * 2)(*[a.ctypes.data for a in idx])
    w, h = np.array([8, 16], np.int32), np.array([8, 4], np.int32)

    def host(ip=ins_p, xp=idx_p, ws=w, nmax=16):
        return L.nq_convert_ragged_indexed(gpu_ctx._h, 0, ip, ws.ctypes.data, h.ctypes.data, 2, nmax, 1, None, xp, None, None, None, None)

    assert host(xp=None) == -2                                                   # no index array
    assert host(xp=(ctypes.c_void_p * 2)(idx[0].ctypes.data, None)) == -2        # a null index buffer
    assert host(ip=(ctypes.c_void_p * 2)(imgs[0].ctypes.data, None)) == -2      # a null image pointer
    assert host(ws=np.array([8, 0], np.int32)) == -2                             # a zero width
    assert host(nmax=1) == -2
    d_in = torch.zeros(8 * 8 + 16 * 4 + 8, dtype=torch.int32, device="cuda")
    d_idx = torch.zeros(256, dtype=torch.uint8, device="cuda")

    def dev(ip, xp, op=None):
        return L.nq_convert_ragged_indexed_device(gpu_ctx._h, 0, ctypes.c_void_p(ip), w.ctypes.data, h.ctypes.data, 2, 16, 1, None,
                                                  ctypes.c_void_p(xp) if xp else None, ctypes.c_void_p(op) if op else None, None, None, None)

    assert dev(d_in.data_ptr(), None) == -2                                      # no index plane
    assert dev(d_in.data_ptr(), d_idx.data_ptr() + 3) == -2                      # index plane not 16-byte aligned
    assert dev(d_in.data_ptr() + 4, d_idx.data_ptr()) == -2                      # input not 16-byte aligned
    assert dev(d_in.data_ptr(), d_idx.data_ptr(), d_in.data_ptr() + 8) == -2     # output not 16-byte aligned
    assert host() == 0
    for i, im in enumerate(imgs):
        o, pal, plen, _ = gpu_ctx.convert_batch(0, im.reshape(1, -1), im.shape[1], im.shape[0], 16, True)
        assert np.array_equal(pal[0, :plen[0]][idx[i].reshape(-1)], o[0])
