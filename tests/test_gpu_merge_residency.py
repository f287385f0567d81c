"""k_merge_lab has two instances: k_merge_lab<4> (128 registers, 5632 heap slots in shared memory) and k_merge_lab<8>
(64 registers, 2048 heap slots, eight CTAs per SM). The host launches <8> when more merge loops run at once than <4> holds
in one wave, so a 1024-image batch runs all its merge loops in one wave on 148 SMs. Below the shared slots the heap sits
in global memory (three levels for a 128x128 noisy image at <8>, four for a 4K one); the merge sequence must stay the
reference's, bin for bin, in both instances."""
import hashlib
import json
import os

import numpy as np
import pytest

from nquant_android_b200.synth import make_image

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
# the oracle's merge sequence of BASELINE.json configs[3] image 0 (31 148 merges, (tb, nb) int32 pairs in merge order):
# the oracle needs a minute for it, so only its SHA-256 travels
MERGES_4K_IMG0_SHA = "a793b57fdda3c5cc381f553efbc5486660a03bbe874a43637f6f5cfb45e02fec"


def _sha(a, dtype):
    return hashlib.sha256(np.ascontiguousarray(a).astype(dtype).tobytes()).hexdigest()


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_batch_beyond_one_wave_of_four_per_sm_runs_eight_per_sm(gpu_ctx, oracle):
    """4 x SMs + 1 images of 128x128 (11 216 bins): k_merge_lab<8>, against the oracle and against the same image alone,
    which runs on k_merge_lab<4>."""
    w = h = 128
    n = 4 * _sms() + 1
    imgs = np.stack([make_image(w, h, "noisy", "opaque", seed=3 + i) for i in range(n)])
    seeds = [3 + i for i in range(n)]
    gpu_ctx.set_debug(True)
    try:
        out, pal, plen, _ = gpu_ctx.convert_batch(1, imgs, w, h, 256, True, seeds=seeds)
        infos = [gpu_ctx.image_info(k) for k in (0, n - 1)]
        merges = [gpu_ctx.debug_merges(k) for k in (0, n - 1)]
        out1, pal1, plen1, _ = gpu_ctx.convert_batch(1, imgs[:1], w, h, 256, True, seeds=seeds[:1])
        info1 = gpu_ctx.image_info(0)
        merges1 = gpu_ctx.debug_merges(0)
    finally:
        gpu_ctx.set_debug(False)
    assert infos[0]["merge_ctas_per_sm"] >= 7 and info1["merge_ctas_per_sm"] < infos[0]["merge_ctas_per_sm"]
    assert infos[0]["maxbins"] > 4 * 2048
    for j, k in enumerate((0, n - 1)):
        ref = oracle.convert(1, imgs[k], w, h, 256, True, seed=seeds[k])
        assert np.array_equal(merges[j], ref.merges), f"image {k}: merge sequence differs"
        assert np.array_equal(pal[k, :plen[k]], ref.palette) and np.array_equal(out[k], ref.out), k
    assert np.array_equal(merges1, merges[0]) and np.array_equal(out1[0], out[0])
    for key in ("rescans", "merge_rounds", "rescans_discarded", "heap_pops"):
        assert info1[key] == infos[0][key], key


def test_4k_image_in_one_wave_of_eight_per_sm(gpu_ctx):
    """BASELINE.json configs[3] image 0 inside a device-resident batch of 4 x SMs + 1 4K images (k_merge_lab<8>, four heap
    levels in global memory): the frozen oracle output and the reference's rescans."""
    import torch
    case = next(c for c in json.load(open(os.path.join(HERE, "golden", "oracle_big_cases.json")))
                if c["name"] == "config3_4k_lab_img0")
    w, h = case["w"], case["h"]
    n = 4 * _sms() + 1
    din = torch.empty(n * w * h, dtype=torch.int32, device="cuda")
    dout = torch.empty_like(din)
    gpu_ctx.synth_device(din.data_ptr(), n, w, h, 1, 0, case["img_seed"])
    pal = np.zeros((n, 256), dtype=np.uint32)
    plen = np.zeros(n, dtype=np.int32)
    seeds = np.arange(n, dtype=np.uint64) + case["seed"]
    gpu_ctx.convert_batch_ptr(1, din.data_ptr(), dout.data_ptr(), n, w, h, case["k"], bool(case["dither"]), seeds=seeds,
                              device=True, palettes=pal, palette_lens=plen)
    torch.cuda.synchronize()
    info = gpu_ctx.image_info(0)
    out0 = dout[:w * h].cpu().numpy()
    del din, dout
    assert info["merge_ctas_per_sm"] >= 7 and info["maxbins"] == case["maxbins"]
    assert info["rescans"] == 92165
    assert _sha(pal[0, :plen[0]], "<u4") == case["palette_sha"] and _sha(out0, "<u4") == case["output_sha"]


def test_4k_heap_through_global_levels_matches_oracle(gpu_ctx):
    """The same image alone (k_merge_lab<4>): the oracle's merge sequence, bin for bin."""
    case = next(c for c in json.load(open(os.path.join(HERE, "golden", "oracle_big_cases.json")))
                if c["name"] == "config3_4k_lab_img0")
    w, h = case["w"], case["h"]
    img = make_image(w, h, case["cls"], case["alpha"], seed=case["img_seed"])
    gpu_ctx.set_debug(True)
    try:
        out, pal, plen, _ = gpu_ctx.convert_batch(1, img[None, :], w, h, case["k"], bool(case["dither"]), seeds=[case["seed"]])
        info = gpu_ctx.image_info(0)
        merges = gpu_ctx.debug_merges(0)
    finally:
        gpu_ctx.set_debug(False)
    assert info["maxbins"] == case["maxbins"] and case["maxbins"] > 4 * 2048
    assert merges.shape == (31148, 2) and _sha(merges, "<i4") == MERGES_4K_IMG0_SHA, "merge sequence differs"
    assert info["rescans"] == 92165                        # the reference's rescans, one at a time
    assert info["merges"] < info["merge_rounds"] < info["rescans"], info
    assert _sha(pal[0, :plen[0]], "<u4") == case["palette_sha"] and _sha(out[0], "<u4") == case["output_sha"]
