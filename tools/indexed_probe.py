#!/usr/bin/env python3
"""Index maps on one GPU: what nq_convert_ragged_indexed buys a caller who wants palette indices (PNG8, GIF, palette
textures) over converting to colours and recovering the indices on the host.

Workload: 256 noisy 3840x2160 images, PnnLABQuantizer, 256 colours, dither on, in pinned host buffers (generated on the
device with nq_synth_device and copied there once). Legs, each warmed up once and then timed with a host clock around the
call (every host-buffer call returns after its last copy):
  (a) colours  nq_convert_ragged into pinned ARGB buffers, then imageio.to_indices on the host. The host part is timed on
               8 images on one core and EXTRAPOLATED to the batch (it takes minutes on the whole batch).
  (b) indices  nq_convert_ragged_indexed into pinned index buffers, no colours copied back.
The indices of (b) must equal to_indices of (a)'s colours on 8 images drawn with a fixed seed, and the palettes must be
equal. Prints one JSON line with Mpixels/s of each leg, the device name and its power limit.
--profile: a separate run instead, one indexed call under torch.profiler (CUDA activities): k_index_map's kernel time,
launches, and its bytes/s (4 B read + 1 B written per pixel) against the HBM data-sheet peak of a B200 (7.7 TB/s).
Not part of bench.py.
Usage: indexed_probe.py [--images 256] [--profile] [--seed 7]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from nquant_android_b200.imageio import to_indices
from nquant_android_b200.quantizer import Context

W, H = 3840, 2160
HBM_PEAK = 7.7e12   # bytes/s, NVIDIA HGX B200 data sheet, one GPU


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=256)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("indexed_probe: no CUDA device")
    n, npix = args.images, W * H
    total = n * npix
    ctx = Context(0)
    L = ctx._L
    seeds = (np.arange(n) + 0xC0FFEE).astype(np.uint64)
    ws, hs = np.full(n, W, np.int32), np.full(n, H, np.int32)

    d = torch.empty(total, dtype=torch.int32, device="cuda")
    ctx.synth_device(d.data_ptr(), n, W, H, 1, 0, 0x5EED0000)
    h_in = torch.empty(total, dtype=torch.int32, pin_memory=True)
    h_in.copy_(d)
    del d
    torch.cuda.synchronize()
    h_idx = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    in_p = (ctypes.c_void_p * n)(*[h_in.data_ptr() + 4 * i * npix for i in range(n)])
    idx_p = (ctypes.c_void_p * n)(*[h_idx.data_ptr() + i * npix for i in range(n)])
    pal_b, plen_b = np.zeros((n, 256), np.uint32), np.zeros(n, np.int32)

    def leg_b():
        rc = L.nq_convert_ragged_indexed(ctx._h, 1, in_p, ws.ctypes.data, hs.ctypes.data, n, 256, 1, seeds.ctypes.data, idx_p, None,
                                         pal_b.ctypes.data, plen_b.ctypes.data, None)
        if rc:
            sys.exit(f"nq_convert_ragged_indexed: {rc} {L.nq_last_error().decode()}")

    props = torch.cuda.get_device_properties(0)
    head = {"probe": "indexed", "device": props.name, "power_limit": power_limit(), "images": n, "size": f"{W}x{H}",
            "mpixels": round(total / 1e6, 1), "kind": "PnnLABQuantizer", "colors": 256, "dither": True}

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        leg_b()                                                    # warm-up
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            leg_b()
        us, launches = 0.0, 0
        for e in prof.key_averages():
            if "k_index_map" in e.key:
                us += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                launches += e.count
        if not launches:
            sys.exit("indexed_probe: no k_index_map launch in the profile")
        bps = 5.0 * total / (us / 1e6)
        print(json.dumps({**head, "k_index_map_ms": round(us / 1e3, 3), "k_index_map_launches": launches,
                          "k_index_map_bytes": 5 * total, "k_index_map_tb_s": round(bps / 1e12, 2),
                          "share_of_hbm_peak": round(bps / HBM_PEAK, 3), "hbm_peak_tb_s": HBM_PEAK / 1e12,
                          "note": "kernel time summed over its launches (torch.profiler, CUDA activities); bytes = 4 read + 1 written per pixel"}),
              flush=True)
        ctx.close()
        return

    h_out = torch.empty(total, dtype=torch.int32, pin_memory=True)
    out_p = (ctypes.c_void_p * n)(*[h_out.data_ptr() + 4 * i * npix for i in range(n)])
    pal_a, plen_a = np.zeros((n, 256), np.uint32), np.zeros(n, np.int32)

    def leg_a_gpu():
        rc = L.nq_convert_ragged(ctx._h, 1, in_p, ws.ctypes.data, hs.ctypes.data, n, 256, 1, seeds.ctypes.data, out_p,
                                 pal_a.ctypes.data, plen_a.ctypes.data, None)
        if rc:
            sys.exit(f"nq_convert_ragged: {rc} {L.nq_last_error().decode()}")

    def timed(fn):
        t = time.perf_counter()
        fn()
        return time.perf_counter() - t

    leg_a_gpu()
    leg_b()
    t_a_gpu = min(timed(leg_a_gpu), timed(leg_a_gpu))
    t_b = min(timed(leg_b), timed(leg_b))
    out = h_out.numpy().view(np.uint32)
    idx = h_idx.numpy()
    sample = np.sort(np.random.default_rng(args.seed).choice(n, size=min(8, n), replace=False))
    t_host, identical = 0.0, bool(np.array_equal(pal_a, pal_b) and np.array_equal(plen_a, plen_b))
    for i in sample:
        o = out[i * npix:(i + 1) * npix]
        t = time.perf_counter()
        ref = to_indices(o, pal_a[i, :plen_a[i]])
        t_host += time.perf_counter() - t
        identical = identical and np.array_equal(ref, idx[i * npix:(i + 1) * npix])
    t_host_all = t_host / len(sample) * n
    t_a = t_a_gpu + t_host_all
    print(json.dumps({**head,
                      "a_colours_gpu_s": round(t_a_gpu, 3), "a_colours_gpu_mpix_s": round(total / t_a_gpu / 1e6, 1),
                      "a_to_indices_one_core_s_per_image": round(t_host / len(sample), 3),
                      "a_to_indices_extrapolated_s": round(t_host_all, 1),
                      "a_total_extrapolated_mpix_s": round(total / t_a / 1e6, 1),
                      "b_indexed_s": round(t_b, 3), "b_indexed_mpix_s": round(total / t_b / 1e6, 1),
                      "b_over_a_gpu_only": round(t_a_gpu / t_b, 3),
                      "host_copy_bytes_a": 4 * total, "host_copy_bytes_b": total,
                      "sample": [int(i) for i in sample], "indices_identical_on_sample": bool(identical)}), flush=True)
    ctx.close()
    if not identical:
        sys.exit("indexed_probe: indices differ from to_indices of the colours")


if __name__ == "__main__":
    main()
