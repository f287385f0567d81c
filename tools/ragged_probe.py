#!/usr/bin/env python3
"""Mixed-size batch on one GPU: what nq_convert_ragged_device buys over what a caller could do without it.

Workload: 2 noisy images per SM (296 on a B200), PnnLABQuantizer, 256 colours, dither on, sizes drawn with a fixed seed from
nine common photo / video sizes, generated in HBM with nq_synth_device (one call per image into the packed buffer).
Legs, timed with CUDA events on the stream the library is ordered with, after a warm-up of every size:
  (a) ragged   one nq_convert_ragged_device call for the whole mixed batch
  (b) by_size  one nq_convert_batch_device call per distinct size (the images of each size packed together)
  (c) single   nq_convert (host buffers) on 8 of the images one by one, EXTRAPOLATED to the whole batch
(a) and (b) must give identical outputs and palettes per image (SHA-256). Prints one JSON line: Mpixels/s per leg, the
device name and its power limit. Not part of bench.py.
Usage: ragged_probe.py [--per-sm 2] [--seed 7]"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from nquant_android_b200.quantizer import Context

SIZES = [(495, 438), (640, 480), (800, 600), (1024, 768), (1280, 720), (1920, 1080), (1080, 1920), (2048, 1536), (3840, 2160)]


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def timed(stream, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-sm", type=int, default=2)
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ragged_probe: no CUDA device")
    props = torch.cuda.get_device_properties(0)
    n = args.per_sm * props.multi_processor_count
    pick = np.random.default_rng(args.seed).integers(0, len(SIZES), n)
    ws = np.array([SIZES[k][0] for k in pick], np.int32)
    hs = np.array([SIZES[k][1] for k in pick], np.int32)
    npix = ws.astype(np.int64) * hs
    off = np.concatenate([[0], np.cumsum(npix)])
    total = int(off[-1])
    seeds = (np.arange(n) + 0xC0FFEE).astype(np.uint64)

    ctx = Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    din = torch.empty(total, dtype=torch.int32, device="cuda")
    for i in range(n):
        ctx.synth_device(din.data_ptr() + 4 * int(off[i]), 1, int(ws[i]), int(hs[i]), 1, 0, 0x5EED0000 + i)
    dout_a = torch.empty_like(din)
    pal_a, plen_a = np.zeros((n, 256), np.uint32), np.zeros(n, np.int32)

    # (b) input: the images of each size packed together, in order of first appearance
    groups = {}
    for i in range(n):
        groups.setdefault((int(ws[i]), int(hs[i])), []).append(i)
    din_b = torch.cat([din[int(off[i]):int(off[i + 1])] for g in groups.values() for i in g])
    dout_b = torch.empty_like(din_b)
    pal_b, plen_b = np.zeros((n, 256), np.uint32), np.zeros(n, np.int32)

    def leg_a():
        ctx.convert_ragged_ptr(1, din.data_ptr(), dout_a.data_ptr(), ws, hs, 256, True, seeds=seeds, palettes=pal_a, palette_lens=plen_a)

    def leg_b():
        at = 0
        for (w, h), idx in groups.items():
            p, pl = np.zeros((len(idx), 256), np.uint32), np.zeros(len(idx), np.int32)
            ctx.convert_batch_ptr(1, din_b.data_ptr() + 4 * at, dout_b.data_ptr() + 4 * at, len(idx), w, h, 256, True, seeds=seeds[idx],
                                  device=True, palettes=p, palette_lens=pl)
            pal_b[idx], plen_b[idx] = p, pl
            at += len(idx) * w * h

    leg_b()                      # warm-up: every size's order table, the workspace, the speculative pool
    leg_a()
    t_a = timed(stream, leg_a)
    t_b = timed(stream, leg_b)

    out_a = dout_a.cpu().numpy()
    out_b = dout_b.cpu().numpy()
    pos_b, at = {}, 0
    for idx in groups.values():
        for i in idx:
            pos_b[i] = at
            at += int(npix[i])
    identical = all(
        hashlib.sha256(out_a[off[i]:off[i + 1]].tobytes()).digest() == hashlib.sha256(out_b[pos_b[i]:pos_b[i] + npix[i]].tobytes()).digest()
        for i in range(n)) and np.array_equal(pal_a, pal_b) and np.array_equal(plen_a, plen_b)

    # (c) 8 images one by one through the host entry, extrapolated to the batch
    sample = np.linspace(0, n - 1, 8).astype(int)
    t_c8, px_c8 = 0.0, 0
    for i in sample:
        img = din[int(off[i]):int(off[i + 1])].cpu().numpy().view(np.uint32).reshape(1, -1)
        ctx.convert_batch(1, img, int(ws[i]), int(hs[i]), 256, True, seeds=[int(seeds[i])])   # warm-up of this size on the host path
        t_c8 += timed(stream, lambda: ctx.convert_batch(1, img, int(ws[i]), int(hs[i]), 256, True, seeds=[int(seeds[i])]))
        px_c8 += int(npix[i])
    t_c = t_c8 / px_c8 * total

    print(json.dumps({
        "probe": "ragged", "device": props.name, "power_limit": power_limit(), "images": n, "mpixels": round(total / 1e6, 1),
        "sizes": {f"{w}x{h}": len(idx) for (w, h), idx in groups.items()}, "kind": "PnnLABQuantizer", "colors": 256, "dither": True,
        "a_ragged_s": round(t_a, 3), "a_ragged_mpix_s": round(total / t_a / 1e6, 1),
        "b_by_size_s": round(t_b, 3), "b_by_size_mpix_s": round(total / t_b / 1e6, 1),
        "c_single_extrapolated_s": round(t_c, 1), "c_single_extrapolated_mpix_s": round(total / t_c / 1e6, 2),
        "c_note": "extrapolated from 8 images converted one by one (host buffers)",
        "a_over_b": round(t_b / t_a, 2), "outputs_identical_a_b": bool(identical),
    }), flush=True)
    ctx.close()
    if not identical:
        sys.exit("ragged_probe: legs (a) and (b) differ")


if __name__ == "__main__":
    main()
