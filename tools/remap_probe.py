#!/usr/bin/env python3
"""Remap on one GPU: what nq_remap_ragged_device costs against nq_convert_ragged_device on the same images, when the
palettes are the ones convert produced (so the two outputs must be identical, which is checked on the device).

Workloads (device-resident inputs from nq_synth_device, noisy opaque):
  configs3   1024 x 3840x2160, PnnLABQuantizer, 256 colours, dither on (bench.py's configs[3])
  1080p_x592  592 x 1920x1080, PnnLABQuantizer, 256 colours, dither on
  512_single    1 x 512x512,   PnnQuantizer,    256 colours, dither on (configs[0])
  1080p_single  1 x 1920x1080, PnnLABQuantizer, 256 colours, dither on (configs[1])
Each workload: one convert and one remap as warm-up, then --reps rounds of convert followed by remap, each call bracketed
by CUDA events on the stream the context is ordered on. Prints one JSON line per workload: the best time of each leg,
Mpixels/s, per-stage device times of the last round (nq_get_stage_times), the speed-up, and whether every remap output
equals the convert output. The device name and its power limit are read in the same run. Not part of bench.py.
Usage: remap_probe.py [--reps 2] [--only NAME[,NAME]]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from nquant_android_b200.quantizer import Context

WORKLOADS = [("configs3", 1024, 3840, 2160, 1), ("1080p_x592", 592, 1920, 1080, 1), ("512_single", 1, 512, 512, 0),
             ("1080p_single", 1, 1920, 1080, 1)]


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def run(ctx, name, n, w, h, kind, reps, head):
    total = n * w * h
    d_in = torch.empty(total, dtype=torch.int32, device="cuda")
    ctx.synth_device(d_in.data_ptr(), n, w, h, 1, 0, 0x5EED0000)
    d_conv = torch.empty_like(d_in)
    d_remap = torch.empty_like(d_in)
    ws, hs = [w] * n, [h] * n
    seeds = (np.arange(n) + 0xC0FFEE).astype(np.uint64)
    pal, plen = np.zeros((n, 256), np.uint32), np.zeros(n, np.int32)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)

    def convert():
        ctx.convert_ragged_ptr(kind, d_in.data_ptr(), d_conv.data_ptr(), ws, hs, 256, True, seeds=seeds, palettes=pal, palette_lens=plen)

    def remap():
        ctx.remap_ptr(kind, d_in.data_ptr(), ws, hs, [pal[i, :plen[i]] for i in range(n)], True, n_max_colors=256, seeds=seeds,
                      out_ptr=d_remap.data_ptr())

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.stage_times(reset=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b) / 1e3, {k: round(v[0], 1) for k, v in ctx.stage_times(reset=True).items()}

    convert()
    remap()
    identical = bool(torch.equal(d_conv, d_remap))
    best = {"convert": None, "remap": None}
    stages = {}
    for _ in range(reps):
        for leg, fn in (("convert", convert), ("remap", remap)):
            t, st = timed(fn)
            best[leg] = t if best[leg] is None else min(best[leg], t)
            stages[leg] = st
        identical = identical and bool(torch.equal(d_conv, d_remap))
    ctx.reset_stream()
    print(json.dumps({**head, "workload": name, "images": n, "size": f"{w}x{h}", "kind": ["PnnQuantizer", "PnnLABQuantizer"][kind],
                      "colors": 256, "dither": True, "mpixels": round(total / 1e6, 1), "reps": reps,
                      "convert_s": round(best["convert"], 4), "remap_s": round(best["remap"], 4),
                      "convert_mpix_s": round(total / best["convert"] / 1e6, 1), "remap_mpix_s": round(total / best["remap"] / 1e6, 1),
                      "speedup": round(best["convert"] / best["remap"], 2),
                      "stage_ms_convert": stages["convert"], "stage_ms_remap": stages["remap"],
                      "outputs_identical": identical}), flush=True)
    del d_in, d_conv, d_remap
    torch.cuda.empty_cache()
    return identical


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("remap_probe: no CUDA device")
    only = set(args.only.split(",")) - {""}
    head = {"probe": "remap", "device": torch.cuda.get_device_properties(0).name, "power_limit": power_limit()}
    ctx = Context(0)
    ok = True
    for name, n, w, h, kind in WORKLOADS:
        if not only or name in only:
            ok = run(ctx, name, n, w, h, kind, args.reps, head) and ok
    ctx.close()
    if not ok:
        sys.exit("remap_probe: a remap output differs from the convert output")


if __name__ == "__main__":
    main()
