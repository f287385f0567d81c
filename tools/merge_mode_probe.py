#!/usr/bin/env python3
"""A/B of k_merge_lab variants: one device-resident batch per mode in one process, merge stage time + phase clocks, and a
hash of all palettes (the modes must agree bit for bit). The modes are the NQ_MERGE_MODE bits of the experimental kernel
kept as profiles/r2_merge_variants.diff (not applied: the shipped library ignores the variable, every mode is the shipped
kernel); NQ_AB_LIB=path loads another build of the library instead, for an old-vs-new comparison in one session.
Usage: merge_mode_probe.py W H batch mode[,mode...]"""
import ctypes, hashlib, os, sys, time
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch
from nquant_android_b200 import _lib
if os.environ.get("NQ_AB_LIB"):          # an older build of the library, for an A/B in the same session
    _lib.SO = os.path.abspath(os.environ["NQ_AB_LIB"])
    _lib.SYMBOLS = []
    _old_size, _fields = ctypes.CDLL(_lib.SO).nq_sizeof_image_info(), list(_lib.ImageInfo._fields_)
    while ctypes.sizeof(type("_I", (ctypes.Structure,), {"_fields_": _fields})) > _old_size:   # built before the last counters
        _fields.pop()
    if len(_fields) < len(_lib.ImageInfo._fields_):

        class _OldImageInfo(ctypes.Structure):
            _fields_ = _fields
            as_dict = _lib.ImageInfo.as_dict

        _lib.ImageInfo = _OldImageInfo
from nquant_android_b200.quantizer import Context


def main():
    W, H, batch = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
    modes = [int(m) for m in sys.argv[4].split(",")]
    npix = W * H
    din = torch.empty(batch * npix, dtype=torch.int32, device="cuda")
    dout = torch.empty_like(din)
    seeds = np.arange(batch, dtype=np.uint64) + 0xC0FFEE
    first = None
    for mode in modes:
        os.environ["NQ_MERGE_MODE"] = str(mode)
        ctx = Context(0)
        ctx.set_chunk_images(batch)
        ctx.synth_device(din.data_ptr(), batch, W, H, 1, 0, 0x5EED0000)
        pal = np.zeros((batch, 256), dtype=np.uint32)
        plen = np.zeros(batch, dtype=np.int32)
        for rep in range(2):
            ctx.stage_times(reset=True)
            ctx.kernel_times(reset=True)
            torch.cuda.synchronize()
            t0 = time.time()
            ctx.convert_batch_ptr(1, din.data_ptr(), dout.data_ptr(), batch, W, H, 256, True, seeds=seeds, device=True, palettes=pal, palette_lens=plen)
            torch.cuda.synchronize()
            dt = time.time() - t0
        st = ctx.stage_times()
        info = ctx.image_info(0)
        mc = info["merge_cycles"]
        names = ["heap", "first32", "blocktest", "screen", "full", "merge"]
        hp = hashlib.sha256(pal.tobytes()).hexdigest()[:16]
        ho = hashlib.sha256(dout[:npix].cpu().numpy().tobytes()).hexdigest()[:16]
        first = first or (hp, ho)
        print(f"mode={mode:2d} {batch} x {W}x{H}: {dt:.3f} s {batch * npix / dt / 1e6:.1f} Mpix/s  merge={st['merge'][0]:.1f} ms  sweep={st['find_nn_sweep'][0]:.1f} ms  "
              f"palettes={hp} out0={ho} same_as_first={(hp, ho) == first}", flush=True)
        print("   merge Mcycles (image 0): " + "  ".join(f"{n}={c / 1e6:.0f}" for n, c in zip(names, mc)) +
              f"  rescans={info['rescans']} rounds={info.get('merge_rounds', '-')} discarded={info.get('rescans_discarded', '-')} "
              f"full_evals={info['full_evals']} live_blocks={info['live_blocks']} screened={info['screened']} "
              f"merge_ctas_per_sm={info.get('merge_ctas_per_sm', '-')}", flush=True)
        ctx.close()


main()
