"""Image I/O either side of the hot path (SURVEY.md section 8f rank 3). The reference decodes a file into an
ARGB_8888 Bitmap before quantizing (PnnQuantizer.java:39-49) and hands the result back as an ARGB_8888 Bitmap
(PnnQuantizer.java:455) because Android cannot display indexed bitmaps (reference README.md:24). Here the caller
owns `int[]` buffers, so this module only converts: file -> ARGB uint32 array, and quantized ARGB + palette ->
an indexed PNG (8 bits per pixel with PLTE/tRNS), which is what a palette of <= 256 colours is for.

The PNG writer is self-contained (zlib + struct); decoding uses Pillow when it is installed.
"""
import struct
import zlib

import numpy as np


def load_argb(path):
    """Decode an image file to (argb uint32 array of height*width, width, height), non-premultiplied 0xAARRGGBB
    like Bitmap.getPixels (PnnQuantizer.java:39-44)."""
    from PIL import Image   # optional dependency, only for decoding
    im = Image.open(path).convert("RGBA")
    w, h = im.size
    a = np.asarray(im, dtype=np.uint8).reshape(-1, 4).astype(np.uint32)
    return (a[:, 3] << 24) | (a[:, 0] << 16) | (a[:, 1] << 8) | a[:, 2], w, h


def to_indices(out_argb, palette):
    """Palette index per pixel of a quantized image (convert() returns palette COLOURS, GilbertCurve.java:278-279).
    Duplicate palette entries map to their first occurrence."""
    out = np.ascontiguousarray(out_argb, dtype=np.uint32).ravel()
    pal = np.ascontiguousarray(palette, dtype=np.uint32).ravel()
    if pal.size == 0 or pal.size > 256:
        raise ValueError("palette must hold 1..256 colours")
    order = np.argsort(pal, kind="stable")
    spal = pal[order]
    pos = np.searchsorted(spal, out, side="left")
    pos = np.minimum(pos, spal.size - 1)
    if not np.array_equal(spal[pos], out):
        raise ValueError("the image holds a colour that is not in the palette")
    return order[pos].astype(np.uint8)


def _chunk(tag, data):
    return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)


def write_indexed_png(path, out_argb, palette, width, height, level=6):
    """Write the quantized image as an 8-bit indexed PNG (colour type 3). Alpha goes to a tRNS chunk."""
    return write_png8(path, to_indices(out_argb, palette), palette, width, height, level)


def write_png8(path, indices, palette, width, height, level=6):
    """Write an index map (one uint8 palette index per pixel, row-major, e.g. from Context.convert_indexed) and its palette
    as an 8-bit indexed PNG (colour type 3). Alpha goes to a tRNS chunk. Returns the file's size in bytes."""
    idx = np.ascontiguousarray(indices, dtype=np.uint8).reshape(height, width)
    pal = np.ascontiguousarray(palette, dtype=np.uint32).ravel()
    if pal.size == 0 or pal.size > 256:
        raise ValueError("palette must hold 1..256 colours")
    if idx.size and int(idx.max()) >= pal.size:
        raise ValueError("an index is past the end of the palette")
    plte = np.stack([(pal >> 16) & 0xFF, (pal >> 8) & 0xFF, pal & 0xFF], axis=1).astype(np.uint8).tobytes()
    alpha = ((pal >> 24) & 0xFF).astype(np.uint8)
    raw = np.concatenate([np.zeros((height, 1), np.uint8), idx], axis=1).tobytes()   # filter type 0 on every row
    png = b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", struct.pack(">IIBBBBB", width, height, 8, 3, 0, 0, 0)) + _chunk(b"PLTE", plte)
    if (alpha != 255).any():
        last = int(np.nonzero(alpha != 255)[0].max()) + 1
        png += _chunk(b"tRNS", alpha[:last].tobytes())
    png += _chunk(b"IDAT", zlib.compress(raw, level)) + _chunk(b"IEND", b"")
    with open(path, "wb") as f:
        f.write(png)
    return len(png)
