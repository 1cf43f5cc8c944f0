"""PNG decoding restated serially: ``zlib.decompress`` and the five row filters of the PNG specification in numpy.

The reference for md2_png_decode (monodepth2_b200/csrc/md2_png.cu) on 8-bit truecolour non-interlaced files, pinned
byte for byte against the installed Pillow by tests/test_png_decode.py.  ``decode`` raises where Pillow raises on the
image data: corrupt deflate data, too little of it, a filter type above 4.  Like Pillow it reads the first
``height * (3 * width + 1)`` inflated bytes and ignores what follows them; it checks the Adler-32 trailer when the
stream ends exactly there or earlier.  A stream that ends early (with its trailer) after a positive whole number of
rows gives the image with the missing rows zero, as Pillow does.
"""
from __future__ import annotations

import struct
import zlib

import numpy as np


def chunks(data: bytes):
    """(type, payload) of every chunk."""
    p, out = 8, []
    while p + 12 <= len(data):
        n = struct.unpack(">I", data[p:p + 4])[0]
        out.append((data[p + 4:p + 8], data[p + 8:p + 8 + n]))
        p += 12 + n
    return out


def inflate(z: bytes, raw_bytes: int, row_bytes: int) -> bytes:
    """The first raw_bytes of the zlib stream z, as zlib gives them to Pillow: a stream that ends (Adler-32 checked)
    after a positive whole number of rows is padded with zeros, any other shortfall raises."""
    d = zlib.decompressobj()
    out = d.decompress(z, raw_bytes)
    if len(out) < raw_bytes:
        if not (d.eof and len(out) > 0 and len(out) % row_bytes == 0):
            raise ValueError("image file is truncated")
        out += bytes(raw_bytes - len(out))
    return out


def unfilter(raw: np.ndarray, h: int, w: int) -> np.ndarray:
    """(h, w, 3) uint8 from the inflated rows (a filter byte, then 3 * w bytes)."""
    rows = raw.reshape(h, 3 * w + 1)
    out = np.zeros((h, 3 * w), np.int32)
    prior = np.zeros(3 * w, np.int32)
    for y in range(h):
        f = int(rows[y, 0])
        x = rows[y, 1:].astype(np.int32)
        if f == 0:
            cur = x
        elif f == 2:
            cur = (x + prior) & 255
        elif f in (1, 3, 4):
            cur = np.zeros(3 * w, np.int32)
            for i in range(3 * w):
                a = cur[i - 3] if i >= 3 else 0
                b = prior[i]
                c = prior[i - 3] if i >= 3 else 0
                if f == 1:
                    p = a
                elif f == 3:
                    p = (a + b) >> 1
                else:
                    q = a + b - c
                    pa, pb, pc = abs(q - a), abs(q - b), abs(q - c)
                    p = a if pa <= pb and pa <= pc else (b if pb <= pc else c)
                cur[i] = (x[i] + p) & 255
        else:
            raise ValueError("unrecognized data stream contents")
        out[y] = cur
        prior = cur
    return out.astype(np.uint8).reshape(h, w, 3)


def decode(data: bytes) -> np.ndarray:
    """np.array(Image.open(f).convert("RGB")) of an 8-bit truecolour non-interlaced PNG."""
    cs = chunks(data)
    w, h, depth, ctype, _, _, interlace = struct.unpack(">IIBBBBB", cs[0][1])
    assert cs[0][0] == b"IHDR" and (depth, ctype, interlace) == (8, 2, 0)
    z = b"".join(p for t, p in cs if t == b"IDAT")
    raw = inflate(z, h * (3 * w + 1), 3 * w + 1)
    return unfilter(np.frombuffer(raw, np.uint8), h, w)
