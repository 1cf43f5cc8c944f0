"""PNG decoding on the GPU (md2_png_decode, monodepth2_b200/png.py) against Pillow and oracle/png_decode.py.

CPU: the oracle against Pillow, the parser's accept / decline rule and the mixin's fallback, a g++ build of md2_png.h
running the kernels' finder / count / walk / write / marker / filter passes serially against the oracle and Pillow
(with the finder and without it, so every block is also decoded where the walk meets it), the same build under
AddressSanitizer on truncated, bit-flipped and random streams, the ABI's validation and the job layout, the mixin's
draws and the ptxas log.  GPU: decode_png byte-exact with Pillow on the corpus, the statuses of corrupt files,
MonoBatch fed by PNG items equal to MonoBatch fed by native frames, a CUDA graph over other batches, a two-worker
DataLoader, and identical bytes run to run.

The corpus is written by a small PNG writer of its own (a filter per row, zlib level and strategy, IDAT split), by
Pillow at every compress_level class, and by a hand-made deflate stream with a distance of 32768 across a block."""
import ctypes as C
import io
import os
import random
import re
import struct
import subprocess
import zlib

import numpy as np
import pytest
import torch
from PIL import Image

from monodepth2_b200 import png as PN
from monodepth2_b200 import synthetic as S
from monodepth2_b200.mono_batch import NativeFramesMixin
from oracle import png_decode as OP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "monodepth2_b200", "csrc")


def _frame(seed, h, w):
    """Smooth colour fields plus noise, like a camera frame."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    base = np.stack([120 + 90 * np.sin(x / (17.0 + seed % 7) + c) * np.cos(y / 11.0 - c) for c in (0.0, 1.3, 2.6)], -1)
    return np.clip(base + rng.normal(0, 12, (h, w, 3)), 0, 255).astype(np.uint8)


def pil_rgb(data):
    return np.array(Image.open(io.BytesIO(data)).convert("RGB"))


def _chunk(t, d, crc=None):
    return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) if crc is None else crc)


def _filter(a, f):
    """The raw rows of a (h, w, 3) uint8 image with filter f (an int, or one per row)."""
    h, w, _ = a.shape
    x = a.reshape(h, 3 * w).astype(np.int32)
    fs = [f] * h if isinstance(f, int) else list(f)
    rows = []
    for y in range(h):
        cur = x[y]
        prior = x[y - 1] if y else np.zeros_like(cur)
        left = np.concatenate([np.zeros(3, np.int32), cur[:-3]])
        upleft = np.concatenate([np.zeros(3, np.int32), prior[:-3]])
        if fs[y] == 0:
            pred = 0
        elif fs[y] == 1:
            pred = left
        elif fs[y] == 2:
            pred = prior
        elif fs[y] == 3:
            pred = (left + prior) >> 1
        else:
            p = left + prior - upleft
            pa, pb, pc = np.abs(p - left), np.abs(p - prior), np.abs(p - upleft)
            pred = np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, prior, upleft))
        rows.append(bytes([fs[y]]) + ((cur - pred) & 255).astype(np.uint8).tobytes())
    return b"".join(rows)


def write_png(a, f=0, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, split=None, z=None, extra_before=b""):
    """An 8-bit RGB PNG of ``a``: filter ``f`` per row, zlib ``level`` / ``strategy``, the zlib stream (or ``z``)
    cut into IDAT chunks of ``split`` bytes (a list of sizes, cycled; 0 makes an empty chunk)."""
    h, w, _ = a.shape
    if z is None:
        c = zlib.compressobj(level, zlib.DEFLATED, 15, 8, strategy)
        z = c.compress(_filter(a, f)) + c.flush()
    parts = [z]
    if split:
        parts, p, k = [], 0, 0
        while p < len(z):
            n = split[k % len(split)]
            parts.append(z[p:p + n])
            p += n
            k += 1
    return (PN.SIGNATURE + _chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)) + extra_before +
            b"".join(_chunk(b"IDAT", d) for d in parts) + _chunk(b"IEND", b""))


def pil_png(a, **kw):
    b = io.BytesIO()
    Image.fromarray(a).save(b, "PNG", **kw)
    return b.getvalue()


class _Bits:
    """A deflate bit writer (LSB first; Huffman codes MSB first)."""

    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, v, n):
        self.v |= v << self.n
        self.n += n

    def code(self, c, n):
        self.put(int(format(c, "0%db" % n)[::-1], 2), n)

    def lit(self, s):                                 # the fixed literal/length code
        if s < 144:
            self.code(0x30 + s, 8)
        elif s < 256:
            self.code(0x190 + s - 144, 9)
        elif s < 280:
            self.code(s - 256, 7)
        else:
            self.code(0xC0 + s - 280, 8)

    def align(self):
        self.n = (self.n + 7) // 8 * 8

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def distance_32768_png():
    """A 5461x4 frame (rows of 16384 bytes): rows 0-1 in a stored block, rows 2-3 copied at distance 32768 by a fixed
    block, so every byte of the second block is a marker into the first."""
    a = np.random.default_rng(5).integers(0, 256, (4, 5461, 3), dtype=np.uint8)
    a[2:] = a[:2]
    raw = _filter(a, 0)
    assert raw[32768:] == raw[:32768]
    b = _Bits()
    b.put(0, 1)
    b.put(0, 2)
    b.align()
    b.put(32768, 16)
    b.put(32768 ^ 0xFFFF, 16)
    for c in raw[:32768]:
        b.put(c, 8)
    b.put(1, 1)
    b.put(1, 2)
    for length in [258] * 126 + [257, 3]:
        if length == 258:
            b.lit(285)
        elif length == 257:
            b.lit(284)
            b.put(257 - 227, 5)
        else:
            b.lit(257)
        b.code(29, 5)
        b.put(32768 - 24577, 13)
    b.lit(256)
    z = b"\x78\x01" + b.bytes() + struct.pack(">I", zlib.adler32(raw))
    return write_png(a, z=z)


def corpus(sizes=((1, 1), (1, 7), (7, 1), (5, 9), (16, 16), (33, 47))):
    """(id, bytes) of the decodable corpus."""
    out = []
    for h, w in sizes:
        a = _frame(h * 31 + w, h, w)
        for lvl in (0, 1, 6, 9):
            out.append(("%dx%d-pil%d" % (w, h, lvl), pil_png(a, compress_level=lvl)))
        for st in ("Z_FIXED", "Z_HUFFMAN_ONLY", "Z_RLE", "Z_FILTERED"):
            out.append(("%dx%d-%s" % (w, h, st), write_png(a, f=h % 5, strategy=getattr(zlib, st))))
        for f in range(5):
            out.append(("%dx%d-f%d" % (w, h, f), write_png(a, f=f)))
        out.append(("%dx%d-fmix" % (w, h), write_png(a, f=[y % 5 for y in range(h)], level=9)))
        out.append(("%dx%d-split" % (w, h), write_png(a, f=4, split=[1, 0, 3, 1000])))
        out.append(("%dx%d-const" % (w, h), write_png(np.full((h, w, 3), 77, np.uint8), f=0)))
    return out


def big_corpus():
    """KITTI-size frames: Pillow's default and fast levels, every filter, a constant frame (runs of 258 at distance 1
    across many blocks), the five native sizes, and the distance-32768 stream."""
    out = []
    for k, (h, w) in enumerate(S.KITTI_NATIVE_SIZES):
        a = _frame(k, h, w)
        out.append(("kitti-%dx%d-pil6" % (w, h), pil_png(a)))
    a = _frame(9, 375, 1242)
    out.append(("kitti-pil1", pil_png(a, compress_level=1)))
    out.append(("kitti-pil0", pil_png(a, compress_level=0)))
    out.append(("kitti-fmix", write_png(a, f=[y % 5 for y in range(375)], split=[65536])))
    out.append(("kitti-const", write_png(np.full((375, 1242, 3), 200, np.uint8), f=0, level=9)))
    out.append(("kitti-rle", write_png(a, f=2, strategy=zlib.Z_RLE)))
    out.append(("distance-32768", distance_32768_png()))
    return out


def _rebuild(png, z):
    """png with its IDAT data replaced by z (one chunk)."""
    cs = OP.chunks(png)
    out, done = PN.SIGNATURE, False
    for t, p in cs:
        if t == b"IDAT":
            if not done:
                out += _chunk(b"IDAT", z)
            done = True
        else:
            out += _chunk(t, p)
    return out


def trap_cases(h, w):
    """(name, bytes, status bit or 0) of the corrupt and odd streams whose outcome is pinned against Pillow: a bit
    where Pillow raises on the image data, 0 where it decodes the image."""
    a = _frame(1, h, w)
    raw = _filter(a, 1)
    good = write_png(a, f=1)
    z = b"".join(p for t, p in OP.chunks(good) if t == b"IDAT")
    c = zlib.compressobj(6)
    no_final = c.compress(raw) + c.flush(zlib.Z_SYNC_FLUSH)
    bad_idat_crc = bytearray(good)
    i = good.index(b"IDAT") + 4 + len(z)
    bad_idat_crc[i] ^= 1
    bad_filter = bytearray(raw)
    bad_filter[(h - 1) * (3 * w + 1)] = 5
    flip = lambda q: q[:-1] + bytes([q[-1] ^ 1])
    rb = 3 * w + 1
    short = []                                         # complete zlib streams that end early
    for rows, bit in ((h - 1, 0), (1, 0), (0, PN.EXHAUSTED)):   # a whole number of rows: Pillow keeps them
        zs = zlib.compress(raw[:rows * rb])
        short += [("%d rows of %d" % (rows, h), _rebuild(good, zs), bit),
                  ("%d rows of %d, adler flipped" % (rows, h), _rebuild(good, flip(zs)), PN.CHECKSUM)]
    zs = zlib.compress(raw[:(h - 1) * rb + 5])
    short += [("ends mid-row", _rebuild(good, zs), PN.EXHAUSTED),
              ("ends mid-row, adler flipped", _rebuild(good, flip(zs)), PN.CHECKSUM),
              ("%d rows, no trailer" % (h - 1), _rebuild(good, zlib.compress(raw[:(h - 1) * rb])[:-4]), PN.EXHAUSTED),
              ("%d rows, no final block" % (h - 1), _rebuild(good, (lambda c: c.compress(raw[:(h - 1) * rb]) +
                                                                    c.flush(zlib.Z_SYNC_FLUSH))(zlib.compressobj())),
               PN.EXHAUSTED)]
    return short + [("adler flipped", _rebuild(good, z[:-1] + bytes([z[-1] ^ 1])), PN.CHECKSUM),
            ("adler missing", _rebuild(good, z[:-4]), 0),
            ("adler cut to 2 bytes", _rebuild(good, z[:-2]), 0),
            ("junk after the stream", _rebuild(good, z + b"junkjunk"), 0),
            ("adler flipped, junk after", _rebuild(good, z[:-1] + bytes([z[-1] ^ 1]) + b"junk"), PN.CHECKSUM),
            ("filter 5 on the last row", _rebuild(good, zlib.compress(bytes(bad_filter))), PN.BAD_FILTER),
            ("deflate data cut in half", _rebuild(good, z[:len(z) // 2]), PN.EXHAUSTED),
            ("one byte too little", _rebuild(good, zlib.compress(raw[:-1])), PN.EXHAUSTED),
            ("a row too much, bad adler", _rebuild(good, (lambda q: q[:-1] + bytes([q[-1] ^ 1]))(
                zlib.compress(raw + bytes(3 * w + 1)))), 0),
            ("no final block", _rebuild(good, no_final), 0),
            ("bad IDAT CRC", bytes(bad_idat_crc), 0),
            ("BTYPE 3", _rebuild(good, b"\x78\x9c\x07" + z[3:]), PN.BAD_CODE)]


@pytest.mark.parametrize("size", [(40, 64), (375, 1242)], ids=["64x40", "1242x375"])
def test_trailer_in_a_later_idat_piece(host_lib, size):
    """Pillow feeds zlib one IDAT piece (a chunk, read at most 64 KB at a time) per call and stops once the last row is
    complete, so it never sees a bad Adler-32 trailer that lies in a later piece than the bytes completing the image.
    The decoder reads the joined stream and checks it: the one documented case where it flags a file Pillow decodes.
    The pixels are Pillow's either way."""
    a = _frame(1, *size)
    c = zlib.compressobj(6)
    z = c.compress(_filter(a, 1)) + c.flush()
    bad = z[:-1] + bytes([z[-1] ^ 1])
    for tail in (1, 2, 4):
        d = write_png(a, z=bad, split=[len(bad) - tail, tail])
        assert not _pillow_raises(d)
        st, out, _, _ = _host_decode(host_lib, PN.parse_png(d))
        assert st == PN.CHECKSUM and np.array_equal(out, pil_rgb(d))


def _pillow_raises(d):
    try:
        pil_rgb(d)
        return False
    except (OSError, SyntaxError, ValueError, zlib.error):
        return True


# ------------------------------------------------------------------ CPU: the oracle, the writer, the traps
def test_oracle_equals_pillow():
    for name, d in corpus() + big_corpus():
        assert np.array_equal(OP.decode(d), pil_rgb(d)), name


def test_corpus_covers_the_block_types_and_filters():
    """The corpus reaches what it is meant to: every filter type in Pillow's own files or the writer's, and stored,
    fixed and dynamic blocks."""
    seen_f, seen_t = set(), set()
    for name, d in corpus() + big_corpus():
        s = PN.parse_png(d)
        raw = OP.inflate(b"\x78\x9c" + s.stream.tobytes(), s.raw_bytes, 3 * s.width + 1)
        seen_f |= set(np.frombuffer(raw, np.uint8)[::3 * s.width + 1].tolist())
        seen_t.add(int(s.stream[0]) >> 1 & 3)
    assert seen_f == {0, 1, 2, 3, 4} and seen_t == {0, 1, 2}


@pytest.mark.parametrize("size", [(40, 64), (375, 1242)], ids=["64x40", "1242x375"])
def test_trap_cases_as_pillow_sees_them(size):
    for name, d, bit in trap_cases(*size):
        assert _pillow_raises(d) == bool(bit), name
        if not bit:
            assert np.array_equal(OP.decode(d), pil_rgb(d)), name
        else:
            with pytest.raises((ValueError, zlib.error)):
                OP.decode(d)


# ------------------------------------------------------------------ CPU: the parser and the mixin
def test_parse_accepts_the_supported_class():
    for name, d in corpus():
        s = PN.parse_png(d)
        assert s is not None, name
        assert s.shape == pil_rgb(d).shape, name
    a = _frame(2, 9, 11)
    assert PN.parse_png(write_png(a, extra_before=_chunk(b"tEXt", b"k\x00v") + _chunk(b"gAMA", b"\0\1\x86\xa0")))


def _unsupported():
    a = _frame(1, 20, 30)
    good = write_png(a)
    ihdr = lambda depth, ctype, il=0: (PN.SIGNATURE + _chunk(b"IHDR", struct.pack(">IIBBBBB", 30, 20, depth, ctype, 0, 0, il)))
    rest = good[33:]
    bad_crc = bytearray(good)
    bad_crc[29] ^= 1
    z = b"".join(p for t, p in OP.chunks(good) if t == b"IDAT")
    dict_z = bytes([0x78, 0xBB]) + b"\0\0\0\1" + z[2:]
    split = write_png(a, split=[10])
    i = split.index(b"IDAT", 40) - 4
    return {"palette": _pil_mode(a, "P"),
            "grey": _pil_mode(a, "L"), "rgba": _pil_mode(a, "RGBA"), "sixteen-bit": ihdr(16, 2) + rest,
            "adam7": _pil_interlaced(a), "preset-dictionary": _rebuild(good, dict_z),
            "unknown-critical": good[:33] + _chunk(b"ABCD", b"xx") + good[33:],
            "bad-crc-before-idat": bytes(bad_crc),
            "idat-not-consecutive": split[:i] + _chunk(b"tEXt", b"a\x00b") + split[i:],
            "jpeg": _pil_jpeg(a)}


def _pil_mode(a, mode):
    b = io.BytesIO()
    Image.fromarray(a).convert(mode).save(b, "PNG")
    return b.getvalue()


def _pil_interlaced(a):
    """An Adam7 file: Pillow cannot write one, so the header says interlaced over Pillow's own data; the parser
    declines it on the header alone."""
    d = bytearray(pil_png(a))
    d[28] = 1
    d[29:33] = struct.pack(">I", zlib.crc32(bytes(d[12:29])))
    return bytes(d)


def _pil_jpeg(a):
    b = io.BytesIO()
    Image.fromarray(a).save(b, "JPEG")
    return b.getvalue()


class _PngDataset:
    """The part of the reference's KITTIRAWDataset the mixins use, on .png files (pil_loader)."""

    def __init__(self, root, filenames, frame_idxs, is_train=True):
        from oracle import mono_batch as OM
        self.data_path, self.filenames, self.frame_idxs, self.is_train = root, filenames, frame_idxs, is_train
        self.brightness, self.contrast, self.saturation, self.hue = OM.BRIGHTNESS, OM.CONTRAST, OM.SATURATION, OM.HUE
        self.load_depth = False

    def __len__(self):
        return len(self.filenames)

    def get_image_path(self, folder, frame_index, side):
        return os.path.join(self.data_path, folder, "image_0%d" % {"l": 2, "r": 3}[side], "data",
                            "%010d.png" % frame_index)

    def get_color(self, folder, frame_index, side, do_flip):
        with open(self.get_image_path(folder, frame_index, side), "rb") as f:
            color = Image.open(f).convert("RGB")
        if do_flip:
            color = color.transpose(Image.FLIP_LEFT_RIGHT)
        return color


from monodepth2_b200.jpeg import JpegFramesMixin, JpegStream  # noqa: E402


class _GpuPng(PN.PngFramesMixin, JpegFramesMixin, NativeFramesMixin, _PngDataset):
    pass


class _HostPng(NativeFramesMixin, _PngDataset):
    pass


@pytest.mark.parametrize("kind", sorted(_unsupported()))
def test_parse_declines_the_rest_and_the_mixin_falls_back(tmp_path, kind):
    d = _unsupported()[kind]
    assert PN.parse_png(d) is None
    ds = _GpuPng(str(tmp_path), ["d 1 l"], [0])
    p = tmp_path / "d" / "image_02" / "data" / "0000000001.png"
    p.parent.mkdir(parents=True)
    p.write_bytes(d)
    if _pillow_raises(d):
        with pytest.raises((OSError, SyntaxError)):
            ds.native_color("d", 1, "l")
        return
    got = ds.native_color("d", 1, "l")
    if kind == "jpeg":
        assert isinstance(got, JpegStream)
        return
    assert isinstance(got, np.ndarray) and np.array_equal(got, pil_rgb(d))


def _write_png_drive(root, folder, size_of, n_frames, odd=None, level=6):
    """KITTI-like image_02 / image_03 .png frames; ``odd`` maps (side, index) to "jpeg" (JPEG bytes in a .png file)
    or "palette" (a file the GPU decoders decline)."""
    for side, cam in (("l", 2), ("r", 3)):
        d = os.path.join(root, folder, "image_0%d" % cam, "data")
        os.makedirs(d, exist_ok=True)
        for i in range(n_frames):
            h, w = size_of(side, i)
            a = _frame(i * 2 + cam, h, w)
            kind = (odd or {}).get((side, i))
            data = _pil_jpeg(a) if kind == "jpeg" else _pil_mode(a, "P") if kind == "palette" else \
                pil_png(a, compress_level=level)
            with open(os.path.join(d, "%010d.png" % i), "wb") as f:
                f.write(data)


def test_mixin_makes_the_native_mixins_draws(tmp_path):
    pytest.importorskip("torchvision")
    _write_png_drive(str(tmp_path), "d", lambda s, i: (30, 50), 4, odd={("r", 2): "palette", ("l", 1): "jpeg"})
    names = ["d 1 l", "d 2 r", "d 1 r"]
    gpu, host = _GpuPng(str(tmp_path), names, [0, -1, 1, "s"]), _HostPng(str(tmp_path), names, [0, -1, 1, "s"])
    kinds = set()
    for seed in range(12):
        random.seed(seed); torch.manual_seed(seed)
        a = gpu[seed % 3]
        after = (random.random(), float(torch.rand(1)))
        random.seed(seed); torch.manual_seed(seed)
        b = host[seed % 3]
        assert after == (random.random(), float(torch.rand(1)))
        assert (a["do_flip"], a["do_color_aug"], a["side"]) == (b["do_flip"], b["do_color_aug"], b["side"])
        for f in b["frames"]:
            x = a["frames"][f]
            kinds.add(type(x).__name__)
            if isinstance(x, np.ndarray):
                assert np.array_equal(x, b["frames"][f])
            else:
                assert x.shape == b["frames"][f].shape and x.name.endswith(".png")
    assert kinds == {"PngStream", "JpegStream", "ndarray"}


# ------------------------------------------------------------------ CPU: md2_png.h compiled with g++
@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("png_host")
    so = d / "ph.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(ROOT, "tests", "png", "md2_png_host.cpp"), "-o", str(so)])
    return C.CDLL(str(so))


def _packed(streams):
    outs, total = [], 0
    for s in streams:
        outs.append(total)
        total = PN._align(total + s.nbytes)
    body = PN._align(len(streams) * PN.JOB_DTYPE.itemsize, 64)
    h = np.zeros(body + PN.body_bytes(streams), np.uint8)
    sb, rb = PN.pack(h, 0, body, streams, outs)
    return h, sb, rb, total


def _host_decode(lib, s, use_finder=1):
    h = _packed([s])[0]
    out = np.zeros(s.shape, np.uint8)
    nc, nw = C.c_int(0), C.c_int(0)
    st = lib.decode_host(h.ctypes.data_as(C.c_void_p), h.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                         use_finder, C.byref(nc), C.byref(nw))
    return st, out, nc.value, nw.value


@pytest.mark.parametrize("use_finder", [1, 0], ids=["finder", "walk-only"])
def test_host_decode_equals_oracle_and_pillow(host_lib, use_finder):
    for name, d in corpus():
        st, out, _, _ = _host_decode(host_lib, PN.parse_png(d), use_finder)
        assert st == 0, name
        assert np.array_equal(out, pil_rgb(d)), name


def test_host_decode_kitti_size_takes_the_blocks_from_the_finder(host_lib):
    for name, d in big_corpus():
        s = PN.parse_png(d)
        st, out, n_cands, n_walked = _host_decode(host_lib, s)
        assert st == 0 and np.array_equal(out, OP.decode(d)), name
        if name.endswith("pil6") or name == "kitti-fmix":      # zlib's dynamic blocks: every one found
            assert n_walked >= 10 and n_cands < n_walked * 4 + 200, (name, n_cands, n_walked)


@pytest.mark.parametrize("size", [(40, 64), (375, 1242)], ids=["64x40", "1242x375"])
def test_host_decode_traps(host_lib, size):
    for name, d, bit in trap_cases(*size):
        s = PN.parse_png(d)
        st, out, _, _ = _host_decode(host_lib, s)
        assert st == bit, (name, st)
        if not bit:
            assert np.array_equal(out, pil_rgb(d)), name


def test_host_decode_of_corrupt_streams_stays_in_bounds(tmp_path):
    """AddressSanitizer build: truncated, bit-flipped and random streams terminate and touch nothing outside their
    buffers; every one Pillow rejects sets the status word."""
    exe = tmp_path / "ph_asan"
    try:
        subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address", "-fno-omit-frame-pointer",
                               "-DMD2_PNG_HOST_MAIN", "-I", CSRC, os.path.join(ROOT, "tests", "png", "md2_png_host.cpp"),
                               "-o", str(exe)], stderr=subprocess.DEVNULL)
    except subprocess.CalledProcessError:
        pytest.skip("g++ cannot build with AddressSanitizer here")
    rng = np.random.default_rng(7)
    goods = [write_png(_frame(3, 31, 47), f=4), write_png(_frame(4, 40, 64), f=1, strategy=zlib.Z_FIXED),
             pil_png(_frame(5, 24, 40), compress_level=0)]
    flagged = agree = 0
    for k in range(36):
        d = goods[k % 3]
        s = PN.parse_png(d)
        z = s.stream.copy()
        if k % 4 == 0:                                    # truncated
            z = z[:int(rng.integers(0, len(z)))]
        elif k % 4 == 1:                                  # a few flipped bits
            for _ in range(1 + k % 3):
                i = int(rng.integers(0, len(z) * 8))
                z[i // 8] ^= 1 << (i % 8)
        else:                                             # random bytes
            z = rng.integers(0, 256, len(z), dtype=np.uint8)
            if k % 4 == 3:
                z[:] = 0xFF if k % 8 == 3 else 0
        s.stream = z
        h = _packed([s])[0]
        path = tmp_path / ("s%d.bin" % k)
        path.write_bytes(h.tobytes())
        for use_finder in ("1", "0"):
            r = subprocess.run([str(exe), str(path), use_finder], capture_output=True, text=True, timeout=300,
                               env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
            assert r.returncode == 0, r.stderr[-2000:]
            st = int(r.stdout.split()[0])
            flagged += st != 0
        d2 = _rebuild(d, b"\x78\x9c" + z.tobytes())
        agree += (st != 0) == _pillow_raises(d2)
    assert flagged >= 50 and agree == 36


# ------------------------------------------------------------------ CPU: ABI, layout, ptxas
def test_job_layout_matches_header(tmp_path):
    src = tmp_path / "job.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "md2_loss.h"', 'int main(void) {',
             'printf("job %zu\\n", sizeof(md2_png_job));', 'printf("side %d\\n", MD2_PNG_MAX_SIDE);']
    lines += ['printf("%s %%zu\\n", offsetof(md2_png_job, %s));' % (n, n) for n in PN.JOB_DTYPE.names]
    lines += ['printf("bit%d %%u\\n", %s);' % (i, m) for i, m in enumerate(
        ["MD2_PNG_BAD_CODE", "MD2_PNG_DISTANCE", "MD2_PNG_EXHAUSTED", "MD2_PNG_BAD_FILTER", "MD2_PNG_CHECKSUM",
         "MD2_PNG_CAPACITY"])]
    src.write_text("\n".join(lines + ['return 0; }']))
    exe = tmp_path / "job"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["job"]) == PN.JOB_DTYPE.itemsize and int(got["side"]) == PN.MAX_SIDE
    for n in PN.JOB_DTYPE.names:
        assert int(got[n]) == PN.JOB_DTYPE.fields[n][1], n
    assert [int(got["bit%d" % i]) for i in range(6)] == [PN.BAD_CODE, PN.DISTANCE, PN.EXHAUSTED, PN.BAD_FILTER,
                                                         PN.CHECKSUM, PN.CAPACITY]


@pytest.fixture(scope="module")
def lib():
    from monodepth2_b200 import _capi, build
    build.build()
    return _capi.load_library()


def test_png_abi_validation_without_gpu(lib):
    n = C.c_size_t(0)
    assert lib.md2_png_decode_scratch_bytes(0, 10, 10, C.byref(n)) == -1
    assert lib.md2_png_decode_scratch_bytes(1, 0, 10, C.byref(n)) == -1
    assert lib.md2_png_decode_scratch_bytes(1, 10, 0, C.byref(n)) == -1
    assert lib.md2_png_decode_scratch_bytes(1, 10, 10, None) == -1
    streams = [PN.parse_png(write_png(_frame(k, 17, 33), f=k)) for k in (0, 4)]
    h, sb, rb, total = _packed(streams)
    assert lib.md2_png_decode_scratch_bytes(2, sb, rb, C.byref(n)) == 0
    need = n.value
    assert need >= rb * 5
    dummy = np.zeros(64, np.uint8).ctypes.data

    def call(jobs=None, n_images=2, data_bytes=len(h), frames_bytes=total, max_stream=sb, max_raw=rb,
             scratch_bytes=need, data=h.ctypes.data, status=dummy):
        j = h[:2 * PN.JOB_DTYPE.itemsize].view(PN.JOB_DTYPE).copy() if jobs is None else jobs
        return lib.md2_png_decode(data, data_bytes, j.ctypes.data, dummy, n_images, dummy, frames_bytes, status,
                                  max_stream, max_raw, dummy, scratch_bytes, None)

    def jobs(**kw):
        j = h[:2 * PN.JOB_DTYPE.itemsize].view(PN.JOB_DTYPE).copy()
        for k, v in kw.items():
            j[k][1] = v
        return j
    assert call(n_images=0) == -1 and call(data=None) == -1 and call(status=None) == -1
    assert call(max_stream=0) == -1 and call(max_raw=0) == -1
    assert call(jobs(height=0)) == -1 and call(jobs(width=PN.MAX_SIDE + 1)) == -1     # dimensions
    assert call(jobs(stream_bytes=-1)) == -1
    assert call(jobs(stream_index=0)) == -1 and call(jobs(raw_offset=0)) == -1        # not the running sums
    assert call(jobs(stream_offset=len(h))) == -1                                     # the stream outside `data`
    assert call(jobs(stream_offset=int(h[:48].view(PN.JOB_DTYPE)["stream_offset"][0]) + 2)) == -1   # misaligned
    assert call(data_bytes=len(h) - 64) == -1
    end = int(h[:96].view(PN.JOB_DTYPE)["out_offset"][1]) + streams[1].nbytes
    assert call(frames_bytes=end - 1) == -1                                           # the frame outside `frames`
    assert call(max_stream=sb - 1) == -2 and call(max_raw=rb - 1) == -2               # over the capacity
    assert call(scratch_bytes=need - 1) == -3


def test_ptxas_reports_no_spills(lib):
    log = os.path.join(ROOT, "monodepth2_b200", "lib", "libmd2loss.md2_png.cu.ptxas.log")
    txt = open(log).read()
    kernels = re.findall(r"Compiling entry function '\S*?\d(md2_png_[a-z]+)E", txt)
    assert sorted(set(kernels)) == ["md2_png_chain", "md2_png_count", "md2_png_find", "md2_png_resolve",
                                    "md2_png_unfilter", "md2_png_write"]
    spills = re.findall(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", txt)
    assert len(spills) == 6 and all(s == ("0", "0", "0") for s in spills), spills


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_decode_png_equals_pillow_one_per_call_and_mixed():
    items = corpus() + big_corpus()
    wants = [pil_rgb(d) for _, d in items]
    for (name, d), want in zip(items, wants):
        got = PN.decode_png([d])[0]
        assert np.array_equal(got.cpu().numpy(), want), name
    order = np.random.default_rng(0).permutation(len(items))
    got = PN.decode_png([items[i][1] for i in order])
    for g, i in zip(got, order):
        assert np.array_equal(g.cpu().numpy(), wants[i]), items[i][0]
    again = PN.decode_png([items[i][1] for i in order])
    assert all(torch.equal(a, b) for a, b in zip(got, again))


@pytest.mark.gpu
def test_decode_png_statuses_of_corrupt_files():
    from monodepth2_b200 import _capi
    lib = _capi.load_library()
    for size in ((40, 64), (375, 1242)):
        cases = trap_cases(*size)
        streams = [PN.parse_png(d, name) for name, d, _ in cases]
        h, sb, rb, total = _packed(streams)
        buf = torch.from_numpy(h).pin_memory()
        flat = buf.cuda()
        frames = torch.empty(total, dtype=torch.uint8, device="cuda")
        status = torch.empty(len(cases), dtype=torch.int32, device="cuda")
        PN.run(lib, flat, buf.data_ptr(), 0, len(cases), frames, status, sb, rb)
        st = status.cpu().tolist()
        for (name, d, bit), s in zip(cases, st):
            assert s == bit, (size, name, s)
        with pytest.raises(ValueError, match="adler flipped"):
            PN.decode_png(streams)


@pytest.mark.gpu
def test_graph_replay_over_the_capacity_skips_the_image():
    """md2_png_decode checks the capacity on the host; a replayed graph does not call it.  The kernels check it again:
    an image past the capacity the graph was captured with is skipped and flagged, the others decode."""
    from monodepth2_b200 import _capi
    lib = _capi.load_library()
    small = [PN.parse_png(write_png(_frame(k, 16, 20), f=k)) for k in (1, 2)]
    big = [small[0], PN.parse_png(pil_png(_frame(3, 375, 1242)))]
    hs, sb, rb, _ = _packed(small)
    hb, _, _, total = _packed(big)
    flat = torch.zeros(len(hb), dtype=torch.uint8, device="cuda")
    frames = torch.zeros(total, dtype=torch.uint8, device="cuda")
    status = torch.zeros(2, dtype=torch.int32, device="cuda")
    flat[:len(hs)].copy_(torch.from_numpy(hs))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        PN.run(lib, flat, hs.ctypes.data, 0, 2, frames, status, sb, rb)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        PN.run(lib, flat, hs.ctypes.data, 0, 2, frames, status, sb, rb)
    flat.copy_(torch.from_numpy(hb))
    g.replay()
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0, PN.CAPACITY]
    assert np.array_equal(frames[:small[0].nbytes].view(16, 20, 3).cpu().numpy(), _frame(1, 16, 20))


def _batches(root, names, fids, seeds):
    from monodepth2_b200.mono_batch import collate_native
    gpu, host = _GpuPng(root, names, fids), _HostPng(root, names, fids)
    out = []
    for seed in seeds:
        order = list(np.random.default_rng(seed).permutation(len(names)))
        random.seed(seed); torch.manual_seed(seed)
        a = collate_native([gpu[i] for i in order])
        random.seed(seed); torch.manual_seed(seed)
        b = collate_native([host[i] for i in order])
        out.append((a, b))
    return out


def _assert_same(got, want):
    assert sorted(map(str, got)) == sorted(map(str, want))
    for k, v in want.items():
        g = got[k]
        if v.dtype == torch.float32:
            g, v = g.view(torch.int32), v.view(torch.int32)
        assert torch.equal(g, v), k


MB_CASES = [((192, 640), [0, -1, 1]), ((320, 1024), [0, -1, 1, "s"])]


@pytest.mark.gpu
@pytest.mark.parametrize("case", MB_CASES, ids=lambda c: "%dx%d-%s" % (c[0][1], c[0][0], "".join(map(str, c[1]))))
def test_mono_batch_from_png_equals_from_native_frames(tmp_path, case):
    (H, W), fids = case
    sizes = S.KITTI_NATIVE_SIZES
    _write_png_drive(str(tmp_path), "d", lambda s, i: sizes[(i + (s == "r")) % len(sizes)], 4,
                     odd={("l", 3): "palette", ("r", 0): "jpeg"})
    names = ["d %d %s" % (i, s) for i in (1, 2) for s in "lr"]
    from monodepth2_b200.mono_batch import MonoBatch
    mb = MonoBatch(H, W, fids, 4)
    for a, b in _batches(str(tmp_path), names, fids, range(2)):
        assert a.png_jobs_offset >= 0 and a.jpeg_jobs_offset >= 0 and len(a.jpeg_copies) >= 1   # all three kinds
        got = mb(a)
        mb.check_png()
        mb.check_jpeg()
        _assert_same(got, mb(b))
        assert a.buffer.numel() < b.buffer.numel()


@pytest.mark.gpu
def test_mono_batch_with_velodyne_mixin(tmp_path):
    from monodepth2_b200.kitti_depth import VelodyneDepthMixin
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    import test_velo_depth as TV
    folders = TV._write_kitti_drive(str(tmp_path), 3)            # its frames are .png files

    class Raw(TV._KittiRaw):
        def get_image_path(self, folder, frame_index, side):
            return os.path.join(self.data_path, folder, "image_0%d" % self.side_map[side], "data", "%010d.png" % frame_index)

    class Gpu(VelodyneDepthMixin, PN.PngFramesMixin, NativeFramesMixin, Raw):
        pass

    class Host(VelodyneDepthMixin, NativeFramesMixin, Raw):
        pass
    names = ["%s %d %s" % (f, i, s) for f in folders for i in (1,) for s in "lr"]
    fids = [0, -1, 1]
    g, h = Gpu(str(tmp_path), names, fids), Host(str(tmp_path), names, fids)
    mb = MonoBatch(64, 96, fids, 2)
    random.seed(3); torch.manual_seed(3)
    a = collate_native([g[i] for i in range(len(names))])
    random.seed(3); torch.manual_seed(3)
    b = collate_native([h[i] for i in range(len(names))])
    assert a.png_jobs_offset >= 0
    _assert_same(mb(a), mb(b))
    mb.check_png()


@pytest.mark.gpu
def test_cuda_graph_replays_other_compressed_lengths_and_sizes(tmp_path):
    from monodepth2_b200.mono_batch import MonoBatch
    fids = [0, -1, "s"]
    roots = []
    for k, (lvl, sizes) in enumerate([(6, S.KITTI_NATIVE_SIZES[:3]), (1, S.KITTI_NATIVE_SIZES[2:]),
                                      (9, [(300, 1000), (375, 1242), (60, 100)])]):
        r = str(tmp_path / str(k))
        _write_png_drive(r, "d", lambda s, i, sizes=sizes: sizes[(i + (s == "r")) % len(sizes)], 3, level=lvl)
        roots.append(r)
    names = ["d %d %s" % (i, s) for i in (1,) for s in "lr"] + ["d 2 l"]
    pairs = [_batches(r, names, fids, [k])[0] for k, r in enumerate(roots)]
    natives = [a for a, _ in pairs]
    cap = tuple(max(v) for v in zip(*[(n.native_bytes, n.png_stream_bytes, n.png_raw_bytes) for n in natives]))
    mb = MonoBatch(32, 64, fids, 2, png_capacity=cap)
    eager = [{k: v.clone() for k, v in mb(n).items()} for n in natives]
    for (a, b), e in zip(pairs, eager):
        _assert_same(e, mb(b))
    assert len({n.buffer.numel() for n in natives}) == 3
    flat = torch.zeros(max(n.buffer.numel() for n in natives), dtype=torch.uint8, device="cuda")
    first = natives[0]
    flat[:first.buffer.numel()].copy_(first.buffer)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        mb.build(first, flat)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = mb.build(first, flat)
    for i, n in enumerate(natives[1:] + natives):
        flat.zero_()
        flat[:n.buffer.numel()].copy_(n.buffer)
        g.replay()
        torch.cuda.synchronize()
        want = eager[(i + 1) % len(natives)]
        for k, v in want.items():
            assert torch.equal(out[k].view(torch.int32) if v.dtype == torch.float32 else out[k],
                               v.view(torch.int32) if v.dtype == torch.float32 else v), (i, k)


@pytest.mark.gpu
def test_dataloader_with_workers_end_to_end(tmp_path):
    from torch.utils.data import DataLoader
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    _write_png_drive(str(tmp_path), "d", lambda s, i: S.KITTI_NATIVE_SIZES[i % 5], 6)
    names = ["d %d %s" % (i, s) for i in (1, 2, 3, 4) for s in "lr"]
    fids = [0, -1, 1]
    gpu, host = _GpuPng(str(tmp_path), names, fids), _HostPng(str(tmp_path), names, fids)
    mb = MonoBatch(96, 320, fids, 4)
    torch.manual_seed(0)
    loader = DataLoader(gpu, batch_size=4, shuffle=False, num_workers=2, pin_memory=True, collate_fn=collate_native)
    n = 0
    for native in loader:
        assert native.buffer.is_pinned() and native.png_jobs_offset >= 0
        got = mb(native)
        mb.check_png()
        items = []
        for b in range(native.batch_size):                      # the worker's draws, the host's frames
            it = host[n + b]
            it.update(do_flip=bool(native.do_flip[b]), do_color_aug=bool(native.do_color_aug[b]),
                      color_aug=native.color_aug[b])
            items.append(it)
        _assert_same(got, mb(collate_native(items)))
        n += native.batch_size
    assert n == len(names)
