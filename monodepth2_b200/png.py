"""The training frames' PNG files decoded on the GPU (md2_png_decode), byte for byte what ``pil_loader`` gives.

KITTI raw ships its frames as PNG, and the reference trains on them with ``--png``.  Pillow's decode of one 1242x375
frame is mostly zlib's inflate, about as long on one core as the whole GPU loss step.  Here a dataloader worker only
walks the file's chunks (``parse_png``: the header, the CRCs Pillow checks, the zlib header, the IDAT payloads joined
into one deflate stream; nothing is inflated), ``collate_native`` packs the streams, and ``MonoBatch`` decodes them on
the device into the native-frame buffer its batch builder reads.  A file outside the supported class (8-bit RGB
without interlace: palette, grey, alpha, 16-bit, Adam7, a preset dictionary, an unknown critical chunk, a bad CRC
before the image data, IDAT chunks that are not consecutive) is decoded on the host by the dataset's own
``get_color``, as before, so Pillow's behaviour and errors are kept for it.

    class GpuKITTIRAW(PngFramesMixin, JpegFramesMixin, NativeFramesMixin, KITTIRAWDataset): pass
    loader = DataLoader(GpuKITTIRAW(...), ..., collate_fn=collate_native)

or, on its own, ``decode_png([open(p, "rb").read() for p in paths])``.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import zlib
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _capi

BAD_CODE, DISTANCE, EXHAUSTED, BAD_FILTER, CHECKSUM, CAPACITY = 1, 2, 4, 8, 16, 32
MAX_SIDE = 16384                                       # MD2_PNG_MAX_SIDE
JOB_DTYPE = np.dtype([("out_offset", "<i8"), ("stream_offset", "<i8"), ("stream_index", "<i8"), ("raw_offset", "<i8"),
                      ("stream_bytes", "<i4"), ("height", "<i4"), ("width", "<i4"), ("reserved", "<i4")])  # md2_png_job
SIGNATURE = b"\x89PNG\r\n\x1a\n"
_KNOWN_CRITICAL = {b"IHDR", b"IDAT", b"IEND"}


def _align(n: int, a: int = 16) -> int:
    return (n + a - 1) // a * a


@dataclasses.dataclass
class PngStream:
    """A parsed 8-bit truecolour PNG: its size and its deflate data (the IDAT payloads joined, from the byte after the
    2-byte zlib header to the end of the last IDAT, so the Adler-32 trailer and anything after it included) as one
    uint8 array.  ``name`` is the file it came from, for error messages."""
    height: int
    width: int
    stream: np.ndarray
    name: str = ""

    @property
    def shape(self) -> tuple:
        return (self.height, self.width, 3)

    @property
    def nbytes(self) -> int:                       # of the decoded frame
        return self.height * self.width * 3

    @property
    def raw_bytes(self) -> int:                    # of the inflated data: a filter byte per row
        return self.height * (3 * self.width + 1)


def parse_png(data: bytes, name: str = "") -> Optional[PngStream]:
    """A ``PngStream`` for an 8-bit truecolour, non-interlaced PNG that Pillow opens (what ``md2_png_decode``
    decodes), None for anything else.  Chunks before the first IDAT must have good CRCs (Pillow checks those);
    ancillary chunks are ignored; IDAT CRCs are not checked, as Pillow does not check them."""
    b = memoryview(data)
    n = len(b)
    if n < 8 or bytes(b[:8]) != SIGNATURE:
        return None
    p, size, parts, idat_done = 8, None, [], False
    while True:
        if p + 12 > n:
            return None
        ln = int.from_bytes(b[p:p + 4], "big")
        cid = bytes(b[p + 4:p + 8])
        if ln > 0x7FFFFFFF or p + 12 + ln > n or not cid.isalpha():
            return None
        if cid == b"IDAT":
            if idat_done:
                return None                            # IDAT chunks must be consecutive
            parts.append(b[p + 8:p + 8 + ln])
        else:
            if parts:
                idat_done = True
            if not parts:                              # Pillow checks every CRC before the image data
                if zlib.crc32(b[p + 4:p + 8 + ln]) != int.from_bytes(b[p + 8 + ln:p + 12 + ln], "big"):
                    return None
            if size is None and cid != b"IHDR":
                return None
            if cid == b"IHDR":
                if size is not None or ln != 13:
                    return None
                w, h = int.from_bytes(b[p + 8:p + 12], "big"), int.from_bytes(b[p + 12:p + 16], "big")
                depth, ctype, comp, filt, interlace = bytes(b[p + 16:p + 21])
                if (depth, ctype, comp, filt, interlace) != (8, 2, 0, 0, 0):
                    return None
                if not (1 <= w <= MAX_SIDE and 1 <= h <= MAX_SIDE):
                    return None
                size = (h, w)
            elif cid == b"IEND":
                break
            elif not (cid[0] & 0x20) or cid in _KNOWN_CRITICAL:
                return None                            # PLTE, or an unknown critical chunk
        p += 12 + ln
    if size is None or not parts:
        return None
    z = np.concatenate([np.frombuffer(x, np.uint8) for x in parts]) if len(parts) > 1 else \
        np.frombuffer(parts[0], np.uint8)
    if len(z) < 2:
        return None
    cmf, flg = int(z[0]), int(z[1])
    if cmf & 15 != 8 or cmf >> 4 > 7 or (cmf * 256 + flg) % 31 or flg & 0x20:
        return None                                    # not deflate, a window over 32K, a bad FCHECK, a dictionary
    if len(z) - 2 > 1 << 28:
        return None
    return PngStream(size[0], size[1], z[2:], name)


# ------------------------------------------------------------------ packing
def body_bytes(streams: Sequence[PngStream]) -> int:
    """Bytes ``pack`` writes from its ``body_off`` on."""
    return sum(_align(len(s.stream), 64) for s in streams)


def pack(h: np.ndarray, jobs_off: int, body_off: int, streams: Sequence[PngStream], out_offsets) -> tuple:
    """Writes the md2_png_job table at ``jobs_off`` of the uint8 array ``h`` and every stream, 64-byte aligned, from
    ``body_off`` on (offsets count from the start of ``h``; ``body_off`` must be 64-byte aligned).  Image i decodes to
    byte ``out_offsets[i]`` of the frame buffer.  Returns (stream bytes, inflated bytes) of the batch."""
    jobs = h[jobs_off:jobs_off + len(streams) * JOB_DTYPE.itemsize].view(JOB_DTYPE)
    off, total, raw = body_off, 0, 0
    for i, s in enumerate(streams):
        nb = len(s.stream)
        h[off:off + nb] = s.stream
        h[off + nb:off + _align(nb, 64)] = 0
        jobs[i] = (int(out_offsets[i]), off, total, raw, nb, s.height, s.width, 0)
        off += _align(nb, 64)
        total += nb
        raw += s.raw_bytes
    return total, raw


def run(lib, flat: torch.Tensor, host_jobs: int, jobs_off: int, n: int, frames: torch.Tensor, status: torch.Tensor,
        max_stream_bytes: int, max_raw_bytes: int) -> None:
    """Enqueues md2_png_decode on the current stream for ``n`` jobs at ``jobs_off`` of ``flat`` (the device copy of a
    packed buffer whose host job table is at address ``host_jobs``) into the device uint8 buffer ``frames``."""
    nb = C.c_size_t(0)
    _capi.check(lib, lib.md2_png_decode_scratch_bytes(n, max_stream_bytes, max_raw_bytes, C.byref(nb)),
                "md2_png_decode_scratch_bytes")
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=flat.device)
    base = flat.data_ptr()
    with torch.cuda.device(flat.device):
        st = lib.md2_png_decode(base, flat.numel(), host_jobs, base + jobs_off, n, frames.data_ptr(), frames.numel(),
                                status.data_ptr(), max_stream_bytes, max_raw_bytes, scratch.data_ptr(), scratch.numel(),
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _capi.check(lib, st, "md2_png_decode")


def status_error(status: Sequence[int], names: Sequence[str]) -> Optional[str]:
    """A message naming every stream whose status word is set, or None."""
    what = {BAD_CODE: "invalid deflate data", DISTANCE: "distance too far back", EXHAUSTED: "data ended before the last row",
            BAD_FILTER: "unknown row filter", CHECKSUM: "Adler-32 mismatch",
            CAPACITY: "outside the decoder's capacity"}
    bad = ["%s: %s" % (nm or "stream %d" % i, ", ".join(v for k, v in what.items() if int(s) & k))
           for i, (s, nm) in enumerate(zip(status, names)) if int(s)]
    return "corrupt PNG data in " + "; ".join(bad) if bad else None


def decode_png(streams: List[bytes], device=None) -> List[torch.Tensor]:
    """Decodes 8-bit truecolour PNG files (their bytes) on the GPU into (h, w, 3) uint8 tensors, each equal to
    ``np.array(Image.open(f).convert("RGB"))``.  Raises ValueError for a stream ``parse_png`` declines and where
    Pillow raises on the image data (this synchronises)."""
    parsed = []
    for i, d in enumerate(streams):
        s = d if isinstance(d, PngStream) else parse_png(d)
        if s is None:
            raise ValueError("stream %d is not an 8-bit truecolour PNG this decoder supports" % i)
        parsed.append(s)
    if not parsed:
        return []
    n = len(parsed)
    outs, total = [], 0
    for s in parsed:
        outs.append(total)
        total = _align(total + s.nbytes)
    body = _align(n * JOB_DTYPE.itemsize, 64)
    buf = torch.empty(body + body_bytes(parsed), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    stream_bytes, raw_bytes = pack(buf.numpy(), 0, body, parsed, outs)
    dev = torch.device(device if device is not None else "cuda")
    flat = buf.to(dev, non_blocking=True)
    frames = torch.empty(total, dtype=torch.uint8, device=flat.device)
    status = torch.empty(n, dtype=torch.int32, device=flat.device)
    lib = _capi.load_library()
    run(lib, flat, buf.data_ptr(), 0, n, frames, status, max(1, stream_bytes), raw_bytes)
    err = status_error(status.cpu().tolist(), [s.name for s in parsed])
    if err:
        raise ValueError(err)
    return [frames[o:o + s.nbytes].view(s.height, s.width, 3) for o, s in zip(outs, parsed)]


class PngFramesMixin:
    """Put in front of ``NativeFramesMixin`` (and of ``JpegFramesMixin``, when both kinds of file may come):
    ``class GpuKITTIRAW(PngFramesMixin, JpegFramesMixin, NativeFramesMixin, KITTIRAWDataset)``.  Every frame the
    dataset's ``get_image_path`` names is read and parsed in the worker; its item carries the ``PngStream`` instead of
    a decoded array, and ``MonoBatch`` decodes it on the device.  A file ``parse_png`` declines goes to the next
    mixin's ``native_color``.  The random draws are ``NativeFramesMixin``'s, in the same order."""

    def native_color(self, folder, frame_index, side):
        path = self.get_image_path(folder, frame_index, side)
        with open(path, "rb") as f:
            s = parse_png(f.read(), path)
        if s is not None:
            return s
        return super().native_color(folder, frame_index, side)
