"""The training frames' JPEG files decoded on the GPU (md2_jpeg_decode), byte for byte what ``pil_loader`` gives.

The reference decodes every frame on the host with ``Image.open(f).convert("RGB")`` (Pillow's libjpeg-turbo).  Here a
dataloader worker only walks the file's markers (``parse_jpeg``: derived Huffman tables, quantisation tables, the
entropy-coded segments with stuffing and restart markers removed), ``collate_native`` packs the compressed streams,
and ``MonoBatch`` decodes them on the device into the native-frame buffer its batch builder reads.  A file outside the
supported class (progressive, arithmetic-coded, 12-bit, grayscale, CMYK or RGB, other samplings, PNG) is decoded on
the host by the dataset's own ``get_color``, as before (PNG files on the device, with ``png.PngFramesMixin`` in front).

    class GpuKITTIRAW(JpegFramesMixin, NativeFramesMixin, KITTIRAWDataset): pass
    loader = DataLoader(GpuKITTIRAW(...), ..., collate_fn=collate_native)

or, on its own, ``decode_jpeg([open(p, "rb").read() for p in paths])``.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _capi

CHUNK_BYTES = 64                                      # MD2_JPEG_CHUNK_BYTES
BAD_CODE, EXHAUSTED, BAD_INDEX, BAD_SEGMENT = 1, 2, 4, 8
HUFF_DTYPE = np.dtype([("look", "<u2", (256,)), ("maxcode", "<i4", (18,)), ("valoffset", "<i4", (18,)),
                       ("huffval", "u1", (256,))])     # md2_jpeg_huff
TABLES_DTYPE = np.dtype([("dc", HUFF_DTYPE, (2,)), ("ac", HUFF_DTYPE, (2,)), ("quant", "<u2", (4, 64))])
SEGMENT_DTYPE = np.dtype([("chunk", "<i4"), ("bytes", "<i4")])
JOB_DTYPE = np.dtype([("out_offset", "<i8"), ("entropy_offset", "<i8"), ("segments_offset", "<i8"),
                      ("tables_offset", "<i8"), ("block_offset", "<i8"), ("chunk_offset", "<i4"), ("n_chunks", "<i4"),
                      ("n_segments", "<i4"), ("restart_interval", "<i4"), ("height", "<i4"), ("width", "<i4"),
                      ("h_samp", "<i4"), ("v_samp", "<i4"), ("dc_table", "<i4", (3,)), ("ac_table", "<i4", (3,)),
                      ("quant_table", "<i4", (3,)), ("reserved", "<i4")])    # md2_jpeg_job
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                   7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                   39, 46, 53, 60, 61, 54, 47, 55, 62, 63], np.int64)
_SAMPLINGS = {(1, 1), (2, 1), (2, 2)}


def _align(n: int, a: int = 16) -> int:
    return (n + a - 1) // a * a


@dataclasses.dataclass
class JpegStream:
    """A parsed baseline JPEG: its size, luma sampling, restart interval, table ids per component, the
    ``TABLES_DTYPE`` record, and the entropy-coded segments (unstuffed, restart markers removed) as one uint8 array
    with each segment's start and length.  ``name`` is the file it came from, for error messages."""
    height: int
    width: int
    h_samp: int
    v_samp: int
    restart_interval: int
    dc_table: tuple
    ac_table: tuple
    quant_table: tuple
    tables: np.ndarray
    entropy: np.ndarray
    seg_start: np.ndarray
    seg_bytes: np.ndarray
    name: str = ""

    @property
    def shape(self) -> tuple:
        return (self.height, self.width, 3)

    @property
    def nbytes(self) -> int:                       # of the decoded frame
        return self.height * self.width * 3

    @property
    def n_blocks(self) -> int:
        mx = -(-self.width // (8 * self.h_samp))
        my = -(-self.height // (8 * self.v_samp))
        return mx * my * (self.h_samp * self.v_samp + 2)

    @property
    def seg_chunks(self) -> np.ndarray:
        return np.maximum(1, -(-self.seg_bytes // CHUNK_BYTES))

    @property
    def n_chunks(self) -> int:
        return int(self.seg_chunks.sum())


def derived_table(bits: Sequence[int], huffval: Sequence[int], is_dc: bool) -> Optional[np.ndarray]:
    """jpeg_make_d_derived_tbl as a HUFF_DTYPE record (lookahead entries of codes longer than 8 bits are 0), or None
    where libjpeg rejects the table."""
    bits = [0] + list(bits)
    huffsize, code, codes = [], 0, []
    for l in range(1, 17):
        huffsize += [l] * bits[l]
    if len(huffsize) > 256 or len(huffval) < len(huffsize):
        return None
    p, si = 0, huffsize[0] if huffsize else 0
    while p < len(huffsize):
        while p < len(huffsize) and huffsize[p] == si:
            codes.append(code)
            code += 1
            p += 1
        if code >= (1 << si):
            return None
        code <<= 1
        si += 1
    if is_dc and any(v > 15 for v in huffval[:len(huffsize)]):
        return None
    t = np.zeros((), HUFF_DTYPE)
    t["maxcode"][:] = -1
    t["maxcode"][17] = 0xFFFFF
    p = 0
    for l in range(1, 17):
        if bits[l]:
            t["valoffset"][l] = p - codes[p]
            p += bits[l]
            t["maxcode"][l] = codes[p - 1]
    t["huffval"][:len(huffsize)] = huffval[:len(huffsize)]
    p = 0
    for l in range(1, 9):
        for _ in range(bits[l]):
            look = codes[p] << (8 - l)
            t["look"][look:look + (1 << (8 - l))] = (l << 8) | huffval[p]
            p += 1
    return t


def unstuff(scan: np.ndarray):
    """The entropy-coded data of a scan (uint8 array from the first byte after SOS): returns (data with 0xFF00 ->
    0xFF, fill bytes and RSTn markers removed, the start of each segment in it, the RSTn numbers in order, the
    scan length consumed up to the marker that ends it)."""
    a = np.asarray(scan, np.uint8)
    ff = np.flatnonzero(a[:-1] == 0xFF)
    nxt = a[ff + 1]
    marker = (nxt != 0x00) & (nxt != 0xFF)
    rst = marker & (nxt >= 0xD0) & (nxt <= 0xD7)
    end_at = ff[marker & ~rst]
    end = int(end_at[0]) if end_at.size else len(a)
    keep = np.ones(end, bool)
    inside = ff < end
    ffi, nxi, rsti = ff[inside], nxt[inside], rst[inside]
    keep[ffi[nxi == 0xFF]] = False                              # fill bytes before a marker or a stuffed byte
    keep[ffi[nxi == 0x00] + 1] = False                          # stuffing
    keep[ffi[rsti]] = False
    keep[ffi[rsti] + 1] = False
    new_pos = np.cumsum(keep) - keep                            # index in the output of every input byte
    starts = np.concatenate([[0], new_pos[ffi[rsti]]]).astype(np.int64)
    return a[:end][keep], starts, (nxi[rsti] - 0xD0).astype(np.int64), end


def parse_jpeg(data: bytes, name: str = "") -> Optional[JpegStream]:
    """A ``JpegStream`` for a baseline 8-bit Huffman-coded three-component YCbCr JPEG with luma sampling 1x1, 2x1 or
    2x2 and chroma 1x1 (what ``md2_jpeg_decode`` decodes), None for anything else."""
    b = np.frombuffer(data, np.uint8)
    if len(b) < 4 or b[0] != 0xFF or b[1] != 0xD8:
        return None
    quant, dc, ac = {}, {}, {}
    jfif = adobe = False
    transform = -1
    restart = 0
    sof = None
    p = 2
    n = len(b)
    try:
        while True:
            if b[p] != 0xFF:
                return None
            while b[p] == 0xFF:
                p += 1
            m = int(b[p])
            p += 1
            if m == 0xD8 or m == 0xD9 or 0xD0 <= m <= 0xD7 or m == 0x01:
                return None
            ln = (int(b[p]) << 8) | int(b[p + 1])
            if ln < 2 or p + ln > n:
                return None
            pay = b[p + 2:p + ln]
            p += ln
            if m == 0xE0 and len(pay) >= 5 and bytes(pay[:5]) == b"JFIF\0":
                jfif = True
            elif m == 0xEE and len(pay) >= 12 and bytes(pay[:5]) == b"Adobe":
                adobe, transform = True, int(pay[11])
            elif 0xE0 <= m <= 0xEF or m == 0xFE:
                pass
            elif m == 0xDB:
                q = 0
                while q < len(pay):
                    pq, tq = int(pay[q]) >> 4, int(pay[q]) & 15
                    k = 128 if pq else 64
                    if pq > 1 or tq > 3 or q + 1 + k > len(pay):
                        return None
                    raw = pay[q + 1:q + 1 + k]
                    vals = raw.view(">u2").astype(np.int64) if pq else raw.astype(np.int64)
                    t = np.zeros(64, np.uint16)
                    t[ZIGZAG] = vals
                    quant[tq] = t
                    q += 1 + k
            elif m == 0xC4:
                q = 0
                while q < len(pay):
                    tc, th = int(pay[q]) >> 4, int(pay[q]) & 15
                    if q + 17 > len(pay):
                        return None
                    bits = [int(x) for x in pay[q + 1:q + 17]]
                    k = sum(bits)
                    if tc > 1 or th > 1 or q + 17 + k > len(pay):
                        return None
                    t = derived_table(bits, [int(x) for x in pay[q + 17:q + 17 + k]], tc == 0)
                    if t is None:
                        return None
                    (ac if tc else dc)[th] = t
                    q += 17 + k
            elif m == 0xDD:
                if len(pay) < 2:
                    return None
                restart = (int(pay[0]) << 8) | int(pay[1])
            elif m == 0xC0:
                if len(pay) < 15 or pay[0] != 8 or pay[5] != 3 or sof is not None:
                    return None
                H, W = (int(pay[1]) << 8) | int(pay[2]), (int(pay[3]) << 8) | int(pay[4])
                comps = [(int(pay[6 + 3 * i]), int(pay[7 + 3 * i]) >> 4, int(pay[7 + 3 * i]) & 15, int(pay[8 + 3 * i]))
                         for i in range(3)]
                if H == 0 or W == 0 or (comps[0][1], comps[0][2]) not in _SAMPLINGS:
                    return None
                if any((c[1], c[2]) != (1, 1) for c in comps[1:]) or any(c[3] > 3 for c in comps):
                    return None
                sof = (H, W, comps)
            elif m == 0xDA:
                break
            else:                                      # SOF1-15, DAC, DNL, DHP, EXP, JPGn, ...
                return None
        if sof is None:
            return None
        H, W, comps = sof
        if len(pay) != 1 + 2 * 3 + 3 or pay[0] != 3:
            return None
        ids = [int(pay[1 + 2 * i]) for i in range(3)]
        if ids != [c[0] for c in comps] or len(set(ids)) != 3:
            return None                                # the MCU's block order must be the frame's
        if (int(pay[7]), int(pay[8]), int(pay[9])) != (0, 63, 0):
            return None
        if not jfif and (adobe and transform == 0 or not adobe and ids == [82, 71, 66]):
            return None                                # libjpeg takes these for RGB
        dct = [int(pay[2 + 2 * i]) >> 4 for i in range(3)]
        act = [int(pay[2 + 2 * i]) & 15 for i in range(3)]
        if any(t not in dc for t in dct) or any(t not in ac for t in act) or any(c[3] not in quant for c in comps):
            return None
        ent, starts, rst, end = unstuff(b[p:])
        rest = b[p + end:]
        if len(rest) < 2 or rest[0] != 0xFF or int(rest[np.argmax(rest != 0xFF)]) != 0xD9:
            return None                                # another scan (or anything but EOI) follows
        hs, vs = comps[0][1], comps[0][2]
        mcus = -(-W // (8 * hs)) * -(-H // (8 * vs))
        n_seg = -(-mcus // restart) if restart else 1
        if len(starts) != n_seg or np.any(rst != np.arange(len(rst)) % 8):
            return None
    except IndexError:
        return None
    tables = np.zeros((), TABLES_DTYPE)
    for k, t in dc.items():
        tables["dc"][k] = t
    for k, t in ac.items():
        tables["ac"][k] = t
    for k, t in quant.items():
        tables["quant"][k] = t
    seg_bytes = np.diff(np.concatenate([starts, [len(ent)]])).astype(np.int64)
    return JpegStream(H, W, hs, vs, restart, tuple(dct), tuple(act), tuple(c[3] for c in comps), tables,
                      np.ascontiguousarray(ent), starts, seg_bytes, name)


# ------------------------------------------------------------------ packing
def body_bytes(streams: Sequence[JpegStream]) -> int:
    """Bytes ``pack`` writes from its ``body_off`` on."""
    n = 0
    for s in streams:
        n = _align(n + TABLES_DTYPE.itemsize, 64)
        n = _align(n + len(s.seg_bytes) * SEGMENT_DTYPE.itemsize, 64)
        n += s.n_chunks * CHUNK_BYTES
    return n


def pack(h: np.ndarray, jobs_off: int, body_off: int, streams: Sequence[JpegStream], out_offsets) -> tuple:
    """Writes the md2_jpeg_job table at ``jobs_off`` of the uint8 array ``h`` and every stream's tables, segment table
    and chunk-aligned entropy segments from ``body_off`` on (offsets count from the start of ``h``).  Image i decodes
    to byte ``out_offsets[i]`` of the frame buffer.  Returns (chunks, blocks) of the batch."""
    jobs = h[jobs_off:jobs_off + len(streams) * JOB_DTYPE.itemsize].view(JOB_DTYPE)
    off, chunks, blocks = body_off, 0, 0
    for i, s in enumerate(streams):
        tab = off
        h[tab:tab + TABLES_DTYPE.itemsize] = s.tables.reshape(1).view(np.uint8)
        off = _align(tab + TABLES_DTYPE.itemsize, 64)
        segs = np.zeros(len(s.seg_bytes), SEGMENT_DTYPE)
        sc = s.seg_chunks
        segs["chunk"] = np.cumsum(sc) - sc
        segs["bytes"] = s.seg_bytes
        seg_off = off
        h[seg_off:seg_off + segs.nbytes] = segs.view(np.uint8)
        off = _align(seg_off + segs.nbytes, 64)
        ent = off
        area = h[ent:ent + s.n_chunks * CHUNK_BYTES]
        area[:] = 0
        for c0, st, nb in zip(segs["chunk"], s.seg_start, s.seg_bytes):
            area[c0 * CHUNK_BYTES:c0 * CHUNK_BYTES + nb] = s.entropy[st:st + nb]
        off = ent + s.n_chunks * CHUNK_BYTES
        jobs[i] = (int(out_offsets[i]), ent, seg_off, tab, blocks, chunks, s.n_chunks, len(s.seg_bytes),
                   s.restart_interval, s.height, s.width, s.h_samp, s.v_samp, s.dc_table, s.ac_table, s.quant_table, 0)
        chunks += s.n_chunks
        blocks += s.n_blocks
    return chunks, blocks


def run(lib, flat: torch.Tensor, host_jobs: int, jobs_off: int, n: int, frames: torch.Tensor, status: torch.Tensor,
        max_chunks: int, max_blocks: int) -> None:
    """Enqueues md2_jpeg_decode on the current stream for ``n`` jobs at ``jobs_off`` of ``flat`` (the device copy of a
    packed buffer whose host job table is at address ``host_jobs``) into the device uint8 buffer ``frames``."""
    nb = C.c_size_t(0)
    _capi.check(lib, lib.md2_jpeg_decode_scratch_bytes(n, max_chunks, max_blocks, C.byref(nb)),
                "md2_jpeg_decode_scratch_bytes")
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=flat.device)
    base = flat.data_ptr()
    with torch.cuda.device(flat.device):
        st = lib.md2_jpeg_decode(base, flat.numel(), host_jobs, base + jobs_off, n, frames.data_ptr(), frames.numel(),
                                 status.data_ptr(), max_chunks, max_blocks, scratch.data_ptr(), scratch.numel(),
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _capi.check(lib, st, "md2_jpeg_decode")


def status_error(status: Sequence[int], names: Sequence[str]) -> Optional[str]:
    """A message naming every stream whose status word is set, or None."""
    what = {BAD_CODE: "bad Huffman code", EXHAUSTED: "data ended before the last MCU",
            BAD_INDEX: "coefficient index past 63", BAD_SEGMENT: "bad segment table"}
    bad = ["%s: %s" % (nm or "stream %d" % i, ", ".join(v for k, v in what.items() if int(s) & k))
           for i, (s, nm) in enumerate(zip(status, names)) if int(s)]
    return "corrupt JPEG data in " + "; ".join(bad) if bad else None


def decode_jpeg(streams: List[bytes], device=None) -> List[torch.Tensor]:
    """Decodes baseline JPEG files (their bytes) on the GPU into (h, w, 3) uint8 tensors, each equal to
    ``np.array(Image.open(f).convert("RGB"))``.  Raises ValueError for a stream ``parse_jpeg`` declines and for
    corrupt entropy data (this synchronises)."""
    parsed = []
    for i, d in enumerate(streams):
        s = d if isinstance(d, JpegStream) else parse_jpeg(d)
        if s is None:
            raise ValueError("stream %d is not a baseline YCbCr JPEG this decoder supports" % i)
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
    chunks, blocks = pack(buf.numpy(), 0, body, parsed, outs)
    dev = torch.device(device if device is not None else "cuda")
    flat = buf.to(dev, non_blocking=True)
    frames = torch.empty(total, dtype=torch.uint8, device=flat.device)
    status = torch.empty(n, dtype=torch.int32, device=flat.device)
    lib = _capi.load_library()
    run(lib, flat, buf.data_ptr(), 0, n, frames, status, chunks, blocks)
    err = status_error(status.cpu().tolist(), [s.name for s in parsed])
    if err:
        raise ValueError(err)
    return [frames[o:o + s.nbytes].view(s.height, s.width, 3) for o, s in zip(outs, parsed)]


class JpegFramesMixin:
    """Put in front of ``NativeFramesMixin``: ``class GpuKITTIRAW(JpegFramesMixin, NativeFramesMixin,
    KITTIRAWDataset)``.  Every frame the dataset's ``get_image_path`` names is read and parsed in the worker; its item
    carries the ``JpegStream`` instead of a decoded array, and ``MonoBatch`` decodes it on the device.  A file
    ``parse_jpeg`` declines is loaded by the dataset's own ``get_color``, as ``NativeFramesMixin`` does.  The random
    draws are ``NativeFramesMixin``'s, in the same order."""

    def native_color(self, folder, frame_index, side):
        path = self.get_image_path(folder, frame_index, side)
        with open(path, "rb") as f:
            s = parse_jpeg(f.read(), path)
        if s is not None:
            return s
        return super().native_color(folder, frame_index, side)
