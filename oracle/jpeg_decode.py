"""CPU restatement of Pillow's baseline JPEG decode (TEST INFRASTRUCTURE: only tests/ and benchmarks/ may import this).

The reference loads every training frame with ``pil_loader``, ``Image.open(f).convert("RGB")``.  For a baseline,
8-bit, Huffman-coded YCbCr JPEG the installed Pillow (12.2.0, libjpeg-turbo) runs integer arithmetic only:
jdhuff.c's sequential Huffman decode, jidctint.c's ``jpeg_idct_islow`` with ``prepare_range_limit_table``'s masked
range limit, jdsample.c's fancy h2v1 / h2v2 up-sampling (its SIMD form, which repeats the edge sample of a component
row; jdmainct.c's context rows, which repeat the first and last real row; plain replication for components at most
two samples wide, as jinit_upsampler chooses) and jdcolor.c's ``ycc_rgb_convert``
tables.  This module restates that chain serially in Python and numpy; tests/test_jpeg_decode.py pins it byte for byte
against the installed Pillow."""
import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                   7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                   39, 46, 53, 60, 61, 54, 47, 55, 62, 63], np.int64)     # jpeg_natural_order: zig-zag k -> natural


def _segments(data: bytes):
    """(marker, payload) for every marker segment up to SOS, then ("SOS", payload, entropy bytes up to EOI)."""
    assert data[:2] == b"\xff\xd8", "not a JPEG"
    p = 2
    out = []
    while True:
        while data[p] != 0xFF:
            p += 1
        while data[p] == 0xFF:
            p += 1
        m = data[p]
        p += 1
        n = (data[p] << 8) | data[p + 1]
        out.append((m, data[p + 2:p + n]))
        p += n
        if m == 0xDA:
            end = data.rfind(b"\xff\xd9")
            out.append(("scan", data[p:end if end >= p else len(data)]))
            return out


def _unstuff(scan: bytes):
    """The entropy-coded segments of a scan: 0xFF00 -> 0xFF, split at RSTn markers."""
    segs, cur, i = [], bytearray(), 0
    while i < len(scan):
        b = scan[i]
        if b == 0xFF and i + 1 < len(scan):
            nx = scan[i + 1]
            if nx == 0x00:
                cur.append(0xFF)
                i += 2
                continue
            if 0xD0 <= nx <= 0xD7:
                segs.append(bytes(cur))
                cur = bytearray()
                i += 2
                continue
            if nx == 0xFF:
                i += 1
                continue
            break
        cur.append(b)
        i += 1
    segs.append(bytes(cur))
    return segs


def _huff_table(payload):
    counts = list(payload[:16])
    vals = list(payload[16:16 + sum(counts)])
    maxcode, valptr, mincode = [-1] * 18, [0] * 17, [0] * 17
    code = k = 0
    for l in range(1, 17):
        if counts[l - 1]:
            valptr[l] = k
            mincode[l] = code
            code += counts[l - 1]
            k += counts[l - 1]
            maxcode[l] = code - 1
        code <<= 1
    maxcode[17] = 0xFFFFF
    return maxcode, valptr, mincode, vals


class _Bits:
    def __init__(self, seg: bytes):
        self.s = "".join(format(b, "08b") for b in seg)
        self.p = 0

    def get(self, n):
        """n bits (zeros past the end, as fill_bit_buffer supplies them)."""
        s = self.s[self.p:self.p + n]
        self.p += n
        return int(s.ljust(n, "0"), 2) if n else 0


def _decode_symbol(bits, t):
    maxcode, valptr, mincode, vals = t
    l, code = 1, bits.get(1)
    while code > maxcode[l]:
        code = (code << 1) | bits.get(1)
        l += 1
    if l > 16:
        return 0                                    # jpeg_huff_decode's fake zero
    return vals[valptr[l] + code - mincode[l]]


def _extend(v, s):
    return v - (1 << s) + 1 if v < (1 << (s - 1)) else v


def decode_coefficients(data: bytes):
    """Parses the stream and runs the Huffman decode: returns (info, coefs) where coefs[c] is an int16 array
    (blocks_y, blocks_x, 64) in natural order, not dequantised, of component c's padded plane."""
    q, dc, ac = {}, {}, {}
    restart = 0
    for m, pay in _segments(data):
        if m == 0xDB:
            p = 0
            while p < len(pay):
                pq, tq = pay[p] >> 4, pay[p] & 15
                n = 128 if pq else 64
                raw = np.frombuffer(pay[p + 1:p + 1 + n], ">u2" if pq else "u1").astype(np.int64)
                t = np.zeros(64, np.int64)
                t[ZIGZAG] = raw
                q[tq] = t
                p += 1 + n
        elif m == 0xC4:
            p = 0
            while p < len(pay):
                tc, th = pay[p] >> 4, pay[p] & 15
                n = 17 + sum(pay[p + 1:p + 17])
                (ac if tc else dc)[th] = _huff_table(pay[p + 1:p + n])
                p += n
        elif m == 0xC0:
            H, W = (pay[1] << 8) | pay[2], (pay[3] << 8) | pay[4]
            comps = [(pay[6 + 3 * i], pay[7 + 3 * i] >> 4, pay[7 + 3 * i] & 15, pay[8 + 3 * i]) for i in range(pay[5])]
        elif m == 0xDD:
            restart = (pay[0] << 8) | pay[1]
        elif m == 0xDA:
            sel = {pay[1 + 2 * i]: (pay[2 + 2 * i] >> 4, pay[2 + 2 * i] & 15) for i in range(pay[0])}
        elif m == "scan":
            scan = pay
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    mx, my = -(-W // (8 * hmax)), -(-H // (8 * vmax))
    coefs = [np.zeros((my * c[2], mx * c[1], 64), np.int16) for c in comps]
    segs = _unstuff(scan)
    n_mcu = mx * my
    per = restart if restart else n_mcu
    for s, seg in enumerate(segs):
        bits = _Bits(seg)
        last = [0] * len(comps)
        for m in range(s * per, min(n_mcu, (s + 1) * per)):
            r0, c0 = divmod(m, mx)
            for ci, (cid, h, v, tq) in enumerate(comps):
                tdc, tac = dc[sel[cid][0]], ac[sel[cid][1]]
                for by in range(v):
                    for bx in range(h):
                        blk = np.zeros(64, np.int64)
                        t = _decode_symbol(bits, tdc)
                        d = _extend(bits.get(t), t) if t else 0
                        last[ci] = (last[ci] + d + 2 ** 31) % 2 ** 32 - 2 ** 31
                        blk[0] = last[ci]
                        k = 1
                        while k < 64:
                            sym = _decode_symbol(bits, tac)
                            r, sz = sym >> 4, sym & 15
                            if sz:
                                k += r
                                blk[ZIGZAG[min(k, 63)]] = _extend(bits.get(sz), sz)
                            elif r != 15:
                                break
                            else:
                                k += 15
                            k += 1
                        coefs[ci][r0 * v + by, c0 * h + bx] = ((blk + 32768) % 65536 - 32768).astype(np.int16)
    info = dict(height=H, width=W, comps=comps, q=q, hmax=hmax, vmax=vmax, mcus=(my, mx))
    return info, coefs


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def range_limit(v):
    """idct_table[v & RANGE_MASK] of prepare_range_limit_table (8-bit samples)."""
    x = np.asarray(v, np.int64) & 1023
    return np.where(x < 128, x + 128, np.where(x < 512, 255, np.where(x < 896, 0, x - 896))).astype(np.uint8)


def _idct_1d(c0, c1, c2, c3, c4, c5, c6, c7, shift_even):
    z2, z3 = c2, c6
    z1 = (z2 + z3) * 4433
    tmp2 = z1 + z3 * -15137
    tmp3 = z1 + z2 * 6270
    tmp0 = (c0 + c4) << 13
    tmp1 = (c0 - c4) << 13
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    t0, t1, t2, t3 = c7, c5, c3, c1
    z1, z2, z3, z4 = t0 + t3, t1 + t2, t0 + t2, t1 + t3
    z5 = (z3 + z4) * 9633
    t0, t1, t2, t3 = t0 * 2446, t1 * 16819, t2 * 25172, t3 * 12299
    z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069, z4 * -3196
    z3 = z3 + z5
    z4 = z4 + z5
    t0 = t0 + z1 + z3
    t1 = t1 + z2 + z4
    t2 = t2 + z2 + z3
    t3 = t3 + z1 + z4
    n = shift_even
    return [_descale(t10 + t3, n), _descale(t11 + t2, n), _descale(t12 + t1, n), _descale(t13 + t0, n),
            _descale(t13 - t0, n), _descale(t12 - t1, n), _descale(t11 - t2, n), _descale(t10 - t3, n)]


def idct_islow(coef, qt):
    """jpeg_idct_islow on (..., 64) natural-order int16 blocks with a natural-order quant table -> (..., 8, 8) uint8."""
    d = coef.astype(np.int64) * qt                           # DEQUANTIZE
    d = d.reshape(coef.shape[:-1] + (8, 8))                  # [row u][col v]
    # pass 1: columns; a column whose AC terms are all zero is the DC << PASS1_BITS
    cols = [d[..., k, :] for k in range(8)]
    ac_zero = np.all(d[..., 1:, :] == 0, axis=-2)
    ws = _idct_1d(*cols, 13 - 2)
    ws = [np.where(ac_zero, cols[0] << 2, w) for w in ws]
    ws = np.stack(ws, axis=-2)                               # ws[..., row, col]
    # pass 2: rows; a row whose AC terms are all zero is range_limit(DESCALE(dc, PASS1_BITS + 3))
    rows = [ws[..., :, k] for k in range(8)]
    row_zero = np.all(ws[..., :, 1:] == 0, axis=-1)
    out = _idct_1d(*rows, 13 + 2 + 3)
    dcv = _descale(rows[0], 2 + 3)
    out = [np.where(row_zero, dcv, o) for o in out]
    return range_limit(np.stack(out, axis=-1))


def _planes(info, coefs):
    out = []
    for (cid, h, v, tq), c in zip(info["comps"], coefs):
        px = idct_islow(c, info["q"][tq])                    # (by, bx, 8, 8)
        by, bx = px.shape[:2]
        out.append(px.transpose(0, 2, 1, 3).reshape(by * 8, bx * 8))
    return out


def _fancy_h2(x, v2):
    """h2v1 (v2=False) or h2v2 (column sums given) fancy up-sampling of rows x, edges repeated."""
    left = np.concatenate([x[:, :1], x[:, :-1]], 1)
    right = np.concatenate([x[:, 1:], x[:, -1:]], 1)
    out = np.empty((x.shape[0], 2 * x.shape[1]), np.int64)
    if v2:
        out[:, 0::2] = (3 * x + left + 8) >> 4
        out[:, 1::2] = (3 * x + right + 7) >> 4
    else:
        out[:, 0::2] = (3 * x + left + 1) >> 2
        out[:, 1::2] = (3 * x + right + 2) >> 2
    return out


def upsample(plane, ch, cw, h, v):
    """A chroma plane's real (ch, cw) samples up-sampled by (v, h) in {1, 2} x {1, 2} (h >= v)."""
    x = plane[:ch, :cw].astype(np.int64)
    if h == 1 and v == 1:
        return x
    if cw <= 2:                                 # jinit_upsampler: fancy only for downsampled_width > 2, else replicate
        return np.repeat(np.repeat(x, v, 0), h, 1)
    if v == 1:
        return _fancy_h2(x, False)
    above = np.concatenate([x[:1], x[:-1]], 0)
    below = np.concatenate([x[1:], x[-1:]], 0)
    out = np.empty((2 * ch, 2 * cw), np.int64)
    out[0::2] = _fancy_h2(3 * x + above, True)
    out[1::2] = _fancy_h2(3 * x + below, True)
    return out


def ycc_to_rgb(y, cb, cr):
    """ycc_rgb_convert with build_ycc_rgb_table's tables."""
    i = np.arange(256, dtype=np.int64) - 128
    fix = lambda a: int(a * 65536 + 0.5)
    cr_r = (fix(1.40200) * i + 32768) >> 16
    cb_b = (fix(1.77200) * i + 32768) >> 16
    cr_g = -fix(0.71414) * i
    cb_g = -fix(0.34414) * i + 32768
    y = y.astype(np.int64)
    r = y + cr_r[cr]
    g = y + ((cb_g[cb] + cr_g[cr]) >> 16)
    b = y + cb_b[cb]
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)


def decode(data: bytes) -> np.ndarray:
    """np.array(Image.open(f).convert("RGB")) of a baseline 3-component YCbCr JPEG with 1x1 chroma."""
    info, coefs = decode_coefficients(data)
    H, W, hmax, vmax = info["height"], info["width"], info["hmax"], info["vmax"]
    planes = _planes(info, coefs)
    full = []
    for (cid, h, v, tq), p in zip(info["comps"], planes):
        ch, cw = -(-H * v // vmax), -(-W * h // hmax)
        full.append(upsample(p, ch, cw, hmax // h, vmax // v)[:H, :W])
    return ycc_to_rgb(*full)
