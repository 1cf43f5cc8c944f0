"""Baseline JPEG decoding on the GPU (md2_jpeg_decode, monodepth2_b200/jpeg.py) against Pillow and oracle/jpeg_decode.py.

CPU: the oracle against Pillow, the parser's accept / decline rule and its fallback, unstuffing and the restart index
against a byte loop, a g++ build of md2_jpeg.h running the chunked self-synchronising decode (at the kernel's chunk
size and at one byte, which forces many resynchronisations) against the oracle's coefficients and Pillow's pixels, the
same build under AddressSanitizer on truncated and random-byte streams, the ABI's validation, the mixin's draws and
the ptxas log.  GPU: decode_jpeg byte-exact with Pillow on the corpus, MonoBatch fed by JPEG items equal to MonoBatch
fed by native frames, a CUDA graph over other batches, a two-worker DataLoader, and identical bytes run to run."""
import ctypes as C
import io
import os
import random
import re
import subprocess

import numpy as np
import pytest
import torch
from PIL import Image

from monodepth2_b200 import jpeg as JP
from monodepth2_b200 import synthetic as S
from monodepth2_b200.mono_batch import NativeFramesMixin
from oracle import jpeg_decode as OJ

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "monodepth2_b200", "csrc")
SMALL = [(1, 1), (2, 3), (8, 8), (15, 17), (16, 16), (17, 33), (31, 47)]


def _frame(seed, h, w):
    """Smooth colour fields plus noise, like a camera frame."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    base = np.stack([120 + 90 * np.sin(x / (17.0 + seed % 7) + c) * np.cos(y / 11.0 - c) for c in (0.0, 1.3, 2.6)], -1)
    return np.clip(base + rng.normal(0, 14, (h, w, 3)) + 15, 0, 255).astype(np.uint8)


def _content(kind, seed, h, w):
    if kind == "flat":                                            # every block all-EOB after its DC
        return np.full((h, w, 3), (seed * 37) % 256, np.uint8)
    if kind == "noise":                                           # long codes at q100
        return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    return _frame(seed, h, w)


def encode(a, fmt="JPEG", **kw):
    b = io.BytesIO()
    Image.fromarray(a).save(b, fmt, **kw)
    return b.getvalue()


def pil_rgb(data):
    return np.array(Image.open(io.BytesIO(data)).convert("RGB"))


OPTIONS = [{}, {"optimize": True}, {"restart_marker_blocks": 1}, {"restart_marker_blocks": 5},
           {"restart_marker_rows": 1}]


def corpus(sizes, kinds=("frame", "flat", "noise")):
    """(id, bytes) of every size x subsampling x quality x table / restart option x content, each content at one
    quality (noise at q100, where codes are longest)."""
    out = []
    for h, w in sizes:
        for ss in (0, 1, 2):
            for kind, q in (("frame", 50), ("frame", 92), ("flat", 92), ("noise", 100)):
                if kind not in kinds:
                    continue
                for k, opt in enumerate(OPTIONS):
                    if kind != "frame" and k not in (0, 2):
                        continue
                    d = encode(_content(kind, h * 31 + w + ss, h, w), quality=q, subsampling=ss, **opt)
                    out.append(("%dx%d-ss%d-q%d-%s-o%d" % (w, h, ss, q, kind, k), d))
    return out


# ------------------------------------------------------------------ CPU: the oracle and the parser
@pytest.mark.parametrize("size", SMALL + [(3, 40), (40, 3)], ids=lambda s: "%dx%d" % (s[1], s[0]))
def test_oracle_equals_pillow(size):
    for name, d in corpus([size]):
        assert np.array_equal(OJ.decode(d), pil_rgb(d)), name


def test_oracle_equals_pillow_kitti_size():
    for ss in (0, 2):
        d = encode(_frame(5, 375, 1242), quality=92, subsampling=ss)
        assert np.array_equal(OJ.decode(d), pil_rgb(d))


def _unsupported():
    a = _frame(1, 20, 30)
    cmyk = io.BytesIO()
    Image.fromarray(a).convert("CMYK").save(cmyk, "JPEG")
    return {"progressive": encode(a, progressive=True), "grayscale": encode(a[..., 0]), "cmyk": cmyk.getvalue(),
            "png": encode(a, "PNG")}


def test_parse_accepts_the_supported_class():
    for name, d in corpus(SMALL[:4], kinds=("frame",)):
        s = JP.parse_jpeg(d)
        assert s is not None, name
        assert (s.height, s.width) == pil_rgb(d).shape[:2]


@pytest.mark.parametrize("kind", ["progressive", "grayscale", "cmyk", "png"])
def test_parse_declines_the_rest_and_the_mixin_falls_back(tmp_path, kind):
    d = _unsupported()[kind]
    assert JP.parse_jpeg(d) is None
    ds = _GpuJpeg(str(tmp_path), ["d 1 l"], [0])
    p = tmp_path / "d" / "image_02" / "data" / "0000000001.jpg"
    p.parent.mkdir(parents=True)
    p.write_bytes(d)
    got = ds.native_color("d", 1, "l")
    assert isinstance(got, np.ndarray)
    assert np.array_equal(got, np.array(Image.open(io.BytesIO(d)).convert("RGB")))


def _byte_loop_unstuff(scan: bytes):
    """The entropy data of a scan read byte by byte as fill_bit_buffer / read_restart_marker do."""
    out, starts, rst, i = bytearray(), [0], [], 0
    while i < len(scan):
        c = scan[i]
        if c != 0xFF:
            out.append(c)
            i += 1
            continue
        j = i + 1
        while j < len(scan) and scan[j] == 0xFF:
            j += 1
        if j == len(scan):
            break
        if scan[j] == 0:
            out.append(0xFF)
            i = j + 1
        elif 0xD0 <= scan[j] <= 0xD7:
            starts.append(len(out))
            rst.append(scan[j] - 0xD0)
            i = j + 1
        else:
            break
    return bytes(out), starts, rst


def test_unstuff_and_restart_index_equal_a_byte_loop():
    rng = np.random.default_rng(0)
    cases = [d for _, d in corpus([(31, 47)], kinds=("noise", "frame"))]
    for _ in range(40):                                          # random scans rich in 0xFF, 0x00 and RSTn
        a = rng.choice(np.array([0x00, 0xFF, 0xD0, 0xD3, 0xD7, 0x12, 0xAB], np.uint8), 300)
        cases.append(b"\xff\xd8" + bytes(a) + b"\xff\xd9")
    for d in cases:
        scan = d[2:]
        if d[:2] == b"\xff\xd8" and JP.parse_jpeg(d) is not None:
            scan = OJ._segments(d)[-1][1] + b"\xff\xd9"
        data, starts, rst, _ = JP.unstuff(np.frombuffer(scan, np.uint8))
        want, wstarts, wrst = _byte_loop_unstuff(scan)
        assert bytes(data) == want and list(starts) == wstarts and list(rst) == wrst


# ------------------------------------------------------------------ CPU: md2_jpeg.h compiled with g++
@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("jpeg_host")
    so = d / "jh.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(ROOT, "tests", "jpeg", "md2_jpeg_host.cpp"), "-o", str(so)])
    return C.CDLL(str(so))


def _packed_one(s):
    body = JP._align(JP.JOB_DTYPE.itemsize, 64)
    h = np.zeros(body + JP.body_bytes([s]), np.uint8)
    JP.pack(h, 0, body, [s], [0])
    return h


def _host_decode(lib, d, chunk):
    s = JP.parse_jpeg(d)
    h = _packed_one(s)
    out = np.zeros(s.shape, np.uint8)
    coefs = np.zeros(s.n_blocks * 64, np.int16)
    rounds = C.c_int(0)
    st = lib.decode_host(h.ctypes.data_as(C.c_void_p), h.ctypes.data_as(C.c_void_p), chunk,
                         out.ctypes.data_as(C.c_void_p), coefs.ctypes.data_as(C.c_void_p), C.byref(rounds))
    return st, out, coefs.reshape(-1, 64), rounds.value


def _oracle_blocks(d):
    """The oracle's coefficients in the MCU-interleaved block order of the coefficient buffer."""
    info, coefs = OJ.decode_coefficients(d)
    my, mx = info["mcus"]
    out = []
    for r in range(my):
        for c in range(mx):
            for (cid, h, v, tq), cc in zip(info["comps"], coefs):
                for by in range(v):
                    for bx in range(h):
                        out.append(cc[r * v + by, c * h + bx])
    return np.stack(out)


@pytest.mark.parametrize("chunk", [64, 1], ids=["chunk64", "chunk1"])
def test_host_chunked_decode_equals_serial_and_pillow(host_lib, chunk):
    for name, d in corpus(SMALL):
        st, out, coefs, _ = _host_decode(host_lib, d, chunk)
        assert st == 0, name
        assert np.array_equal(coefs, _oracle_blocks(d)), name
        assert np.array_equal(out, pil_rgb(d)), name


@pytest.mark.parametrize("chunk", [64, 1], ids=["chunk64", "chunk1"])
def test_host_chunked_decode_kitti_size(host_lib, chunk):
    for size, ss, opt in (((375, 1242), 2, {}), ((370, 1224), 1, {"restart_marker_rows": 2})):
        d = encode(_frame(size[1], *size), quality=92, subsampling=ss, **opt)
        st, out, _, rounds = _host_decode(host_lib, d, chunk)
        assert st == 0 and np.array_equal(out, pil_rgb(d)) and rounds >= 2


def test_host_decode_of_corrupt_streams_stays_in_bounds(tmp_path):
    """AddressSanitizer build: truncated segments and random entropy bytes terminate, set the status word and touch
    nothing outside their buffers."""
    exe = tmp_path / "jh_asan"
    try:
        subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address", "-fno-omit-frame-pointer",
                               "-DMD2_JPEG_HOST_MAIN", "-I", CSRC, os.path.join(ROOT, "tests", "jpeg", "md2_jpeg_host.cpp"),
                               "-o", str(exe)], stderr=subprocess.DEVNULL)
    except subprocess.CalledProcessError:
        pytest.skip("g++ cannot build with AddressSanitizer here")
    rng = np.random.default_rng(7)
    good = [encode(_frame(3, 31, 47), quality=92, subsampling=2),
            encode(_frame(4, 40, 64), quality=100, subsampling=0, restart_marker_blocks=3)]
    flagged = 0
    for k in range(24):
        s = JP.parse_jpeg(good[k % 2])
        if k % 3 == 0:                                           # truncated: a segment loses its tail
            i = int(rng.integers(0, len(s.seg_bytes)))
            s.seg_bytes = s.seg_bytes.copy()
            s.seg_bytes[i] = int(rng.integers(0, s.seg_bytes[i]))
        else:                                                    # random bytes in place of the entropy data
            s.entropy = rng.integers(0, 256, len(s.entropy), dtype=np.uint8)
            if k % 3 == 2:
                s.entropy[:] = 0xFF
        h = _packed_one(s)
        path = tmp_path / ("s%d.bin" % k)
        path.write_bytes(h.tobytes())
        for chunk in (64, 3):
            r = subprocess.run([str(exe), str(path), str(chunk)], capture_output=True, text=True, timeout=120,
                               env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
            assert r.returncode == 0, r.stderr[-2000:]
            flagged += int(r.stdout.split()[0]) != 0
    assert flagged >= 40


# ------------------------------------------------------------------ CPU: ABI, layout, mixin, ptxas
def test_job_and_table_layout_matches_header(tmp_path):
    src = tmp_path / "job.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "md2_loss.h"', 'int main(void) {',
             'printf("job %zu\\n", sizeof(md2_jpeg_job));', 'printf("tables %zu\\n", sizeof(md2_jpeg_tables));',
             'printf("huff %zu\\n", sizeof(md2_jpeg_huff));', 'printf("segment %zu\\n", sizeof(md2_jpeg_segment));']
    lines += ['printf("%s %%zu\\n", offsetof(md2_jpeg_job, %s));' % (n, n) for n in JP.JOB_DTYPE.names]
    lines += ['printf("h.%s %%zu\\n", offsetof(md2_jpeg_huff, %s));' % (n, n) for n in JP.HUFF_DTYPE.names]
    lines += ['printf("t.%s %%zu\\n", offsetof(md2_jpeg_tables, %s));' % (n, n) for n in JP.TABLES_DTYPE.names]
    src.write_text("\n".join(lines + ['return 0; }']))
    exe = tmp_path / "job"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["job"]) == JP.JOB_DTYPE.itemsize and int(got["tables"]) == JP.TABLES_DTYPE.itemsize
    assert int(got["huff"]) == JP.HUFF_DTYPE.itemsize and int(got["segment"]) == JP.SEGMENT_DTYPE.itemsize
    for n in JP.JOB_DTYPE.names:
        assert int(got[n]) == JP.JOB_DTYPE.fields[n][1], n
    for n in JP.HUFF_DTYPE.names:
        assert int(got["h." + n]) == JP.HUFF_DTYPE.fields[n][1], n
    for n in JP.TABLES_DTYPE.names:
        assert int(got["t." + n]) == JP.TABLES_DTYPE.fields[n][1], n


@pytest.fixture(scope="module")
def lib():
    from monodepth2_b200 import _capi, build
    build.build()
    return _capi.load_library()


def _packed(streams):
    outs, total = [], 0
    for s in streams:
        outs.append(total)
        total = JP._align(total + s.nbytes)
    body = JP._align(len(streams) * JP.JOB_DTYPE.itemsize, 64)
    h = np.zeros(body + JP.body_bytes(streams), np.uint8)
    chunks, blocks = JP.pack(h, 0, body, streams, outs)
    return h, chunks, blocks, total


def test_jpeg_abi_validation_without_gpu(lib):
    n = C.c_size_t(0)
    assert lib.md2_jpeg_decode_scratch_bytes(0, 10, 10, C.byref(n)) == -1
    assert lib.md2_jpeg_decode_scratch_bytes(1, 0, 10, C.byref(n)) == -1
    assert lib.md2_jpeg_decode_scratch_bytes(1, 10, 0, C.byref(n)) == -1
    assert lib.md2_jpeg_decode_scratch_bytes(1, 10, 10, None) == -1
    streams = [JP.parse_jpeg(encode(_frame(k, 17, 33), quality=92, subsampling=2, restart_marker_blocks=k))
               for k in (0, 2)]
    h, chunks, blocks, total = _packed(streams)
    assert lib.md2_jpeg_decode_scratch_bytes(2, chunks, blocks, C.byref(n)) == 0
    need = n.value
    assert need >= blocks * 192
    dummy = np.zeros(64, np.uint8).ctypes.data

    def call(jobs=None, n_images=2, data_bytes=len(h), frames_bytes=total, max_chunks=chunks, max_blocks=blocks,
             scratch_bytes=need, data=h.ctypes.data, status=dummy):
        j = h[:2 * JP.JOB_DTYPE.itemsize].view(JP.JOB_DTYPE).copy() if jobs is None else jobs
        return lib.md2_jpeg_decode(data, data_bytes, j.ctypes.data, dummy, n_images, dummy, frames_bytes, status,
                                   max_chunks, max_blocks, dummy, scratch_bytes, None)

    def jobs(**kw):
        j = h[:2 * JP.JOB_DTYPE.itemsize].view(JP.JOB_DTYPE).copy()
        for k, v in kw.items():
            j[k][1] = v
        return j
    assert call(n_images=0) == -1 and call(data=None) == -1 and call(status=None) == -1
    assert call(max_chunks=0) == -1
    assert call(jobs(h_samp=1, v_samp=2)) == -2                       # 4:4:0 is not decoded here
    assert call(jobs(height=0)) == -1 and call(jobs(restart_interval=-1)) == -1
    assert call(jobs(dc_table=[0, 2, 0])) == -1 and call(jobs(quant_table=[0, 4, 1])) == -1
    assert call(jobs(n_segments=1)) == -1                              # not ceil(mcus / restart_interval)
    assert call(jobs(chunk_offset=0)) == -1 and call(jobs(block_offset=0)) == -1   # not the running sums
    assert call(jobs(entropy_offset=len(h))) == -1                     # the entropy area outside `data`
    assert call(jobs(tables_offset=4)) == -1                           # misaligned tables
    assert call(frames_bytes=total - 1) == -1 or call(frames_bytes=streams[0].nbytes) == -1
    assert call(max_chunks=chunks - 1) == -2 and call(max_blocks=blocks - 1) == -2   # over the capacity
    assert call(scratch_bytes=need - 1) == -3


class _JpegDataset:
    """The part of the reference's KITTIRAWDataset the mixins use, on .jpg files (pil_loader)."""

    def __init__(self, root, filenames, frame_idxs, is_train=True):
        from oracle import mono_batch as OM
        self.data_path, self.filenames, self.frame_idxs, self.is_train = root, filenames, frame_idxs, is_train
        self.brightness, self.contrast, self.saturation, self.hue = OM.BRIGHTNESS, OM.CONTRAST, OM.SATURATION, OM.HUE
        self.load_depth = False

    def __len__(self):
        return len(self.filenames)

    def get_image_path(self, folder, frame_index, side):
        return os.path.join(self.data_path, folder, "image_0%d" % {"l": 2, "r": 3}[side], "data",
                            "%010d.jpg" % frame_index)

    def get_color(self, folder, frame_index, side, do_flip):
        with open(self.get_image_path(folder, frame_index, side), "rb") as f:
            color = Image.open(f).convert("RGB")
        if do_flip:
            color = color.transpose(Image.FLIP_LEFT_RIGHT)
        return color


class _GpuJpeg(JP.JpegFramesMixin, NativeFramesMixin, _JpegDataset):
    pass


class _HostJpeg(NativeFramesMixin, _JpegDataset):
    pass


def _write_jpeg_drive(root, folder, size_of, n_frames, odd=None, quality=92, subsampling=2):
    """KITTI-like image_02 / image_03 .jpg frames; ``odd`` maps (side, index) to one of _unsupported()'s kinds."""
    for side, cam in (("l", 2), ("r", 3)):
        d = os.path.join(root, folder, "image_0%d" % cam, "data")
        os.makedirs(d, exist_ok=True)
        for i in range(n_frames):
            h, w = size_of(side, i)
            a = _frame(i * 2 + cam, h, w)
            kind = (odd or {}).get((side, i))
            if kind == "png":
                data = encode(a, "PNG")
            elif kind == "progressive":
                data = encode(a, quality=quality, progressive=True)
            else:
                data = encode(a, quality=quality, subsampling=subsampling, restart_marker_rows=(i % 3 == 1) * 2)
            with open(os.path.join(d, "%010d.jpg" % i), "wb") as f:
                f.write(data)


def test_mixin_makes_the_native_mixins_draws(tmp_path):
    pytest.importorskip("torchvision")
    _write_jpeg_drive(str(tmp_path), "d", lambda s, i: (30, 50), 4, odd={("r", 2): "png"})
    names = ["d 1 l", "d 2 r", "d 1 r"]
    gpu, host = _GpuJpeg(str(tmp_path), names, [0, -1, 1, "s"]), _HostJpeg(str(tmp_path), names, [0, -1, 1, "s"])
    kinds = set()
    for seed in range(12):
        random.seed(seed); torch.manual_seed(seed)
        a = gpu[seed % 3]
        after = (random.random(), float(torch.rand(1)))
        random.seed(seed); torch.manual_seed(seed)
        b = host[seed % 3]
        assert after == (random.random(), float(torch.rand(1)))
        assert (a["do_flip"], a["do_color_aug"], a["side"]) == (b["do_flip"], b["do_color_aug"], b["side"])
        assert (a["color_aug"] is None) == (b["color_aug"] is None)
        for f in b["frames"]:
            x = a["frames"][f]
            kinds.add(type(x).__name__)
            if isinstance(x, np.ndarray):
                assert np.array_equal(x, b["frames"][f])
            else:
                assert x.shape == b["frames"][f].shape and x.name.endswith(".jpg")
    assert kinds == {"JpegStream", "ndarray"}


def test_ptxas_reports_no_spills(lib):
    log = os.path.join(ROOT, "monodepth2_b200", "lib", "libmd2loss.md2_jpeg.cu.ptxas.log")
    txt = open(log).read()
    kernels = re.findall(r"Compiling entry function '\S*?\d(md2_jpeg_[a-z]+)E", txt)
    assert sorted(set(kernels)) == ["md2_jpeg_color", "md2_jpeg_huffman", "md2_jpeg_idct", "md2_jpeg_sync"]
    spills = re.findall(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", txt)
    assert len(spills) == 4 and all(s == ("0", "0", "0") for s in spills), spills


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_decode_jpeg_equals_pillow_one_per_call_and_mixed():
    items = corpus(SMALL) + [("kitti-%dx%d-ss%d" % (w, h, ss), encode(_frame(h + ss, h, w), quality=q, subsampling=ss))
                             for (h, w) in S.KITTI_NATIVE_SIZES for ss, q in ((2, 92), (1, 50), (0, 100))]
    wants = [pil_rgb(d) for _, d in items]
    for (name, d), want in zip(items, wants):
        got = JP.decode_jpeg([d])[0]
        assert np.array_equal(got.cpu().numpy(), want), name
    order = np.random.default_rng(0).permutation(len(items))
    got = JP.decode_jpeg([items[i][1] for i in order])
    for g, i in zip(got, order):
        assert np.array_equal(g.cpu().numpy(), wants[i]), items[i][0]
    again = JP.decode_jpeg([items[i][1] for i in order])
    assert all(torch.equal(a, b) for a, b in zip(got, again))


@pytest.mark.gpu
def test_decode_jpeg_reports_corrupt_data():
    d = encode(_frame(1, 64, 96), quality=92)
    s = JP.parse_jpeg(d, "cut.jpg")
    s.seg_bytes = s.seg_bytes // 3
    with pytest.raises(ValueError, match="cut.jpg"):
        JP.decode_jpeg([JP.parse_jpeg(d), s])


def _batches(root, names, fids, seeds):
    from monodepth2_b200.mono_batch import collate_native
    gpu, host = _GpuJpeg(root, names, fids), _HostJpeg(root, names, fids)
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
def test_mono_batch_from_jpeg_equals_from_native_frames(tmp_path, case):
    (H, W), fids = case
    sizes = S.KITTI_NATIVE_SIZES
    _write_jpeg_drive(str(tmp_path), "d", lambda s, i: sizes[(i + (s == "r")) % len(sizes)], 4,
                      odd={("l", 3): "png", ("r", 0): "progressive"})
    names = ["d %d %s" % (i, s) for i in (1, 2) for s in "lr"]
    from monodepth2_b200.mono_batch import MonoBatch
    mb = MonoBatch(H, W, fids, 4)
    for a, b in _batches(str(tmp_path), names, fids, range(2)):
        assert a.jpeg_jobs_offset >= 0 and len(a.jpeg_copies) >= 1          # one batch mixes both kinds of frame
        got = mb(a)
        mb.check_jpeg()
        _assert_same(got, mb(b))
        assert a.buffer.numel() < b.buffer.numel() / 3


@pytest.mark.gpu
def test_mono_batch_with_velodyne_mixin(tmp_path):
    from monodepth2_b200.kitti_depth import VelodyneDepthMixin
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    import test_velo_depth as TV
    folders = TV._write_kitti_drive(str(tmp_path), 3)
    for f in folders:                                           # the drive's frames as .jpg next to the .png
        for cam in (2, 3):
            d = os.path.join(str(tmp_path), f, "image_0%d" % cam, "data")
            for p in os.listdir(d):
                a = np.array(Image.open(os.path.join(d, p)).convert("RGB"))
                Image.fromarray(a).save(os.path.join(d, p.replace(".png", ".jpg")), quality=92)

    class Raw(TV._KittiRaw):
        def get_image_path(self, folder, frame_index, side):
            return os.path.join(self.data_path, folder, "image_0%d" % self.side_map[side], "data", "%010d.jpg" % frame_index)

        def get_color(self, folder, frame_index, side, do_flip):
            with open(self.get_image_path(folder, frame_index, side), "rb") as f:
                return Image.open(f).convert("RGB")

    class Gpu(VelodyneDepthMixin, JP.JpegFramesMixin, NativeFramesMixin, Raw):
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
    _assert_same(mb(a), mb(b))


@pytest.mark.gpu
def test_cuda_graph_replays_other_compressed_lengths_and_sizes(tmp_path):
    from monodepth2_b200.mono_batch import MonoBatch
    fids = [0, -1, "s"]
    roots = []
    for k, (q, sizes) in enumerate([(92, S.KITTI_NATIVE_SIZES[:3]), (100, S.KITTI_NATIVE_SIZES[2:]),
                                    (50, [(300, 1000), (375, 1242), (60, 100)])]):
        r = str(tmp_path / str(k))
        _write_jpeg_drive(r, "d", lambda s, i, sizes=sizes: sizes[(i + (s == "r")) % len(sizes)], 3, quality=q)
        roots.append(r)
    names = ["d %d %s" % (i, s) for i in (1,) for s in "lr"] + ["d 2 l"]
    pairs = [_batches(r, names, fids, [k])[0] for k, r in enumerate(roots)]
    natives = [a for a, _ in pairs]
    cap = tuple(max(v) for v in zip(*[(n.native_bytes, n.jpeg_chunks * JP.CHUNK_BYTES, n.jpeg_blocks) for n in natives]))
    mb = MonoBatch(32, 64, fids, 2, jpeg_capacity=cap)
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
    _write_jpeg_drive(str(tmp_path), "d", lambda s, i: S.KITTI_NATIVE_SIZES[i % 5], 6)
    names = ["d %d %s" % (i, s) for i in (1, 2, 3, 4) for s in "lr"]
    fids = [0, -1, 1]
    gpu, host = _GpuJpeg(str(tmp_path), names, fids), _HostJpeg(str(tmp_path), names, fids)
    mb = MonoBatch(96, 320, fids, 4)
    torch.manual_seed(0)
    loader = DataLoader(gpu, batch_size=4, shuffle=False, num_workers=2, pin_memory=True, collate_fn=collate_native)
    n = 0
    for native in loader:
        assert native.buffer.is_pinned() and native.jpeg_jobs_offset >= 0
        got = mb(native)
        mb.check_jpeg()
        items = []
        for b in range(native.batch_size):                      # the worker's draws, the host's frames
            it = host[n + b]
            it.update(do_flip=bool(native.do_flip[b]), do_color_aug=bool(native.do_color_aug[b]),
                      color_aug=native.color_aug[b])
            items.append(it)
        _assert_same(got, mb(collate_native(items)))
        n += native.batch_size
    assert n == len(names)
