"""KITTI raw depth_gt on the GPU (md2_velo_depth, monodepth2_b200/kitti_depth.py) against oracle/kitti_depth.py.

CPU: the oracle against the reference's own generate_depth_map (when MD2_REFERENCE_DIR names a checkout) and against
scipy's resize calls, the g++ build of md2_velo.h against scipy.ndimage.zoom and numpy, the calibration helper, the job
layout, the dataset mixin, the packing and the ABI's validation.  GPU: byte-equal maps on exact-arithmetic scans (every
float64 product and sum exact, so summation order cannot matter), realistic scans within one float32 ulp, and
MonoBatch, a CUDA graph and a two-worker DataLoader end to end."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from monodepth2_b200 import synthetic as S
from monodepth2_b200.kitti_depth import VelodyneDepthMixin
from monodepth2_b200.mono_batch import NativeFramesMixin
from oracle import kitti_depth as OK

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = (375, 1242)
# a dyadic camera: P_rect_02 / P_rect_03 with R_rect_00 = I and a velodyne -> camera rotation of signed unit vectors
DYADIC_CAM = {"R_rect_00": [1, 0, 0, 0, 1, 0, 0, 0, 1],
              "P_rect_02": [512, 0, 640, 0, 0, 512, 192, 0, 0, 0, 1, 0],
              "P_rect_03": [512, 0, 608, -256, 0, 512, 176, 4, 0, 0, 1, 0]}
DYADIC_VELO = {"R": [0, -1, 0, 0, 0, -1, 1, 0, 0], "T": [0, 0, -2]}


def _dyadic_P(cam):
    Pr = np.array(DYADIC_CAM["P_rect_0%d" % cam], np.float64).reshape(3, 4)
    Rt = np.eye(4)
    Rt[:3, :3] = np.array(DYADIC_VELO["R"], np.float64).reshape(3, 3)
    Rt[:3, 3] = DYADIC_VELO["T"]
    return Pr @ Rt


# ------------------------------------------------------------------ exact-arithmetic scans
def _point(P, u, v, w):
    """The velodyne point that P maps to (u * w, v * w, w), exactly: P = [[a, b, 0, c], [d, 0, e, f], [1, 0, 0, g]]."""
    x = w - P[2, 3]
    y = (u * w - P[0, 0] * x - P[0, 3]) / P[0, 1]
    z = (v * w - P[1, 0] * x - P[1, 3]) / P[1, 2]
    p = np.array([x, y, z], np.float32)
    assert np.array_equal(p.astype(np.float64), [x, y, z]), (u, v, w)
    assert np.array_equal(P @ np.array([x, y, z, 1.0]), [u * w, v * w, w]), (u, v, w)
    return [x, y, z]


def exact_scan(seed, P, H, W):
    """Every case of the reference's rule on an (H, W) native image, in a shuffled scan order: several points per pixel
    (equal values too), the (r, W-1) / (r+1, 0) sub2ind collision in both orders with several points on each side,
    u / v exactly on .5, w < 0 and w == 0, x < 0 (and -0.0), NaN rows and points outside the image."""
    rng = np.random.default_rng(seed)
    depth = lambda: float(rng.integers(1, 480)) / 8
    off = [-0.5, -0.25, 0.0, 0.25, 0.5]
    loose = []
    for _ in range(400):                                         # pixels holding 1-4 points, anywhere
        r, c = int(rng.integers(0, H)), int(rng.integers(0, W))
        ws = [depth() for _ in range(int(rng.integers(1, 5)))]
        if rng.random() < 0.2:
            ws.append(ws[0])
        for w in ws:
            loose.append(_point(P, c + 1 + rng.choice(off), r + 1 + rng.choice(off), w))
    for c in (0, W - 1):                                         # the first and last columns, ties and all
        for r in rng.integers(0, H, 20):
            loose.append(_point(P, c + 1 + rng.choice(off), int(r) + 1 + rng.choice(off), depth()))
    for u, v in ((0.25, 10), (W + 0.75, 10), (10, -3.0), (10, H + 1.75), (-40.0, -40.0), (W + 300.0, H + 200.0)):
        loose.append(_point(P, u, v, depth()))                   # outside
    for _ in range(30):                                          # landing with w < 0: stored, then clamped to 0
        loose.append(_point(P, int(rng.integers(1, W + 1)), int(rng.integers(1, H + 1)), -float(rng.integers(1, 16)) / 8))
    loose += [[2.0, 1.0, 1.0], [2.0, 0.0, 0.0], [-1.0, 3.0, 0.5], [-0.0, 0.5, 0.5], [np.nan, 0, 0], [1.0, np.nan, 0],
              [4.0, 0.0, np.nan], [np.inf, 0.0, 0.0]]            # w == 0, x < 0, x = -0.0, NaN, inf
    loose = [loose[i] for i in rng.permutation(len(loose))]
    chunks = []
    for k, r in enumerate(list(rng.integers(0, H - 1, 24)) + [H - 1, 0]):    # (r, W-1) ~ (r+1, 0); H-1 has no partner
        r = int(r)
        a = [_point(P, W, r + 1, depth()) for _ in range(int(rng.integers(1, 4)))]
        b = [_point(P, 1, r + 2, depth()) for _ in range(int(rng.integers(1, 4)))] if r + 1 < H else []
        if k % 3 == 0:
            chunks.append(a + b)
        elif k % 3 == 1:
            chunks.append(b + a)
        else:
            chunks.append([p for pair in zip(a, b) for p in pair] + a[len(b):] + b[len(a):])
    for ch in chunks:                                            # each collision group spread over the scan
        pos = np.sort(rng.integers(0, len(loose) + 1, len(ch)))[::-1]
        for p, q in zip(pos, ch[::-1]):
            loose.insert(int(p), q)
    scan = np.array(loose, np.float32)
    return np.concatenate([scan, rng.uniform(0, 1, (len(scan), 1)).astype(np.float32)], 1)


def oracle_depth_gt(scan, P, im_shape, out_shape, flip, vel_depth=False):
    """get_depth from a scan in memory, as MonoDataset.__getitem__ stores it: (1, h, w) float32."""
    velo = scan.copy()
    velo[:, 3] = 1.0                                             # load_velodyne_points
    d = OK.depth_from_points(velo, P, np.array(im_shape, np.int32), vel_depth)
    d = OK.resize_nearest(d, out_shape)
    if flip:
        d = np.fliplr(d)
    return np.expand_dims(d, 0).astype(np.float32)


# ------------------------------------------------------------------ CPU: the oracle
def _reference_module(name):
    ref = os.environ.get("MD2_REFERENCE_DIR", "")
    if not ref or not os.path.exists(os.path.join(ref, "kitti_utils.py")):
        pytest.skip("MD2_REFERENCE_DIR does not name a checkout of the reference")
    sys.path.insert(0, ref)
    try:
        import importlib
        return importlib.import_module(name)
    finally:
        sys.path.remove(ref)


def _write_scan(path, scan):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    scan.astype(np.float32).tofile(path)


@pytest.mark.parametrize("cam", [2, 3])
@pytest.mark.parametrize("vel_depth", [False, True])
def test_oracle_equals_reference_generate_depth_map(tmp_path, monkeypatch, cam, vel_depth):
    kitti_utils = _reference_module("kitti_utils")
    monkeypatch.setattr(np, "int", int, raising=False)
    S.write_kitti_calibration(str(tmp_path / "calib"), (370, 1226))
    for seed in range(2):
        velo = str(tmp_path / ("%d.bin" % seed))
        _write_scan(velo, S.velodyne_scan(seed))
        want = kitti_utils.generate_depth_map(str(tmp_path / "calib"), velo, cam, vel_depth)
        got = OK.generate_depth_map(str(tmp_path / "calib"), velo, cam, vel_depth)
        assert np.array_equal(got.view(np.int64), want.view(np.int64))


@pytest.mark.parametrize("native", S.KITTI_NATIVE_SIZES + [(300, 1000), (375, 1242)])
def test_oracle_resize_is_skimages_scipy_call(native):
    """resize_nearest against the ndimage calls skimage.transform.resize(order=0, mode='constant') makes (and against
    skimage itself where it is installed): below a factor of 1.25 the anti-aliasing filter is the identity, and the
    map is a gather of native pixels."""
    from scipy import ndimage as ndi
    rng = np.random.default_rng(native[0] + native[1])
    img = np.where(rng.random(native) < 0.1, rng.uniform(0.5, 80, native), 0.0)
    factors = np.divide(native, OUT)
    sigma = np.maximum(0, (factors - 1) / 2)
    assert np.array_equal(ndi.gaussian_filter(img, sigma, cval=0, mode="grid-constant"), img)
    want = ndi.zoom(img, [1 / f for f in factors], order=0, mode="grid-constant", cval=0, grid_mode=True)
    got = OK.resize_nearest(img, OUT)
    assert np.array_equal(got, want)
    try:
        from skimage.transform import resize
    except ImportError:
        return
    assert np.array_equal(got, resize(img, OUT, order=0, preserve_range=True, mode="constant"))


# ------------------------------------------------------------------ CPU: md2_velo.h compiled with g++
SHIM = r"""
#include "md2_velo.h"
extern "C" void nearest_axis(int n_in, int n_out, int* out) {
  for (int o = 0; o < n_out; ++o) out[o] = md2_velo_nearest_src(o, n_in, n_out);
}
extern "C" void project(const double* P, const float* pts, int n, int h, int w, int vel, int* row, int* col, double* val) {
  for (int i = 0; i < n; ++i)
    if (!md2_velo_project(P, pts[4 * i], pts[4 * i + 1], pts[4 * i + 2], h, w, vel, row + i, col + i, val + i)) row[i] = -1;
}
"""


@pytest.fixture(scope="module")
def host_rule(tmp_path_factory):
    d = tmp_path_factory.mktemp("velo_rule")
    (d / "shim.cpp").write_text(SHIM)
    so = d / "shim.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-I",
                           os.path.join(ROOT, "monodepth2_b200", "csrc"), str(d / "shim.cpp"), "-o", str(so)])
    return C.CDLL(str(so))


def test_nearest_index_rule_equals_ndimage_zoom(host_rule):
    """Every input size from n_out / 4 to 1.25 n_out, for both axes of 375x1242, including the exact .5 ties."""
    from scipy import ndimage as ndi
    for n_out in OUT:
        for n_in in range(n_out // 4, (5 * n_out - 1) // 4 + 1):
            idx = np.empty(n_out, np.int32)
            host_rule.nearest_axis(n_in, n_out, idx.ctypes.data_as(C.c_void_p))
            ramp = np.arange(1, n_in + 1, dtype=np.float64)
            want = ndi.zoom(ramp, n_out / n_in, order=0, mode="grid-constant", cval=0, grid_mode=True)
            got = np.where(idx >= 0, ramp[np.maximum(idx, 0)], 0.0)
            assert np.array_equal(got, want), (n_in, n_out, np.nonzero(got != want)[0][:4])


def _host_project(lib, P, scan, H, W, vel):
    n = len(scan)
    row, col, val = np.empty(n, np.int32), np.empty(n, np.int32), np.empty(n, np.float64)
    pts = np.ascontiguousarray(scan, np.float32)
    Pc = np.ascontiguousarray(P, np.float64)
    lib.project(Pc.ctypes.data_as(C.c_void_p), pts.ctypes.data_as(C.c_void_p), n, H, W, int(vel),
                row.ctypes.data_as(C.c_void_p), col.ctypes.data_as(C.c_void_p), val.ctypes.data_as(C.c_void_p))
    return row, col, val


def _numpy_project(P, scan, H, W, vel):
    """generate_depth_map's projection and bounds test per point, scan order kept (-1: dropped)."""
    velo = scan.copy()
    velo[:, 3] = 1.0
    with np.errstate(all="ignore"):
        im = np.dot(P, velo.T).T
        im[:, :2] = im[:, :2] / im[:, 2][..., None]
    if vel:
        im[:, 2] = velo[:, 0]
    c, r = np.round(im[:, 0]) - 1, np.round(im[:, 1]) - 1
    ok = (velo[:, 0] >= 0) & (c >= 0) & (r >= 0) & (c < W) & (r < H)
    return np.where(ok, r, -1).astype(np.int32), np.where(ok, c, -1).astype(np.int32), im[:, 2], im[:, :2]


@pytest.mark.parametrize("vel", [False, True])
def test_host_projection_equals_numpy(host_rule, kitti_calib, vel):
    for cam in (2, 3):
        P = _dyadic_P(cam)
        scan = exact_scan(cam, P, 375, 1242)
        r, c, v = _host_project(host_rule, P, scan, 375, 1242, vel)
        wr, wc, wv, _ = _numpy_project(P, scan, 375, 1242, vel)
        assert np.array_equal(r, wr) and np.array_equal(c[r >= 0], wc[r >= 0])
        assert np.array_equal(v[r >= 0], wv[r >= 0])
    P, _ = OK.velo_to_image(kitti_calib(), 2)
    scan = S.velodyne_scan(3)
    r, c, v = _host_project(host_rule, P, scan, 375, 1242, vel)
    wr, wc, wv, uv = _numpy_project(P, scan, 375, 1242, vel)
    assert _boundary_points(uv, scan) == 0
    assert np.array_equal(r, wr) and np.array_equal(c[r >= 0], wc[r >= 0]) and np.count_nonzero(r >= 0) > 10000
    assert np.all(np.abs(v[r >= 0] - wv[r >= 0]) <= 4e-16 * np.abs(wv[r >= 0]))


def _boundary_points(uv, scan, eps=1e-9):
    """Points x >= 0 whose u or v lies within eps px of a rounding boundary: there the order of the float64 sums
    (numpy's BLAS or the kernel's) may decide the pixel."""
    with np.errstate(invalid="ignore"):
        frac = np.abs(uv - np.floor(uv) - 0.5)
        return int(np.sum((scan[:, 0] >= 0) & np.any(frac < eps, axis=1)))


@pytest.fixture(scope="module")
def kitti_calib(tmp_path_factory):
    """im_shape -> a directory holding KITTI's 2011_09_26 calibration with that S_rect_02."""
    dirs = {}

    def get(im_shape=(375, 1242)):
        if im_shape not in dirs:
            dirs[im_shape] = str(tmp_path_factory.mktemp("calib_%dx%d" % im_shape))
            S.write_kitti_calibration(dirs[im_shape], im_shape)
        return dirs[im_shape]
    return get


# ------------------------------------------------------------------ CPU: calibration, layout, mixin, packing, ABI
@pytest.mark.parametrize("cam", [2, 3])
def test_calibration_files_give_the_oracles_P(tmp_path, cam):
    from monodepth2_b200.kitti_depth import velo_to_image
    for k, (shape, cc, vc) in enumerate([((370, 1224), None, None), ((375, 1242), DYADIC_CAM, DYADIC_VELO)]):
        d = str(tmp_path / str(k))
        S.write_kitti_calibration(d, shape, cc, vc)
        P, im_shape = velo_to_image(d, cam)
        want_P, want_shape = OK.velo_to_image(d, cam)
        assert im_shape == tuple(want_shape) == shape
        assert P.dtype == np.float64 and np.array_equal(P.view(np.int64), want_P.view(np.int64))
        if cc is DYADIC_CAM:
            assert np.array_equal(P, _dyadic_P(cam))
        assert velo_to_image(d, cam) is velo_to_image(d, cam)          # cached


def test_job_layout_matches_header(tmp_path):
    from monodepth2_b200.kitti_depth import VELO_JOB_DTYPE
    src = tmp_path / "job.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "md2_loss.h"', 'int main(void) {',
             'printf("sizeof %zu\\n", sizeof(md2_velo_job));']
    lines += ['printf("%s %%zu\\n", offsetof(md2_velo_job, %s));' % (n, n) for n in VELO_JOB_DTYPE.names]
    src.write_text("\n".join(lines + ['return 0; }']))
    exe = tmp_path / "job"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["sizeof"]) == VELO_JOB_DTYPE.itemsize == 128
    for n in VELO_JOB_DTYPE.names:
        assert int(got[n]) == VELO_JOB_DTYPE.fields[n][1], n


DATES = {"2011_09_26": (375, 1242), "2011_09_28": (370, 1224)}


def _write_kitti_drive(root, n_frames=4, frame_size=(60, 100)):
    """A KITTI raw layout with dyadic calibrations: <date>/calib_*.txt, <date>/<drive>/image_0{2,3}/data/*.png and
    velodyne_points/data/*.bin with exact-arithmetic scans for the left camera."""
    from PIL import Image
    folders = []
    for date, shape in DATES.items():
        S.write_kitti_calibration(os.path.join(root, date), shape, DYADIC_CAM, DYADIC_VELO)
        folder = "%s/%s_drive_0001_sync" % (date, date)
        folders.append(folder)
        for i in range(n_frames):
            for cam in (2, 3):
                d = os.path.join(root, folder, "image_0%d" % cam, "data")
                os.makedirs(d, exist_ok=True)
                rng = np.random.default_rng(i * 10 + cam)
                Image.fromarray(rng.integers(0, 256, frame_size + (3,), dtype=np.uint8)).save(
                    os.path.join(d, "%010d.png" % i))
            _write_scan(os.path.join(root, folder, "velodyne_points", "data", "%010d.bin" % i),
                        exact_scan(100 + i + len(folders), _dyadic_P(2), *shape))
    return folders


class _KittiRaw:
    """The part of the reference's KITTIRAWDataset NativeFramesMixin and VelodyneDepthMixin use; get_depth is the
    oracle's restatement of KITTIRAWDataset.get_depth."""
    full_res_shape = (1242, 375)
    side_map = {"2": 2, "3": 3, "l": 2, "r": 3}

    def __init__(self, root, filenames, frame_idxs, is_train=True):
        from oracle import mono_batch as OM
        self.data_path, self.filenames, self.frame_idxs, self.is_train = root, filenames, frame_idxs, is_train
        self.brightness, self.contrast, self.saturation, self.hue = OM.BRIGHTNESS, OM.CONTRAST, OM.SATURATION, OM.HUE
        self.load_depth = True

    def __len__(self):
        return len(self.filenames)

    def get_color(self, folder, frame_index, side, do_flip):
        from PIL import Image
        p = os.path.join(self.data_path, folder, "image_0%d" % self.side_map[side], "data", "%010d.png" % frame_index)
        with open(p, "rb") as f:
            color = Image.open(f).convert("RGB")
        if do_flip:
            color = color.transpose(Image.FLIP_LEFT_RIGHT)
        return color

    def get_depth(self, folder, frame_index, side, do_flip):
        return OK.get_depth(self.data_path, folder, frame_index, side, do_flip)


class _HostDepth(NativeFramesMixin, _KittiRaw):
    pass


class _GpuDepth(VelodyneDepthMixin, NativeFramesMixin, _KittiRaw):
    pass


def _datasets(root, names, fids):
    return _GpuDepth(root, names, fids), _HostDepth(root, names, fids)


def test_mixin_items_carry_the_scan_and_the_same_draws(tmp_path):
    pytest.importorskip("torchvision")
    folders = _write_kitti_drive(str(tmp_path), 3)
    names = ["%s %d %s" % (f, i, s) for f in folders for i in (1,) for s in "lr"]
    gpu, host = _datasets(str(tmp_path), names, [0, -1, 1])
    for seed in range(8):
        random.seed(seed); torch.manual_seed(seed)
        a = gpu[seed % len(names)]
        after = (random.random(), float(torch.rand(1)))
        random.seed(seed); torch.manual_seed(seed)
        b = host[seed % len(names)]
        assert after == (random.random(), float(torch.rand(1)))
        assert "depth_gt" not in a and "velodyne" not in b
        assert (a["do_flip"], a["do_color_aug"], a["side"]) == (b["do_flip"], b["do_color_aug"], b["side"])
        folder, fi, side = names[seed % len(names)].split()
        v = a["velodyne"]
        P, im_shape = OK.velo_to_image(os.path.join(str(tmp_path), folder.split("/")[0]), OK.SIDE_MAP[side])
        raw = np.fromfile(os.path.join(str(tmp_path), folder, "velodyne_points/data/%010d.bin" % int(fi)), np.float32)
        assert np.array_equal(v.scan.reshape(-1).view(np.int32), raw.view(np.int32))
        assert np.array_equal(v.P, P) and tuple(v.im_shape) == tuple(im_shape) and tuple(v.out_shape) == OUT


def test_collate_native_packs_scans_and_jobs():
    from monodepth2_b200.kitti_depth import VELO_JOB_DTYPE, VeloScan
    from monodepth2_b200.mono_batch import collate_native
    items = []
    for b in range(3):
        scan = S.velodyne_scan(b, n_azimuth=7 + b, n_beams=5)
        items.append({"frames": {0: np.full((6, 8, 3), b, np.uint8)}, "do_color_aug": False, "do_flip": b == 1,
                      "color_aug": None, "side": "l", "velodyne": VeloScan(scan, _dyadic_P(2 + b % 2), (370 + b, 1224))})
    nb = collate_native(items, pin_memory=False)
    assert nb.velo_jobs_offset % 16 == 0 and nb.velo_out_shape == OUT and nb.extra == {}
    h = nb.buffer.numpy()
    jobs = h[nb.velo_jobs_offset:nb.velo_jobs_offset + 3 * VELO_JOB_DTYPE.itemsize].view(VELO_JOB_DTYPE)
    for b, it in enumerate(items):
        j = jobs[b]
        assert np.array_equal(j["P"], it["velodyne"].P.reshape(-1))
        assert (j["n_points"], j["height"], j["width"], j["flip"], j["vel_depth"]) == (35 + 5 * b, 370 + b, 1224,
                                                                                       int(b == 1), 0)
        a = int(j["offset"])
        assert a % 16 == 0 and a > nb.frames_offset
        assert np.array_equal(h[a:a + 16 * int(j["n_points"])].view(np.float32).reshape(-1, 4).view(np.int32),
                              it["velodyne"].scan.view(np.int32))
    assert np.array_equal(nb.jobs()["height"], [6, 6, 6])       # the frame jobs are where they were
    other = [dict(it, frames={0: np.zeros((9 + b, 30, 3), np.uint8)},
                  velodyne=VeloScan(it["velodyne"].scan[:b + 1], it["velodyne"].P, (375, 1242))) for b, it in enumerate(items)]
    nb2 = collate_native(other, pin_memory=False)
    assert nb2.buffer.numel() != nb.buffer.numel()
    # every table's place depends on the batch size and the frame ids alone, so one CUDA graph serves both batches
    assert (nb2.velo_jobs_offset, nb2.jobs_offset, nb2.frames_offset) == (nb.velo_jobs_offset, nb.jobs_offset,
                                                                          nb.frames_offset)
    assert nb.velo_jobs_offset + 3 * VELO_JOB_DTYPE.itemsize <= nb.frames_offset


@pytest.fixture(scope="module")
def lib():
    from monodepth2_b200 import _capi, build
    build.build()
    return _capi.load_library()


def test_velo_abi_validation_without_gpu(lib):
    from monodepth2_b200.kitti_depth import VELO_JOB_DTYPE
    n = C.c_size_t(0)
    assert lib.md2_velo_depth_scratch_bytes(0, 375, 1242, C.byref(n)) == -1
    assert lib.md2_velo_depth_scratch_bytes(2, 0, 1242, C.byref(n)) == -1
    assert lib.md2_velo_depth_scratch_bytes(2, 375, 1242, None) == -1
    assert lib.md2_velo_depth_scratch_bytes(2, 375, 1242, C.byref(n)) == 0
    assert n.value == 2 * 468 * 1552 * 12               # the largest native size below 1.25x, 12 bytes a pixel
    need = n.value
    scans = np.zeros(4 * 1000 + 64, np.float32)
    base = (scans.ctypes.data + 15) // 16 * 16
    nbytes = 16000                                      # room for 1000 points
    dummy = np.zeros(64, np.float32).ctypes.data

    def jobs(**kw):
        j = np.zeros(2, VELO_JOB_DTYPE)
        j["n_points"], j["height"], j["width"], j["offset"] = 500, 375, 1242, [0, 8000]
        for k, v in kw.items():
            j[k][1] = v
        return j

    def call(j, n_jobs=2, scratch_bytes=need, out_shape=OUT, scans_ptr=base, scans_bytes=nbytes):
        return lib.md2_velo_depth(scans_ptr, scans_bytes, j.ctypes.data, dummy, n_jobs, dummy, out_shape[0], out_shape[1],
                                  dummy, scratch_bytes, None)
    ok = jobs()
    assert call(ok, n_jobs=0) == -1
    assert call(ok, out_shape=(0, 1242)) == -1 and call(ok, out_shape=(375, -1)) == -1
    assert call(ok, scans_ptr=None) == -1
    assert lib.md2_velo_depth(base, nbytes, None, dummy, 2, dummy, 375, 1242, dummy, need, None) == -1
    assert call(jobs(n_points=-1)) == -1                                  # a negative count
    assert call(jobs(height=0)) == -1 and call(jobs(width=-3)) == -1      # non-positive sizes
    assert call(jobs(offset=-16)) == -1
    assert call(jobs(offset=nbytes + 16)) == -1                           # the scan outside the buffer
    assert call(jobs(offset=8000, n_points=501)) == -1                    # its last point outside
    assert call(jobs(offset=7992)) == -1                                  # not 16-byte aligned
    assert call(jobs(height=469)) == -2 and call(jobs(width=1553)) == -2  # native / out >= 1.25
    assert call(jobs(height=10, width=1)) == -2                           # sub2ind makes every pixel one group
    assert call(ok, scratch_bytes=need - 1) == -3                         # short scratch
    assert call(ok, out_shape=(300, 1242), scratch_bytes=need) == -2      # 375 rows are >= 1.25 x 300


# ------------------------------------------------------------------ GPU: exact cases
def _bitwise(got, want):
    """Bit for bit, but for the sign of a zero: a scan's x of -0.0 stays -0.0 or not in the reference depending on the
    order of numpy's reductions; md2_velo_depth always writes +0.0."""
    got = got.cpu().numpy() if torch.is_tensor(got) else got
    want = want + np.float32(0.0)
    assert got.shape == want.shape and got.dtype == want.dtype == np.float32
    bad = np.nonzero(got.view(np.int32) != want.view(np.int32))
    assert bad[0].size == 0, (bad[0].size, [tuple(int(a[i]) for a in bad) for i in range(min(4, bad[0].size))],
                              got[bad][:4], want[bad][:4])


EXACT_CASES = [(s, OUT) for s in S.KITTI_NATIVE_SIZES] + [((300, 1000), OUT), ((375, 1242), (375, 1242)),
                                                          ((370, 1224), (370, 1224))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", EXACT_CASES, ids=lambda c: "%dx%d-to-%dx%d" % (c[0][1], c[0][0], c[1][1], c[1][0]))
@pytest.mark.parametrize("vel_depth", [False, True], ids=["z", "vel_depth"])
def test_exact_scans_equal_oracle(case, vel_depth):
    from monodepth2_b200.kitti_depth import velo_depth
    native, out = case
    Ps = [_dyadic_P(2), _dyadic_P(2), _dyadic_P(3), _dyadic_P(3), _dyadic_P(2)]
    scans = [exact_scan(native[0] * 7 + k, P, *native) for k, P in enumerate(Ps[:4])] + [np.zeros((0, 4), np.float32)]
    flips = [False, True, False, True, True]
    got = velo_depth(scans, Ps, [native] * 5, out, flips, vel_depth)
    assert got.shape == (5, 1) + out
    want = np.stack([oracle_depth_gt(s, P, native, out, f, vel_depth) for s, P, f in zip(scans, Ps, flips)])
    assert np.count_nonzero(want[:4]) > 1000 and np.count_nonzero(want[4]) == 0
    _bitwise(got, want)
    _bitwise(velo_depth(scans, Ps, [native] * 5, out, flips, vel_depth), want)     # the same bits again


@pytest.mark.gpu
def test_exact_scans_mixed_sizes_in_one_batch():
    from monodepth2_b200.kitti_depth import velo_depth
    sizes = S.KITTI_NATIVE_SIZES + [(300, 1000), (2, 2)]
    Ps = [_dyadic_P(2 + k % 2) for k in range(len(sizes))]
    scans = [exact_scan(k, P, *sh) for k, (P, sh) in enumerate(zip(Ps, sizes))]
    flips = [k % 2 == 1 for k in range(len(sizes))]
    got = velo_depth(scans, Ps, sizes, OUT, flips)
    want = np.stack([oracle_depth_gt(s, P, sh, OUT, f) for s, P, sh, f in zip(scans, Ps, sizes, flips)])
    _bitwise(got, want)


# ------------------------------------------------------------------ GPU: realistic scans
@pytest.mark.gpu
@pytest.mark.parametrize("vel_depth", [False, True], ids=["z", "vel_depth"])
def test_realistic_scans_match_oracle(kitti_calib, vel_depth):
    """121 600-point KITTI-like sweeps with KITTI's own calibration for cams 2 and 3 and the five native sizes.  The
    pixel of every point must agree except within 1e-9 px of a rounding boundary (counted: none at these seeds), and
    every value within one float32 ulp (the sums of P (x, y, z, 1) may round differently from numpy's BLAS)."""
    from monodepth2_b200.kitti_depth import velo_depth, velo_to_image
    scans, Ps, shapes, flips, boundary = [], [], [], [], 0
    for k, shape in enumerate(S.KITTI_NATIVE_SIZES * 2):
        P, im_shape = velo_to_image(kitti_calib(shape), 2 + k % 2)
        scan = S.velodyne_scan(50 + k)
        boundary += _boundary_points(_numpy_project(P, scan, *shape, vel_depth)[3], scan)
        scans.append(scan); Ps.append(P); shapes.append(im_shape); flips.append(k >= 5)
    assert boundary == 0
    got = velo_depth(scans, Ps, shapes, OUT, flips, vel_depth).cpu().numpy()
    want = np.stack([oracle_depth_gt(s, P, sh, OUT, f, vel_depth) for s, P, sh, f in zip(scans, Ps, shapes, flips)])
    want += np.float32(0.0)                                      # +0.0 for every zero, as in _bitwise
    assert np.array_equal(got > 0, want > 0)
    ulps = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1, ulps.max()
    assert np.count_nonzero(want) > 10 * 5000


# ------------------------------------------------------------------ GPU: MonoBatch end to end
def _oracle_inputs(native, host_items, H, W, S_):
    from torch.utils.data import default_collate
    from test_mono_batch import _oracle_batch
    want = _oracle_batch(native, H, W, S_)
    want["depth_gt"] = default_collate([it["depth_gt"] for it in host_items])
    return want


def _assert_inputs(got, want):
    from test_mono_batch import _assert_equal_batch
    _assert_equal_batch(got, want, torch.uint8)


@pytest.mark.gpu
def test_mono_batch_depth_gt_equals_oracle_items(tmp_path):
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    folders = _write_kitti_drive(str(tmp_path), 4)
    fids = [0, -1, 1, "s"]
    names = ["%s %d %s" % (f, i, s) for f in folders for i in (1, 2) for s in "lr"]
    gpu, host = _datasets(str(tmp_path), names, fids)
    mb = MonoBatch(64, 96, fids, 2)
    for seed in range(2):
        order = list(np.random.default_rng(seed).permutation(len(names)))
        random.seed(seed); torch.manual_seed(seed)
        items = [gpu[i] for i in order]
        random.seed(seed); torch.manual_seed(seed)
        host_items = [host[i] for i in order]
        native = collate_native(items)
        assert native.buffer.is_pinned()
        got = mb(native)
        assert got["depth_gt"].shape == (len(names), 1) + OUT and got["depth_gt"].dtype == torch.float32
        want = _oracle_inputs(collate_native(host_items), host_items, 64, 96, 2)
        _assert_inputs(got, want)
        again = mb(native)
        assert torch.equal(again["depth_gt"].view(torch.int32), got["depth_gt"].view(torch.int32))


@pytest.mark.gpu
def test_cuda_graph_replays_batches_of_other_native_sizes():
    """One graph captured on one batch replays batches whose frames and scans both have other native sizes (each
    sample's frames and scan share the drive's size, as in KITTI raw), and other scan lengths: every key equals the
    eager call, and depth_gt the oracle."""
    from monodepth2_b200.kitti_depth import VeloScan
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    fids = [0, -1, "s"]

    def batch(seed, sizes):
        rng = np.random.default_rng(seed)
        items = []
        for b, sh in enumerate(sizes):
            P = _dyadic_P(2 + b % 2)
            items.append({"frames": {f: rng.integers(0, 256, sh + (3,), dtype=np.uint8) for f in fids},
                          "do_color_aug": False, "do_flip": (b + seed) % 2 == 0, "color_aug": None, "side": "lr"[b % 2],
                          "velodyne": VeloScan(exact_scan(seed * 10 + b, P, *sh), P, sh)})
        return collate_native(items)
    natives = [batch(1, S.KITTI_NATIVE_SIZES[:4]), batch(2, S.KITTI_NATIVE_SIZES[1:]),
               batch(3, [(300, 1000), (375, 1242), (60, 100), (370, 1224)])]
    mb = MonoBatch(32, 64, fids, 2)
    eager = [{k: v.clone() for k, v in mb(nb).items()} for nb in natives]     # adds every native size to the plan
    for nb, e in zip(natives, eager):
        want = np.stack([oracle_depth_gt(j.scan, j.P, j.im_shape, OUT, f) for j, f in
                         zip(_velo_items(nb), nb.do_flip.tolist())])
        _bitwise(e["depth_gt"], want)
    assert len({nb.buffer.numel() for nb in natives}) == 3
    flat = torch.zeros(max(nb.buffer.numel() for nb in natives), dtype=torch.uint8, device="cuda")
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
    for i, nb in enumerate(natives[1:] + natives):
        flat.zero_()
        flat[:nb.buffer.numel()].copy_(nb.buffer)
        g.replay()
        torch.cuda.synchronize()
        want = eager[(i + 1) % len(natives)]
        assert sorted(map(str, out)) == sorted(map(str, want))
        for k, v in want.items():
            assert torch.equal(out[k].view(torch.int32) if v.dtype == torch.float32 else out[k],
                               v.view(torch.int32) if v.dtype == torch.float32 else v), (i, k)


def _velo_items(nb):
    """The VeloScan records a NativeBatch holds, read back from its buffer."""
    from monodepth2_b200.kitti_depth import VELO_JOB_DTYPE, VeloScan
    h = nb.buffer.numpy()
    jobs = h[nb.velo_jobs_offset:nb.velo_jobs_offset + nb.batch_size * VELO_JOB_DTYPE.itemsize].view(VELO_JOB_DTYPE)
    return [VeloScan(h[int(j["offset"]):int(j["offset"]) + 16 * int(j["n_points"])].view(np.float32).reshape(-1, 4),
                     j["P"].reshape(3, 4), (int(j["height"]), int(j["width"]))) for j in jobs]


@pytest.mark.gpu
def test_dataloader_with_workers_end_to_end(tmp_path):
    from torch.utils.data import DataLoader
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    folders = _write_kitti_drive(str(tmp_path), 5)
    fids = [0, -1, 1]
    names = ["%s %d %s" % (f, i, s) for f in folders for i in (1, 2, 3) for s in "lr"]
    gpu, _ = _datasets(str(tmp_path), names, fids)
    torch.manual_seed(0)
    loader = DataLoader(gpu, batch_size=4, shuffle=True, num_workers=2, pin_memory=True, collate_fn=collate_native)
    mb = MonoBatch(64, 96, fids, 2)
    n = 0
    for native in loader:
        assert native.buffer.is_pinned()
        got = mb(native)
        want = np.stack([oracle_depth_gt(v.scan, v.P, v.im_shape, OUT, f)
                         for v, f in zip(_velo_items(native), native.do_flip.tolist())])
        _bitwise(got["depth_gt"], want)
        n += native.batch_size
    assert n == len(names)
