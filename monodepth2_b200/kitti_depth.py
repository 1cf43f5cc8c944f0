"""KITTI raw ``depth_gt`` built on the GPU from the velodyne scan (SURVEY.md 8f-3).

The reference's ``KITTIRAWDataset.get_depth`` (datasets/kitti_dataset.py; kitti_utils.py) projects every scan in
float64, resolves duplicate pixels with a ``Counter`` loop, resizes the map with skimage's order-0 resize and flips it,
on the host, for every sample.  Here a dataloader worker only reads the scan (``VelodyneDepthMixin``), and
``md2_velo_depth`` builds the float32 maps of a whole batch in three launches, bit for bit what the reference's chain
rounded to float32 gives.  The projection matrix stays host code: it is computed once per (drive date, camera) by the
reference's own numpy expression and cached.

    class GpuKITTIRAW(VelodyneDepthMixin, NativeFramesMixin, KITTIRAWDataset): pass
    loader = DataLoader(GpuKITTIRAW(...), ..., collate_fn=collate_native)
    build = MonoBatch(opt.height, opt.width, opt.frame_ids, 4)
    for native in loader:
        inputs = build(native)          # inputs["depth_gt"]: (B, 1, 375, 1242) float32 on the device

or, on its own, ``velo_depth(scans, P, native_shapes)``.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import functools
import os
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _capi

# md2_velo_job of include/md2_loss.h
VELO_JOB_DTYPE = np.dtype([("P", "<f8", (12,)), ("offset", "<i8"), ("n_points", "<i4"), ("height", "<i4"),
                           ("width", "<i4"), ("flip", "<i4"), ("vel_depth", "<i4"), ("reserved", "<i4")])
FULL_RES_SHAPE = (375, 1242)                    # KITTIDataset.full_res_shape[::-1], (height, width)


def _align(n: int, a: int = 16) -> int:
    return (n + a - 1) // a * a


def _read_calib_file(path: str) -> dict:
    """kitti_utils.read_calib_file."""
    float_chars = set("0123456789.e+- ")
    data = {}
    with open(path, "r") as f:
        for line in f.readlines():
            key, value = line.split(":", 1)
            value = value.strip()
            data[key] = value
            if float_chars.issuperset(value):
                try:
                    data[key] = np.array(list(map(float, value.split(" "))))
                except ValueError:
                    pass
    return data


@functools.lru_cache(maxsize=None)
def velo_to_image(calib_dir: str, cam: int = 2):
    """(P_velo2im (3, 4) float64, im_shape (height, width)) of a drive date's calibration, by the expressions of
    generate_depth_map (kitti_utils.py), so the 12 doubles are the reference's.  Cached per (directory, camera).
    The returned array is shared: do not write to it."""
    cam2cam = _read_calib_file(os.path.join(calib_dir, "calib_cam_to_cam.txt"))
    velo2cam = _read_calib_file(os.path.join(calib_dir, "calib_velo_to_cam.txt"))
    velo2cam = np.hstack((velo2cam["R"].reshape(3, 3), velo2cam["T"][..., np.newaxis]))
    velo2cam = np.vstack((velo2cam, np.array([0, 0, 0, 1.0])))
    im_shape = cam2cam["S_rect_02"][::-1].astype(np.int32)
    R_cam2rect = np.eye(4)
    R_cam2rect[:3, :3] = cam2cam["R_rect_00"].reshape(3, 3)
    P_rect = cam2cam["P_rect_0" + str(cam)].reshape(3, 4)
    P = np.dot(np.dot(P_rect, R_cam2rect), velo2cam)
    P.flags.writeable = False
    return P, (int(im_shape[0]), int(im_shape[1]))


@dataclasses.dataclass
class VeloScan:
    """One sample's depth source: the velodyne scan as read ((N, 4) float32), P_velo2im (3, 4) float64, the native
    image size (height, width) and the size depth_gt is resized to (height, width)."""
    scan: np.ndarray
    P: np.ndarray
    im_shape: tuple
    out_shape: tuple = FULL_RES_SHAPE


class VelodyneDepthMixin:
    """Put in front of ``NativeFramesMixin``: ``class GpuKITTIRAW(VelodyneDepthMixin, NativeFramesMixin,
    KITTIRAWDataset)``.  Where the dataset loads depth, its items carry ``"velodyne"`` (a ``VeloScan``: the scan read
    as ``load_velodyne_points`` reads it, with the cached calibration of the sample's camera) instead of ``depth_gt``;
    ``collate_native`` packs it and ``MonoBatch`` builds ``inputs["depth_gt"]`` from it.  Only for KITTI raw (the
    velodyne files of ``KITTIRAWDataset``)."""

    def native_depth(self, folder, frame_index, side, do_flip):
        calib_path = os.path.join(self.data_path, folder.split("/")[0])
        velo_filename = os.path.join(self.data_path, folder,
                                     "velodyne_points/data/{:010d}.bin".format(int(frame_index)))
        P, im_shape = velo_to_image(calib_path, self.side_map[side])
        scan = np.fromfile(velo_filename, dtype=np.float32).reshape(-1, 4)
        return {"velodyne": VeloScan(scan, P, im_shape, tuple(self.full_res_shape[::-1]))}


def pack_jobs(h: np.ndarray, jobs_off: int, scans_off: int, scans: Sequence[VeloScan], flips, vel_depth: bool) -> int:
    """Writes the job table at ``jobs_off`` of the uint8 array ``h`` and the scans from ``scans_off`` on (each 16-byte
    aligned; job offsets count from the start of ``h``).  Returns the end of the last scan."""
    jobs = h[jobs_off:jobs_off + len(scans) * VELO_JOB_DTYPE.itemsize].view(VELO_JOB_DTYPE)
    off = scans_off
    for i, v in enumerate(scans):
        a = np.ascontiguousarray(v.scan, dtype=np.float32)
        if a.ndim != 2 or a.shape[1] != 4:
            raise ValueError("a velodyne scan must be an (N, 4) float32 array, got %s" % (a.shape,))
        jobs[i] = (np.asarray(v.P, np.float64).reshape(12), off, a.shape[0], int(v.im_shape[0]), int(v.im_shape[1]),
                   int(bool(flips[i])), int(bool(vel_depth)), 0)
        h[off:off + a.nbytes] = a.view(np.uint8).reshape(-1)
        off = _align(off + a.nbytes)
    return off


def packed_bytes(scans: Sequence[VeloScan]) -> int:
    """Bytes ``pack_jobs`` writes from its ``scans_off`` on."""
    return sum(_align(np.asarray(v.scan).shape[0] * 16) for v in scans)


def run(lib, flat: torch.Tensor, host_jobs: int, jobs_off: int, n: int, out_shape) -> torch.Tensor:
    """Enqueues md2_velo_depth on the current stream for jobs at ``jobs_off`` of ``flat`` (the device copy of a packed
    buffer whose host job table is at address ``host_jobs``) -> (n, 1, h, w) float32."""
    oh, ow = int(out_shape[0]), int(out_shape[1])
    dev = flat.device
    out = torch.empty((n, 1, oh, ow), dtype=torch.float32, device=dev)
    nb = C.c_size_t(0)
    _capi.check(lib, lib.md2_velo_depth_scratch_bytes(n, oh, ow, C.byref(nb)), "md2_velo_depth_scratch_bytes")
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    base = flat.data_ptr()
    with torch.cuda.device(dev):
        st = lib.md2_velo_depth(base, flat.numel(), host_jobs, base + jobs_off, n, out.data_ptr(), oh, ow,
                                scratch.data_ptr(), scratch.numel(), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _capi.check(lib, st, "md2_velo_depth")
    return out


def velo_depth(scans: List[np.ndarray], P, native_shapes, out_shape=FULL_RES_SHAPE, flips=None, vel_depth: bool = False,
               device=None) -> torch.Tensor:
    """depth_gt of KITTIRAWDataset.get_depth for a batch, as (B, 1, out_h, out_w) float32 on the device.

    scans: B (N_b, 4) float32 scans as read; P: B (3, 4) float64 P_velo2im (or one for all); native_shapes: B
    (height, width) im_shape (or one for all); flips: B bools (np.fliplr after the resize).  ``out_shape`` equal to
    the native size gives generate_depth_map itself, ``vel_depth=True`` its vel_depth variant."""
    B = len(scans)
    Ps = [P] * B if np.asarray(P).ndim == 2 else list(P)
    shapes = [native_shapes] * B if np.asarray(native_shapes).ndim == 1 else list(native_shapes)
    flips = [False] * B if flips is None else list(flips)
    if not (len(Ps) == len(shapes) == len(flips) == B) or B == 0:
        raise ValueError("velo_depth needs one P, native shape and flip per scan, and at least one scan")
    items = [VeloScan(s, p, tuple(sh), tuple(out_shape)) for s, p, sh in zip(scans, Ps, shapes)]
    scans_off = _align(B * VELO_JOB_DTYPE.itemsize)
    buf = torch.empty(scans_off + packed_bytes(items), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    pack_jobs(buf.numpy(), 0, scans_off, items, flips, vel_depth)
    dev = torch.device(device if device is not None else "cuda")
    flat = buf.to(dev, non_blocking=True)
    lib = _capi.load_library()
    with torch.cuda.device(flat.device):
        return run(lib, flat, buf.data_ptr(), 0, B, out_shape)
