"""Seeded synthetic batches shaped like the reference's input contract.

Key names and tensor conventions follow ``MonoDataset.__getitem__``
(/root/reference/datasets/mono_dataset.py:114-200), the KITTI normalised
intrinsics (/root/reference/datasets/kitti_dataset.py:29-32) and the
``PoseDecoder`` output scale (/root/reference/networks/pose_decoder.py:49).
All tensors are generated on the CPU from a ``torch.Generator`` so that the CPU
oracle, the PyTorch-CUDA path and the fused kernels see identical bits
(SURVEY.md section 8d: IID seed 0, STRUCTURED seed 5).
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

KITTI_K = np.array([[0.58, 0, 0.5, 0],
                    [0, 1.92, 0.5, 0],
                    [0, 0, 1, 0],
                    [0, 0, 0, 1]], dtype=np.float32)


def _rodrigues(aa: torch.Tensor) -> torch.Tensor:
    """(B,3) axis-angle -> (B,3,3); same parameterisation as layers.py:64-103."""
    ang = aa.norm(dim=1, keepdim=True)
    ax = aa / (ang + 1e-7)
    ca, sa = torch.cos(ang)[:, 0], torch.sin(ang)[:, 0]
    C = 1 - ca
    x, y, z = ax[:, 0], ax[:, 1], ax[:, 2]
    R = torch.stack([
        torch.stack([x * x * C + ca, x * y * C - z * sa, z * x * C + y * sa], 1),
        torch.stack([x * y * C + z * sa, y * y * C + ca, y * z * C - x * sa], 1),
        torch.stack([z * x * C - y * sa, y * z * C + x * sa, z * z * C + ca], 1)], 1)
    return R


def pose_matrix(axisangle: torch.Tensor, translation: torch.Tensor, invert: bool) -> torch.Tensor:
    """(B,3),(B,3) -> (B,4,4): Trans(t)·R, or Rᵀ·Trans(−t) when ``invert`` (layers.py:28-45)."""
    B = axisangle.shape[0]
    R = _rodrigues(axisangle)
    T = torch.zeros(B, 4, 4, dtype=axisangle.dtype)
    T[:, 3, 3] = 1
    if invert:
        Rt = R.transpose(1, 2)
        T[:, :3, :3] = Rt
        T[:, :3, 3] = -(Rt @ translation.unsqueeze(-1))[:, :, 0]
    else:
        T[:, :3, :3] = R
        T[:, :3, 3] = translation
    return T


def intrinsics(batch: int, height: int, width: int, gen: torch.Generator = None,
               jitter: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """Scale-0 K and inv_K = pinv(K), (B,4,4) fp32 (mono_dataset.py:164-173)."""
    Ks, iKs = [], []
    for _ in range(batch):
        K = KITTI_K.copy()
        K[0, :] *= width
        K[1, :] *= height
        if jitter:
            r = torch.rand(4, generator=gen).numpy()
            K[0, 0] *= 0.9 + 0.2 * r[0]
            K[1, 1] *= 0.9 + 0.2 * r[1]
            K[0, 2] += (r[2] * 0.04 - 0.02) * width
            K[1, 2] += (r[3] * 0.04 - 0.02) * height
        Ks.append(torch.from_numpy(K))
        iKs.append(torch.from_numpy(np.linalg.pinv(K).astype(np.float32)))
    return torch.stack(Ks), torch.stack(iKs)


def _box_blur(x: torch.Tensor, k: int) -> torch.Tensor:
    return F.avg_pool2d(F.pad(x, (k // 2,) * 4, mode="reflect"), k, 1)


def make_batch(batch: int = 12, height: int = 192, width: int = 640,
               frame_ids: Sequence = (0, -1, 1), num_scales: int = 4, seed: int = 0,
               kind: str = "iid", jitter_K: bool = False,
               noise_seed: int = 99, n_id: int = None, all_scale_K: bool = False, multiscale_noise: bool = False):
    """Returns ``(inputs, outputs, pose, noise)`` on the CPU in fp32.

    inputs : {("color", f, s)}, ("K", 0), ("inv_K", 0), "stereo_T"
    outputs: {("disp", s)}, {("cam_T_cam", 0, f)} for temporal sources
    pose   : {f: (axisangle (B,3), translation (B,3))} the leaves behind cam_T_cam
    noise  : list over scales of (B, n_id, H, W) standard-normal tie-break draws
    """
    g = torch.Generator().manual_seed(seed)
    inputs: Dict = {}
    outputs: Dict = {}
    B, H, W = batch, height, width
    if kind == "iid":
        for f in frame_ids:
            for s in range(num_scales):
                inputs[("color", f, s)] = torch.rand(B, 3, H >> s, W >> s, generator=g)
        for s in range(num_scales):
            outputs[("disp", s)] = torch.rand(B, 1, H >> s, W >> s, generator=g)
    elif kind == "structured":
        base = _box_blur(torch.rand(B, 3, H + 64, W + 64, generator=g), 9)
        lo = base.amin(dim=(1, 2, 3), keepdim=True)
        hi = base.amax(dim=(1, 2, 3), keepdim=True)
        base = (base - lo) / (hi - lo)
        shift = {0: 0, -1: 3, 1: -3, "s": 6}
        for f in frame_ids:                       # further temporal neighbours (--frame_ids 0 -2 -1 1 2): 3 px per frame
            if f not in shift:
                shift[f] = -3 * f
        for f in frame_ids:
            x0 = 32 + shift[f]
            frame = base[:, :, 32:32 + H, x0:x0 + W].contiguous()
            for s in range(num_scales):
                inputs[("color", f, s)] = frame if s == 0 else F.avg_pool2d(frame, 2 ** s)
        for s in range(num_scales):
            d = _box_blur(torch.rand(B, 1, H >> s, W >> s, generator=g), 5)
            lo = d.amin(dim=(1, 2, 3), keepdim=True)
            hi = d.amax(dim=(1, 2, 3), keepdim=True)
            outputs[("disp", s)] = (0.2 + 0.6 * (d - lo) / (hi - lo)).contiguous()
    else:
        raise ValueError(kind)

    K, inv_K = intrinsics(B, H, W, g, jitter_K)
    inputs[("K", 0)] = K
    inputs[("inv_K", 0)] = inv_K
    if all_scale_K:      # mono_dataset.py:164-173: one K / inv_K per pyramid level (for --v1_multiscale)
        for s in range(1, num_scales):
            Ks = K.clone()
            Ks[:, 0, :] /= 2 ** s
            Ks[:, 1, :] /= 2 ** s
            inputs[("K", s)] = Ks
            inputs[("inv_K", s)] = torch.from_numpy(
                np.stack([np.linalg.pinv(k.numpy()).astype(np.float32) for k in Ks]))
    stereo_T = torch.eye(4).repeat(B, 1, 1)
    stereo_T[:, 0, 3] = 0.1
    inputs["stereo_T"] = stereo_T

    pose: Dict = {}
    for f in frame_ids[1:]:
        if f == "s":
            continue
        aa = 0.01 * torch.randn(B, 3, generator=g)
        tr = 0.01 * torch.randn(B, 3, generator=g)
        pose[f] = (aa, tr)
        outputs[("cam_T_cam", 0, f)] = pose_matrix(aa, tr, invert=(f < 0))

    n_src = len(frame_ids) - 1
    if n_id is None:
        n_id = n_src
    gn = torch.Generator().manual_seed(noise_seed)
    noise: List[torch.Tensor] = [torch.randn(B, n_id, H >> (s if multiscale_noise else 0),
                                             W >> (s if multiscale_noise else 0), generator=gn)
                                 for s in range(num_scales)]
    return inputs, outputs, pose, noise


# ---- KITTI raw velodyne scans and calibration (depth_gt on the GPU, monodepth2_b200/kitti_depth.py)
# The 2011_09_26 calibration published with KITTI raw, rounded as its text files print it.
KITTI_CAM_TO_CAM = {
    "R_rect_00": [9.999239e-01, 9.837760e-03, -7.445048e-03, -9.869795e-03, 9.999421e-01, -4.278459e-03,
                  7.402527e-03, 4.351614e-03, 9.999631e-01],
    "P_rect_02": [7.215377e+02, 0.0, 6.095593e+02, 4.485728e+01, 0.0, 7.215377e+02, 1.728540e+02, 2.163791e-01,
                  0.0, 0.0, 1.0, 2.745884e-03],
    "P_rect_03": [7.215377e+02, 0.0, 6.095593e+02, -3.395242e+02, 0.0, 7.215377e+02, 1.728540e+02, 2.199936e+00,
                  0.0, 0.0, 1.0, 2.729905e-03],
}
KITTI_VELO_TO_CAM = {
    "R": [7.533745e-03, -9.999714e-01, -6.166020e-04, 1.480249e-02, 7.280733e-04, -9.998902e-01, 9.998621e-01,
          7.523790e-03, 1.480755e-02],
    "T": [-4.069766e-03, -7.631618e-02, -2.717806e-01],
}
KITTI_NATIVE_SIZES = [(375, 1242), (376, 1241), (374, 1238), (370, 1226), (370, 1224)]    # (h, w) of the raw drives


def write_kitti_calibration(calib_dir: str, im_shape=(375, 1242), cam_to_cam: dict = None, velo_to_cam: dict = None):
    """calib_cam_to_cam.txt and calib_velo_to_cam.txt in KITTI's text format (``key: v v v`` in %.6e where that is exact,
    and a calib_time line that read_calib_file keeps as a string)."""
    import os
    cc = dict(KITTI_CAM_TO_CAM if cam_to_cam is None else cam_to_cam)
    vc = dict(KITTI_VELO_TO_CAM if velo_to_cam is None else velo_to_cam)
    fmt = lambda vals: " ".join("%.6e" % v if float("%.6e" % v) == v else repr(float(v)) for v in vals)
    os.makedirs(calib_dir, exist_ok=True)
    with open(os.path.join(calib_dir, "calib_cam_to_cam.txt"), "w") as f:
        f.write("calib_time: 09-Jan-2012 13:57:47\ncorner_dist: 9.950000e-02\n")
        f.write("S_rect_02: %s\nS_rect_03: %s\n" % (fmt([im_shape[1], im_shape[0]]), fmt([im_shape[1], im_shape[0]])))
        for k, v in cc.items():
            f.write("%s: %s\n" % (k, fmt(v)))
    with open(os.path.join(calib_dir, "calib_velo_to_cam.txt"), "w") as f:
        f.write("calib_time: 15-Mar-2012 11:37:16\n")
        for k, v in vc.items():
            f.write("%s: %s\n" % (k, fmt(v)))
        f.write("delta_f: 0.000000e+00 0.000000e+00\ndelta_c: 0.000000e+00 0.000000e+00\n")


def velodyne_scan(seed: int, n_azimuth: int = 1900, n_beams: int = 64) -> np.ndarray:
    """A KITTI-like HDL-64 sweep, (n_beams * n_azimuth, 4) float32 (x forward, y left, z up, reflectance): a ground
    plane 1.73 m below the sensor and walls of a street, ranges clipped to 120 m, range noise, and a few dropped
    returns (NaN).  About a seventh of the points fall inside the left camera's image."""
    rng = np.random.default_rng(seed)
    az = np.linspace(-np.pi, np.pi, n_azimuth, endpoint=False) + rng.uniform(0, 2 * np.pi / n_azimuth)
    el = np.deg2rad(np.linspace(2.0, -24.8, n_beams))
    A, E = np.meshgrid(az, el)
    d = np.stack([np.cos(E) * np.cos(A), np.cos(E) * np.sin(A), np.sin(E)], -1)
    ground = np.where(d[..., 2] < -1e-3, -1.73 / np.minimum(d[..., 2], -1e-3), np.inf)
    wall = np.where(np.abs(d[..., 1]) > 1e-3, (7.0 + 2.0 * np.sin(3 * A)) / np.maximum(np.abs(d[..., 1]), 1e-3), np.inf)
    r = np.minimum(np.minimum(ground, wall), 120.0) * (1 + rng.normal(0, 0.003, A.shape))
    pts = (d * r[..., None]).reshape(-1, 3)
    refl = rng.uniform(0, 1, (pts.shape[0], 1))
    scan = np.concatenate([pts, refl], 1).astype(np.float32)
    scan[rng.random(scan.shape[0]) < 0.002, :3] = np.nan
    return scan
