"""Restatement of the reference's KITTI raw ``depth_gt``: ``KITTIRAWDataset.get_depth`` (datasets/kitti_dataset.py)
over ``kitti_utils.read_calib_file`` / ``load_velodyne_points`` / ``sub2ind`` / ``generate_depth_map``
(kitti_utils.py:8-98) and ``skimage.transform.resize(order=0, preserve_range=True, mode='constant')``.

Two compatibility changes, and nothing else: ``np.int`` (removed from numpy) is ``int``; skimage is not installed, so
its resize is restated on the ``scipy.ndimage`` calls it makes (``resize``: ``gaussian_filter`` when an axis shrinks,
then ``zoom(grid_mode=True, mode='grid-constant')``).  Given the same scan and calibration, ``get_depth`` returns the
reference's map; ``MonoDataset.__getitem__`` then takes ``np.expand_dims(depth_gt, 0).astype(np.float32)``.
"""
from __future__ import annotations

import os
from collections import Counter

import numpy as np

SIDE_MAP = {"2": 2, "3": 3, "l": 2, "r": 3}      # KITTIDataset.side_map
FULL_RES_SHAPE = (1242, 375)                     # KITTIDataset.full_res_shape, (width, height)


def read_calib_file(path):
    """kitti_utils.read_calib_file."""
    float_chars = set("0123456789.e+- ")
    data = {}
    with open(path, "r") as f:
        for line in f.readlines():
            key, value = line.split(":", 1)
            value = value.strip()
            data[key] = value
            if float_chars.issuperset(value):
                # try to cast to float array
                try:
                    data[key] = np.array(list(map(float, value.split(" "))))
                except ValueError:
                    # casting error: data[key] already eq. value, so pass
                    pass
    return data


def load_velodyne_points(filename):
    """kitti_utils.load_velodyne_points."""
    points = np.fromfile(filename, dtype=np.float32).reshape(-1, 4)
    points[:, 3] = 1.0  # homogeneous
    return points


def sub2ind(matrixSize, rowSub, colSub):
    """kitti_utils.sub2ind: the reference's (wrong) linear index, (r, n-1) and (r+1, 0) collide."""
    m, n = matrixSize
    return rowSub * (n - 1) + colSub - 1


def velo_to_image(calib_dir, cam=2):
    """The calibration part of generate_depth_map -> (P_velo2im (3, 4) float64, im_shape)."""
    cam2cam = read_calib_file(os.path.join(calib_dir, "calib_cam_to_cam.txt"))
    velo2cam = read_calib_file(os.path.join(calib_dir, "calib_velo_to_cam.txt"))
    velo2cam = np.hstack((velo2cam["R"].reshape(3, 3), velo2cam["T"][..., np.newaxis]))
    velo2cam = np.vstack((velo2cam, np.array([0, 0, 0, 1.0])))

    # get image shape
    im_shape = cam2cam["S_rect_02"][::-1].astype(np.int32)

    # compute projection matrix velodyne->image plane
    R_cam2rect = np.eye(4)
    R_cam2rect[:3, :3] = cam2cam["R_rect_00"].reshape(3, 3)
    P_rect = cam2cam["P_rect_0" + str(cam)].reshape(3, 4)
    P_velo2im = np.dot(np.dot(P_rect, R_cam2rect), velo2cam)
    return P_velo2im, im_shape


def depth_from_points(velo, P_velo2im, im_shape, vel_depth=False):
    """generate_depth_map after the calibration, on the scan as load_velodyne_points returns it."""
    velo = velo[velo[:, 0] >= 0, :]

    # project the points to the camera
    velo_pts_im = np.dot(P_velo2im, velo.T).T
    velo_pts_im[:, :2] = velo_pts_im[:, :2] / velo_pts_im[:, 2][..., np.newaxis]

    if vel_depth:
        velo_pts_im[:, 2] = velo[:, 0]

    # check if in bounds
    # use minus 1 to get the exact same value as KITTI matlab code
    velo_pts_im[:, 0] = np.round(velo_pts_im[:, 0]) - 1
    velo_pts_im[:, 1] = np.round(velo_pts_im[:, 1]) - 1
    val_inds = (velo_pts_im[:, 0] >= 0) & (velo_pts_im[:, 1] >= 0)
    val_inds = val_inds & (velo_pts_im[:, 0] < im_shape[1]) & (velo_pts_im[:, 1] < im_shape[0])
    velo_pts_im = velo_pts_im[val_inds, :]

    # project to image
    depth = np.zeros((im_shape[:2]))
    depth[velo_pts_im[:, 1].astype(int), velo_pts_im[:, 0].astype(int)] = velo_pts_im[:, 2]

    # find the duplicate points and choose the closest depth
    inds = sub2ind(depth.shape, velo_pts_im[:, 1], velo_pts_im[:, 0])
    dupe_inds = [item for item, count in Counter(inds).items() if count > 1]
    for dd in dupe_inds:
        pts = np.where(inds == dd)[0]
        x_loc = int(velo_pts_im[pts[0], 0])
        y_loc = int(velo_pts_im[pts[0], 1])
        depth[y_loc, x_loc] = velo_pts_im[pts, 2].min()
    depth[depth < 0] = 0

    return depth


def generate_depth_map(calib_dir, velo_filename, cam=2, vel_depth=False):
    """kitti_utils.generate_depth_map."""
    P_velo2im, im_shape = velo_to_image(calib_dir, cam)
    return depth_from_points(load_velodyne_points(velo_filename), P_velo2im, im_shape, vel_depth)


def resize_nearest(image, output_shape):
    """skimage.transform.resize(image, output_shape, order=0, preserve_range=True, mode='constant') on a float64
    image, as skimage implements it: anti-aliasing is on for a float image when an axis shrinks, with
    sigma = max(0, (factor - 1) / 2) and the same mode; then ndi.zoom with grid_mode=True, and _clip_warp_output."""
    from scipy import ndimage as ndi
    image = np.asarray(image, dtype=np.float64)
    output_shape = tuple(output_shape)
    cval = 0
    factors = np.divide(image.shape, output_shape)
    if any(x < y for x, y in zip(output_shape, image.shape)):
        sigma = np.maximum(0, (factors - 1) / 2)
        filtered = ndi.gaussian_filter(image, sigma, cval=cval, mode="grid-constant")
    else:
        filtered = image
    out = ndi.zoom(filtered, [1 / f for f in factors], order=0, mode="grid-constant", cval=cval, grid_mode=True)
    # _clip_warp_output(image, out, 'constant', cval, clip=True)
    min_val, max_val = np.min(image), np.max(image)
    if not min_val <= cval <= max_val and np.min(out) <= cval <= np.max(out):
        min_val, max_val = min(min_val, cval), max(max_val, cval)
    np.clip(out, min_val, max_val, out=out)
    return out


def get_depth(data_path, folder, frame_index, side, do_flip, full_res_shape=FULL_RES_SHAPE):
    """KITTIRAWDataset.get_depth (datasets/kitti_dataset.py)."""
    calib_path = os.path.join(data_path, folder.split("/")[0])

    velo_filename = os.path.join(data_path, folder, "velodyne_points/data/{:010d}.bin".format(int(frame_index)))

    depth_gt = generate_depth_map(calib_path, velo_filename, SIDE_MAP[side])
    depth_gt = resize_nearest(depth_gt, full_res_shape[::-1])

    if do_flip:
        depth_gt = np.fliplr(depth_gt)

    return depth_gt


def depth_item(depth_gt):
    """What MonoDataset.__getitem__ stores under "depth_gt"."""
    import torch
    return torch.from_numpy(np.expand_dims(depth_gt, 0).astype(np.float32))
