"""Restatement of the reference's training item on PIL images: ``MonoDataset.__getitem__`` + ``preprocess``
(/root/reference/datasets/mono_dataset.py:90-109,136-185) with ``KITTIDataset.get_color``'s flip (kitti_dataset.py:
``color.transpose(pil.FLIP_LEFT_RIGHT)``), run with the installed Pillow and torchvision, and default collation.

Two compatibility changes, and nothing else: ``Image.ANTIALIAS`` (removed from Pillow) is ``Image.LANCZOS``, the same
filter; ``ColorJitter.get_params`` returns a tuple in the installed torchvision, applied here the way ColorJitter.forward
applies it (tests/test_color_jitter.py).  Given the same native frames and draws, ``get_item`` builds the reference's dict.
"""
from __future__ import annotations

import random

import numpy as np
import torch
from PIL import Image

KITTI_K = np.array([[0.58, 0, 0.5, 0],
                    [0, 1.92, 0.5, 0],
                    [0, 0, 1, 0],
                    [0, 0, 0, 1]], dtype=np.float32)
# mono_dataset.py:60-70, the tuple form
BRIGHTNESS, CONTRAST, SATURATION, HUE = (0.8, 1.2), (0.8, 1.2), (0.8, 1.2), (-0.1, 0.1)


def jitter_params():
    """One ColorJitter.get_params draw with the reference's ranges."""
    from torchvision import transforms
    return transforms.ColorJitter.get_params(BRIGHTNESS, CONTRAST, SATURATION, HUE)


def draw(is_train: bool = True):
    """The item's random draws in the reference's order (__getitem__, mono_dataset.py:136-185):
    -> (do_color_aug, do_flip, get_params tuple or None)."""
    do_color_aug = is_train and random.random() > 0.5
    do_flip = is_train and random.random() > 0.5
    params = jitter_params() if do_color_aug else None
    return do_color_aug, do_flip, params


def jitter_fn(params):
    """A get_params tuple as the callable the reference expects (torchvision ColorJitter.forward)."""
    from torchvision.transforms import functional as F
    if params is None:
        return lambda x: x
    fn_idx, b, c, s, h = params

    def apply(img):
        for i in fn_idx:
            fac = [b, c, s, h][int(i)]
            if fac is not None:
                img = [F.adjust_brightness, F.adjust_contrast, F.adjust_saturation, F.adjust_hue][int(i)](img, fac)
        return img
    return apply


def get_item(frames: dict, do_flip: bool, color_aug, side, height: int, width: int, num_scales: int = 4, K=KITTI_K):
    """frames: {frame id: native (h, w, 3) uint8}; color_aug: get_params tuple or None; side: "l" / "r" / None."""
    from torchvision import transforms
    to_tensor = transforms.ToTensor()
    resize = {i: transforms.Resize((height // 2 ** i, width // 2 ** i), interpolation=Image.LANCZOS)
              for i in range(num_scales)}                                           # mono_dataset.py:82-86
    inputs = {}
    for i in frames:                                                                # __getitem__
        color = Image.fromarray(np.asarray(frames[i], np.uint8))
        if do_flip:
            color = color.transpose(Image.FLIP_LEFT_RIGHT)                         # kitti_dataset.py get_color
        inputs[("color", i, -1)] = color
    for scale in range(num_scales):                                                 # __getitem__: intrinsics per scale
        Ks = np.array(K, dtype=np.float32).copy()
        Ks[0, :] *= width // (2 ** scale)
        Ks[1, :] *= height // (2 ** scale)
        inputs[("K", scale)] = torch.from_numpy(Ks)
        inputs[("inv_K", scale)] = torch.from_numpy(np.linalg.pinv(Ks))
    aug = jitter_fn(color_aug)
    for k in list(inputs):                                                          # preprocess, mono_dataset.py:98-109
        if "color" in k:
            n, im, _ = k
            for i in range(num_scales):
                inputs[(n, im, i)] = resize[i](inputs[(n, im, i - 1)])
    for k in list(inputs):
        f = inputs[k]
        if "color" in k:
            n, im, i = k
            inputs[(n, im, i)] = to_tensor(f)
            inputs[(n + "_aug", im, i)] = to_tensor(aug(f))
    for i in frames:                                                                # __getitem__: the native frames are dropped
        del inputs[("color", i, -1)]
        del inputs[("color_aug", i, -1)]
    if "s" in frames:                                                               # __getitem__
        stereo_T = np.eye(4, dtype=np.float32)
        baseline_sign = -1 if do_flip else 1
        side_sign = -1 if side == "l" else 1
        stereo_T[0, 3] = side_sign * baseline_sign * 0.1
        inputs["stereo_T"] = torch.from_numpy(stereo_T)
    return inputs


def collate(items):
    """The DataLoader's default collation of a list of items."""
    from torch.utils.data import default_collate
    return default_collate(items)
