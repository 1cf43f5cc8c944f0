"""ctypes mirror of include/md2_loss.h and loader of libmd2loss.so.

The library is the product: if it is missing or does not load, importing the ops
fails loudly (there is no PyTorch/CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import os

MAX_SCALES = 4
MAX_SRC = 4

# md2_dtype: element type of a differentiable leaf (md2_problem.*_dtype, md2_scale_tensors_typed, the typed head)
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2

_fp = C.POINTER(C.c_float)


class Md2Problem(C.Structure):
    _fields_ = [
        ("batch", C.c_int), ("height", C.c_int), ("width", C.c_int),
        ("num_scales", C.c_int), ("num_src", C.c_int),
        ("automask", C.c_int), ("avg_reprojection", C.c_int), ("align_corners", C.c_int),
        ("min_depth", C.c_float), ("max_depth", C.c_float), ("disparity_smoothness", C.c_float),
        ("want_grad", C.c_int), ("rows_per_segment", C.c_int), ("no_ssim", C.c_int),
        ("posecnn", C.c_int), ("predictive_mask", C.c_int),
        ("scale_level", C.c_int * MAX_SCALES),
        ("disp_dtype", C.c_int), ("pose_dtype", C.c_int * MAX_SRC), ("pmask_dtype", C.c_int),
    ]


class Md2Tensors(C.Structure):
    _fields_ = [
        ("target", C.c_void_p),
        ("source", C.c_void_p * MAX_SRC),
        ("T", C.c_void_p * MAX_SRC),
        ("pose_requires_grad", C.c_int * MAX_SRC),
        ("K", C.c_void_p),
        ("inv_K", C.c_void_p),
        ("disp", C.c_void_p * MAX_SCALES),
        ("color", C.c_void_p * MAX_SCALES),
        ("noise", C.c_void_p * MAX_SCALES),
        ("losses", C.c_void_p),
        ("grad_disp", C.c_void_p * MAX_SCALES),
        ("grad_T", C.c_void_p * MAX_SRC),
        ("depth", C.c_void_p * MAX_SCALES),
        ("warped", (C.c_void_p * MAX_SCALES) * MAX_SRC),
        ("identity_selection", C.c_void_p * MAX_SCALES),
        ("grad_depth_dbg", C.c_void_p * MAX_SCALES),
        ("axisangle", C.c_void_p * MAX_SRC),
        ("translation", C.c_void_p * MAX_SRC),
        ("pose_stride", C.c_int * MAX_SRC),
        ("pose_invert", C.c_int * MAX_SRC),
        ("cam_T_cam", C.c_void_p * MAX_SRC),
        ("grad_axisangle", C.c_void_p * MAX_SRC),
        ("grad_translation", C.c_void_p * MAX_SRC),
        ("target_u8", C.c_void_p),
        ("source_u8", C.c_void_p * MAX_SRC),
        ("color_u8", C.c_void_p * MAX_SCALES),
        ("u8_hwc", C.c_int),
        ("pmask", C.c_void_p * MAX_SCALES),
        ("grad_pmask", C.c_void_p * MAX_SCALES),
        ("noise_ready_event", C.c_void_p),
    ]


LIB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
LIB_PATH = os.path.join(LIB_DIR, "libmd2loss.so")

# every symbol include/md2_loss.h declares (tests/test_capi_symbols.py checks the header against this)
SYMBOLS = [
    "md2_version", "md2_status_string", "md2_loss_workspace_bytes", "md2_view_synthesis_loss",
    "md2_profile_enable", "md2_profile_march_ms",
    "md2_disp_to_depth", "md2_disp_to_depth_backward",
    "md2_backproject_depth", "md2_backproject_depth_backward",
    "md2_project3d", "md2_project3d_backward",
    "md2_grid_sample_border", "md2_grid_sample_border_backward",
    "md2_ssim", "md2_ssim_backward",
    "md2_smooth_loss", "md2_smooth_loss_backward",
    "md2_pose_to_matrix", "md2_pose_to_matrix_backward",
    "md2_depth_metrics_scratch_bytes", "md2_depth_metrics",
    "md2_scale_tensors", "md2_scale_tensors_typed", "md2_dispconv_sigmoid", "md2_dispconv_sigmoid_backward",
    "md2_dispconv_sigmoid_typed", "md2_dispconv_sigmoid_backward_typed",
    "md2_resize_plan_create", "md2_resize_plan_destroy", "md2_resize_scratch_bytes", "md2_resize_lanczos_u8",
    "md2_color_jitter_u8", "md2_upcat_pad", "md2_upcat_pad_backward",
    "md2_batch_plan_create", "md2_batch_plan_destroy", "md2_batch_plan_add_native_size", "md2_batch_scratch_bytes",
    "md2_batch_build_u8", "md2_velo_depth_scratch_bytes", "md2_velo_depth",
    "md2_jpeg_decode_scratch_bytes", "md2_jpeg_decode",
]

_lib = None


class Md2Error(RuntimeError):
    pass


def load_library(path: str = None) -> C.CDLL:
    """Loads libmd2loss.so (built in-tree by ``monodepth2_b200.build``); raises if absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("MD2_LIB_PATH") or LIB_PATH
    if not os.path.exists(p):
        raise Md2Error(
            "libmd2loss.so not found at %s - run `python -m monodepth2_b200.build` "
            "(there is no fallback path)" % p)
    lib = C.CDLL(p)
    lib.md2_status_string.restype = C.c_char_p
    lib.md2_status_string.argtypes = [C.c_int]
    lib.md2_version.restype = C.c_int
    lib.md2_loss_workspace_bytes.argtypes = [C.POINTER(Md2Problem), C.POINTER(C.c_size_t)]
    lib.md2_view_synthesis_loss.argtypes = [C.POINTER(Md2Problem), C.POINTER(Md2Tensors), C.c_void_p,
                                            C.c_size_t, C.c_void_p]
    for name in SYMBOLS:
        if name not in ("md2_status_string", "md2_resize_plan_destroy", "md2_batch_plan_destroy") and hasattr(lib, name):
            getattr(lib, name).restype = C.c_int
    lib.md2_scale_tensors.argtypes = [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_longlong),
                                      C.c_void_p, C.c_void_p]
    lib.md2_scale_tensors_typed.argtypes = [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int),
                                            C.POINTER(C.c_longlong), C.c_void_p, C.c_void_p]
    lib.md2_dispconv_sigmoid_typed.argtypes = [C.c_void_p] * 4 + [C.c_int] * 5 + [C.c_void_p]
    lib.md2_dispconv_sigmoid_backward_typed.argtypes = [C.c_void_p] * 7 + [C.c_int] * 5 + [C.c_void_p]
    lib.md2_upcat_pad.argtypes = [C.c_void_p] * 3 + [C.c_int] * 7 + [C.c_void_p]
    lib.md2_upcat_pad_backward.argtypes = [C.c_void_p] * 3 + [C.c_int] * 7 + [C.c_void_p]
    lib.md2_depth_metrics_scratch_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]
    lib.md2_depth_metrics.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t] + [C.c_int] * 9 + [C.c_void_p]
    lib.md2_resize_plan_destroy.restype = None
    lib.md2_resize_plan_destroy.argtypes = [C.c_void_p]
    lib.md2_resize_plan_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    lib.md2_resize_scratch_bytes.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]
    lib.md2_color_jitter_u8.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_void_p]
    lib.md2_resize_lanczos_u8.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int,
                                          C.c_int, C.c_void_p]
    lib.md2_batch_plan_create.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    lib.md2_batch_plan_destroy.restype = None
    lib.md2_batch_plan_destroy.argtypes = [C.c_void_p]
    lib.md2_batch_plan_add_native_size.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.md2_batch_scratch_bytes.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]
    lib.md2_batch_build_u8.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                       C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.md2_velo_depth_scratch_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]
    lib.md2_velo_depth.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                   C.c_void_p, C.c_size_t, C.c_void_p]
    lib.md2_jpeg_decode_scratch_bytes.argtypes = [C.c_int, C.c_longlong, C.c_longlong, C.POINTER(C.c_size_t)]
    lib.md2_jpeg_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t,
                                    C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p, C.c_size_t, C.c_void_p]
    if path is None:
        _lib = lib
    return lib


def check(lib, status: int, what: str = "md2 call") -> None:
    if status != 0:
        raise Md2Error("%s failed: %s (%d)" % (what, lib.md2_status_string(status).decode(), status))
