"""Drop-in for the hot-path symbols of the reference's ``layers.py``.

Same class names, constructor arguments, call signatures and tensor conventions as
/root/reference/layers.py, so ``trainer.py``'s ``from layers import *`` (trainer.py:22)
can point here unchanged.  Every op below launches a hand-written sm_100a kernel of
libmd2loss.so through the C ABI (include/md2_loss.h); autograd is wired with
``torch.autograd.Function``.  Inputs must be CUDA float32 tensors (the disparity head
also takes a bfloat16 / float16 feature map): there is no PyTorch/CPU fallback, a missing
library or a CPU tensor raises.

The fused fast path is ``monodepth2_b200.fused_loss`` (one call replaces
generate_images_pred + compute_losses); these per-layer ops keep the reference's
unfused call graph working on the same kernels' arithmetic.
"""
from __future__ import annotations

import ctypes as C
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _capi

__all__ = ["disp_to_depth", "transformation_from_parameters", "get_translation_matrix",
           "rot_from_axisangle", "BackprojectDepth", "Project3D", "SSIM", "get_smooth_loss",
           "grid_sample_border", "ConvBlock", "Conv3x3", "upsample", "compute_depth_errors",
           "DispConvSigmoid", "fuse_disp_heads", "upcat_pad", "fuse_decoder_stages", "depth_metrics",
           "DEPTH_METRIC_NAMES"]


def _lib():
    return _capi.load_library()


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor (monodepth2_b200.layers has no CPU path)" % name)
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32, got %s" % (name, t.dtype))
    return t.contiguous()


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _call(fn_name, dev, *args):
    lib = _lib()
    with torch.cuda.device(dev):
        st = getattr(lib, fn_name)(*args)
    _capi.check(lib, st, fn_name)


# ------------------------------------------------------------------ disp_to_depth (layers.py:16-25)
class _DispToDepth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, disp, min_depth, max_depth):
        d = _f32c(disp, "disp")
        scaled, depth = torch.empty_like(d), torch.empty_like(d)
        _call("md2_disp_to_depth", d.device, _p(d), C.c_float(min_depth), C.c_float(max_depth), _p(scaled),
              _p(depth), C.c_longlong(d.numel()), _stream(d))
        ctx.save_for_backward(d)
        ctx.lim = (float(min_depth), float(max_depth))
        return scaled, depth

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_scaled, g_depth):
        (d,) = ctx.saved_tensors
        gs = _f32c(g_scaled, "grad") if g_scaled is not None else None
        gd = _f32c(g_depth, "grad") if g_depth is not None else None
        out = torch.empty_like(d)
        _call("md2_disp_to_depth_backward", d.device, _p(d), C.c_float(ctx.lim[0]), C.c_float(ctx.lim[1]),
              _p(gs), _p(gd), _p(out), C.c_longlong(d.numel()), _stream(d))
        return out, None, None


def disp_to_depth(disp, min_depth, max_depth):
    """layers.py:16-25 -> (scaled_disp, depth)."""
    return _DispToDepth.apply(disp, float(min_depth), float(max_depth))


# ------------------------------------------------------------------ pose (layers.py:28-103)
class _PoseToMatrix(torch.autograd.Function):
    @staticmethod
    def forward(ctx, axisangle, translation, invert):
        B = axisangle.shape[0]
        aa = _f32c(axisangle.reshape(B, 3), "axisangle")
        tr = _f32c(translation.reshape(B, 3), "translation")
        T = torch.empty((B, 4, 4), dtype=torch.float32, device=aa.device)
        _call("md2_pose_to_matrix", aa.device, _p(aa), _p(tr), C.c_int(int(invert)), _p(T), C.c_int(B), _stream(aa))
        ctx.save_for_backward(aa, tr)
        ctx.invert = int(invert)
        ctx.shapes = (axisangle.shape, translation.shape)
        return T

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gT):
        aa, tr = ctx.saved_tensors
        g = _f32c(gT, "grad_T")
        gaa, gtr = torch.empty_like(aa), torch.empty_like(tr)
        _call("md2_pose_to_matrix_backward", aa.device, _p(g), _p(aa), _p(tr), C.c_int(ctx.invert), _p(gaa), _p(gtr),
              C.c_int(aa.shape[0]), _stream(aa))
        return gaa.reshape(ctx.shapes[0]), gtr.reshape(ctx.shapes[1]), None


def transformation_from_parameters(axisangle, translation, invert=False):
    """layers.py:28-45.  axisangle, translation: (B,1,3) -> (B,4,4)."""
    return _PoseToMatrix.apply(axisangle, translation, bool(invert))


def get_translation_matrix(translation_vector):
    """layers.py:48-61 (zero rotation through the same kernel)."""
    t = translation_vector.contiguous().view(-1, 1, 3)
    return _PoseToMatrix.apply(torch.zeros_like(t), t, False)


def rot_from_axisangle(vec):
    """layers.py:64-103 (zero translation through the same kernel)."""
    return _PoseToMatrix.apply(vec, torch.zeros_like(vec), False)


# ------------------------------------------------------------------ BackprojectDepth (layers.py:139-168)
class _Backproject(torch.autograd.Function):
    @staticmethod
    def forward(ctx, depth, inv_K, B, H, W):
        d = _f32c(depth, "depth")
        ik = _f32c(inv_K, "inv_K")
        if d.numel() != B * H * W or tuple(ik.shape) != (B, 4, 4):
            raise RuntimeError("BackprojectDepth: depth %s / inv_K %s do not match (batch=%d, %dx%d)"
                               % (tuple(depth.shape), tuple(inv_K.shape), B, H, W))
        out = torch.empty((B, 4, H * W), dtype=torch.float32, device=d.device)
        _call("md2_backproject_depth", d.device, _p(d), _p(ik), _p(out), C.c_int(B), C.c_int(H), C.c_int(W), _stream(d))
        ctx.save_for_backward(ik)
        ctx.dims = (B, H, W, depth.shape)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        (ik,) = ctx.saved_tensors
        B, H, W, shape = ctx.dims
        g = _f32c(g, "grad")
        gd = torch.empty((B, 1, H, W), dtype=torch.float32, device=g.device)
        _call("md2_backproject_depth_backward", g.device, _p(g), _p(ik), _p(gd), C.c_int(B), C.c_int(H), C.c_int(W), _stream(g))
        return gd.reshape(shape), None, None, None, None


class BackprojectDepth(nn.Module):
    """Layer to transform a depth image into a point cloud (layers.py:139-168)."""

    def __init__(self, batch_size, height, width):
        super().__init__()
        self.batch_size, self.height, self.width = batch_size, height, width

    def forward(self, depth, inv_K):
        return _Backproject.apply(depth, inv_K, self.batch_size, self.height, self.width)


# ------------------------------------------------------------------ Project3D (layers.py:171-193)
class _Project(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, K, T, B, H, W, eps):
        pts, K, T = _f32c(points, "points"), _f32c(K, "K"), _f32c(T, "T")
        if tuple(pts.shape) != (B, 4, H * W):
            raise RuntimeError("Project3D: points %s do not match (batch=%d, %dx%d)" % (tuple(points.shape), B, H, W))
        out = torch.empty((B, H, W, 2), dtype=torch.float32, device=pts.device)
        _call("md2_project3d", pts.device, _p(pts), _p(K), _p(T), C.c_float(eps), _p(out), C.c_int(B), C.c_int(H),
              C.c_int(W), _stream(pts))
        ctx.save_for_backward(pts, K, T)
        ctx.dims = (B, H, W, eps)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        pts, K, T = ctx.saved_tensors
        B, H, W, eps = ctx.dims
        g = _f32c(g, "grad")
        gp = torch.empty_like(pts) if ctx.needs_input_grad[0] else None
        gT = torch.empty_like(T) if ctx.needs_input_grad[2] else None
        _call("md2_project3d_backward", g.device, _p(g), _p(pts), _p(K), _p(T), C.c_float(eps), _p(gp), _p(gT),
              C.c_int(B), C.c_int(H), C.c_int(W), _stream(g))
        return gp, None, gT, None, None, None, None


class Project3D(nn.Module):
    """Projects 3D points into a camera with intrinsics K at position T (layers.py:171-193)."""

    def __init__(self, batch_size, height, width, eps=1e-7):
        super().__init__()
        self.batch_size, self.height, self.width, self.eps = batch_size, height, width, eps

    def forward(self, points, K, T):
        return _Project.apply(points, K, T, self.batch_size, self.height, self.width, float(self.eps))


# ------------------------------------------------------------------ grid_sample border (trainer.py:384-387)
class _GridSample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, grid, align_corners):
        img, grid = _f32c(img, "input"), _f32c(grid, "grid")
        B, Cn, IH, IW = img.shape
        _, OH, OW, two = grid.shape
        if grid.shape[0] != B or two != 2:
            raise RuntimeError("grid_sample_border: grid %s does not match input %s" % (tuple(grid.shape), tuple(img.shape)))
        out = torch.empty((B, Cn, OH, OW), dtype=torch.float32, device=img.device)
        _call("md2_grid_sample_border", img.device, _p(img), _p(grid), _p(out), C.c_int(B), C.c_int(Cn), C.c_int(IH),
              C.c_int(IW), C.c_int(OH), C.c_int(OW), C.c_int(int(align_corners)), _stream(img))
        ctx.save_for_backward(img, grid)
        ctx.ac = int(align_corners)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        img, grid = ctx.saved_tensors
        if ctx.needs_input_grad[0]:
            raise RuntimeError("grid_sample_border: gradient w.r.t. the image is not on the path "
                               "(images do not require grad, trainer.py:384-387)")
        g = _f32c(g, "grad")
        B, Cn, IH, IW = img.shape
        _, OH, OW, _ = grid.shape
        gg = torch.empty_like(grid)
        _call("md2_grid_sample_border_backward", g.device, _p(g), _p(img), _p(grid), _p(gg), C.c_int(B), C.c_int(Cn),
              C.c_int(IH), C.c_int(IW), C.c_int(OH), C.c_int(OW), C.c_int(ctx.ac), _stream(g))
        return None, gg, None


def grid_sample_border(input, grid, align_corners=False):
    """F.grid_sample(input, grid, mode="bilinear", padding_mode="border") as trainer.py:384-387 calls it."""
    return _GridSample.apply(input, grid, bool(align_corners))


# ------------------------------------------------------------------ SSIM (layers.py:218-248)
class _SSIM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y):
        x, y = _f32c(x, "x"), _f32c(y, "y")
        if x.shape != y.shape or x.dim() != 4:
            raise RuntimeError("SSIM: x %s and y %s must be equal 4-D shapes" % (tuple(x.shape), tuple(y.shape)))
        B, Cn, H, W = x.shape
        out = torch.empty_like(x)
        _call("md2_ssim", x.device, _p(x), _p(y), _p(out), C.c_int(B), C.c_int(Cn), C.c_int(H), C.c_int(W), _stream(x))
        ctx.save_for_backward(x, y)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        g = _f32c(g, "grad")
        B, Cn, H, W = x.shape
        gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gy = torch.empty_like(y) if ctx.needs_input_grad[1] else None
        _call("md2_ssim_backward", g.device, _p(g), _p(x), _p(y), _p(gx), _p(gy), C.c_int(B), C.c_int(Cn), C.c_int(H),
              C.c_int(W), _stream(g))
        return gx, gy


class SSIM(nn.Module):
    """Layer to compute the SSIM loss between a pair of images (layers.py:218-248)."""

    def __init__(self):
        super().__init__()
        self.C1 = 0.01 ** 2
        self.C2 = 0.03 ** 2

    def forward(self, x, y):
        return _SSIM.apply(x, y)


# ------------------------------------------------------------------ get_smooth_loss (layers.py:202-215)
class _Smooth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, disp, img):
        d, im = _f32c(disp, "disp"), _f32c(img, "img")
        B, one, H, W = d.shape
        if one != 1 or im.shape[0] != B or tuple(im.shape[2:]) != (H, W):
            raise RuntimeError("get_smooth_loss: disp %s / img %s mismatch" % (tuple(d.shape), tuple(im.shape)))
        loss = torch.empty((), dtype=torch.float32, device=d.device)
        scratch = torch.empty(2, dtype=torch.float64, device=d.device)
        _call("md2_smooth_loss", d.device, _p(d), _p(im), _p(loss), _p(scratch), C.c_int(B), C.c_int(im.shape[1]),
              C.c_int(H), C.c_int(W), _stream(d))
        ctx.save_for_backward(d, im)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        d, im = ctx.saved_tensors
        g = _f32c(g.reshape(1), "grad")
        B, _, H, W = d.shape
        gd = torch.empty_like(d)
        _call("md2_smooth_loss_backward", d.device, _p(g), _p(d), _p(im), _p(gd), C.c_int(B), C.c_int(im.shape[1]),
              C.c_int(H), C.c_int(W), _stream(d))
        return gd, None


def get_smooth_loss(disp, img):
    """Edge-aware smoothness of a disparity image (layers.py:202-215); differentiable w.r.t. disp."""
    return _Smooth.apply(disp, img)


# ------------------------------------------------------------------ decoder tail feeding the path (SURVEY.md 8f-4)
_HEAD_DTYPES = {torch.float32: _capi.DTYPE_F32, torch.bfloat16: _capi.DTYPE_BF16, torch.float16: _capi.DTYPE_F16}


def _head_map(t: torch.Tensor, name: str, dtype=None) -> torch.Tensor:
    """A feature-map-side tensor of the head: CUDA, float32 / bfloat16 / float16 (``dtype`` when given)."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor (monodepth2_b200.layers has no CPU path)" % name)
    if t.dtype not in _HEAD_DTYPES or (dtype is not None and t.dtype != dtype):
        raise RuntimeError("%s must be %s, got %s" % (name, dtype or "float32, bfloat16 or float16", t.dtype))
    return t.contiguous()


class _DispHead(torch.autograd.Function):
    """sigmoid(Conv3x3(C -> 1)(x)) in one pass (md2_dispconv_sigmoid_typed): networks/depth_decoder.py:60-63.

    ``x`` may be float32, bfloat16 or float16 (what the decoder gives under ``torch.autocast``); ``disp`` and the
    gradient of ``x`` come back in ``x``'s dtype, the weight and bias gradients in float32.  A reduced-precision ``x`` is
    read at 2 bytes a value and widened exactly; weights and bias are read in float32 as stored - more accurate than
    autocast's own ``conv2d``, which rounds the weights to bfloat16 - and ``disp`` is the float32 result rounded once
    (nearest-even): bitwise the float32 head on ``x.float()``, then ``.to(x.dtype)``."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x, w, b = _head_map(x, "x"), _f32c(weight, "weight"), _f32c(bias, "bias")
        B, Cc, H, W = x.shape
        if tuple(w.shape) != (1, Cc, 3, 3) or b.numel() != 1:
            raise RuntimeError("DispConvSigmoid: weight %s / bias %s do not fit x %s" % (tuple(w.shape), tuple(b.shape), tuple(x.shape)))
        disp = torch.empty((B, 1, H, W), dtype=x.dtype, device=x.device)
        _call("md2_dispconv_sigmoid_typed", x.device, _p(x), _p(w), _p(b), _p(disp), C.c_int(_HEAD_DTYPES[x.dtype]),
              C.c_int(B), C.c_int(Cc), C.c_int(H), C.c_int(W), _stream(x))
        ctx.save_for_backward(x, w, disp)
        return disp

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        x, w, disp = ctx.saved_tensors
        g = _head_map(g, "grad_disp", x.dtype)
        B, Cc, H, W = x.shape
        gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        gw = torch.empty_like(w) if need_w else None
        gb = torch.empty(1, dtype=torch.float32, device=x.device) if need_w else None
        _call("md2_dispconv_sigmoid_backward_typed", x.device, _p(g), _p(disp), _p(x), _p(w),
              _p(gx) if gx is not None else None, _p(gw) if gw is not None else None,
              _p(gb) if gb is not None else None, C.c_int(_HEAD_DTYPES[x.dtype]), C.c_int(B), C.c_int(Cc), C.c_int(H),
              C.c_int(W), _stream(x))
        return gx, (gw if ctx.needs_input_grad[1] else None), (gb if ctx.needs_input_grad[2] else None)


class DispConvSigmoid(nn.Module):
    """Drop-in for ``sigmoid(Conv3x3(C, 1)(x))`` - the disparity head of DepthDecoder
    (/root/reference/networks/depth_decoder.py:43-44,60-63).  Same parameter names as ``Conv3x3`` (``conv.weight``,
    ``conv.bias``), so checkpoints load unchanged; reflection padding only (what the reference uses)."""

    def __init__(self, in_channels, out_channels=1, use_refl=True):
        super().__init__()
        if int(out_channels) != 1 or not use_refl:
            raise RuntimeError("DispConvSigmoid: one output channel, reflection padding")
        self.conv = nn.Conv2d(int(in_channels), 1, 3)

    def forward(self, x):
        return _DispHead.apply(x, self.conv.weight, self.conv.bias)


def fuse_disp_heads(depth_decoder):
    """Replace every ``("dispconv", s)`` Conv3x3 of a reference DepthDecoder by a DispConvSigmoid that shares its
    parameters, and its trailing ``sigmoid`` by the identity: ``decoder.forward`` (depth_decoder.py:48-65) then hands
    ``outputs[("disp", s)]`` straight from the fused head.  Under ``torch.autocast`` the decoder's feature maps are
    bfloat16 / float16 and so are the disparities it hands on (see ``_DispHead``).  Returns the decoder."""
    for key, mod in list(depth_decoder.convs.items()):
        if not (isinstance(key, tuple) and key[0] == "dispconv"):
            continue
        head = DispConvSigmoid(mod.conv.in_channels)
        head.conv = mod.conv                                     # the same Parameter objects
        depth_decoder.convs[key] = head
        for i, m in enumerate(depth_decoder.decoder):
            if m is mod:
                depth_decoder.decoder[i] = head
    depth_decoder.sigmoid = nn.Identity()
    return depth_decoder


class _UpcatPad(torch.autograd.Function):
    """ReflectionPad2d(1)(cat([nearest_up(x, up), skip], 1)) in one pass (md2_upcat_pad), gather-form backward
    without atomics (md2_upcat_pad_backward).  ``x`` and ``skip`` share one dtype here (``upcat_pad`` promotes)."""

    @staticmethod
    def forward(ctx, x, skip, up):
        x = x.contiguous()
        B, Cx, h, w = x.shape
        Cs = 0
        if skip is not None:
            skip = skip.contiguous()
            if skip.dim() != 4 or skip.shape[0] != B or tuple(skip.shape[2:]) != (up * h, up * w):
                raise RuntimeError("upcat_pad: skip %s does not fit x %s up-sampled %dx"
                                   % (tuple(skip.shape), tuple(x.shape), up))
            Cs = skip.shape[1]
        out = torch.empty((B, Cx + Cs, up * h + 2, up * w + 2), dtype=x.dtype, device=x.device)
        ctx.dims = (_HEAD_DTYPES[x.dtype], B, Cx, Cs, h, w, up)
        _call("md2_upcat_pad", x.device, _p(x), _p(skip), _p(out), *ctx.dims, _stream(x))
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        dt, B, Cx, Cs, h, w, up = ctx.dims
        g = g.contiguous()
        gx = torch.empty((B, Cx, h, w), dtype=g.dtype, device=g.device) if ctx.needs_input_grad[0] else None
        gs = (torch.empty((B, Cs, up * h, up * w), dtype=g.dtype, device=g.device)
              if Cs and ctx.needs_input_grad[1] else None)
        if gx is not None or gs is not None:
            _call("md2_upcat_pad_backward", g.device, _p(g), _p(gx), _p(gs), *ctx.dims, _stream(g))
        return gx, gs, None


def upcat_pad(x, skip=None, up=2):
    """``F.pad(torch.cat([upsample(x), skip], 1), (1, 1, 1, 1), mode="reflect")`` - the input of a decoder ConvBlock
    (networks/depth_decoder.py:48-65) - in one pass; ``up=1`` without a skip is the plain reflection pad of Conv3x3
    (layers.py:119-136).  ``x`` (B,Cx,h,w) and ``skip`` (B,Cs,up*h,up*w) are CUDA float32, bfloat16 or float16; the
    forward is bit-identical to torch's chain.  A skip of another dtype is promoted as ``torch.cat`` does (the narrower
    tensor is widened with ``.to()``); each gradient comes back in its input's dtype, summed in float32 without atomics
    and rounded once, so the backward is reproducible under ``torch.use_deterministic_algorithms(True)``."""
    tensors = [(x, "x")] + ([(skip, "skip")] if skip is not None else [])
    for t, name in tensors:
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError("upcat_pad: %s must be a CUDA tensor (monodepth2_b200.layers has no CPU path)" % name)
        if t.dtype not in _HEAD_DTYPES:
            raise RuntimeError("upcat_pad: %s must be float32, bfloat16 or float16, got %s" % (name, t.dtype))
        if t.dim() != 4:
            raise RuntimeError("upcat_pad: %s must be 4-D (B,C,H,W), got %s" % (name, tuple(t.shape)))
    up = int(up)
    if up not in (1, 2):
        raise RuntimeError("upcat_pad: up must be 1 or 2, got %d" % up)
    if skip is not None and skip.dtype != x.dtype:
        dt = torch.promote_types(x.dtype, skip.dtype)
        x, skip = x.to(dt), skip.to(dt)
    return _UpcatPad.apply(x, skip, up)


def _decoder_block(mod, key):
    """The padding-free conv and the nonlinearity of a reference ConvBlock (layers.py:106-118) with a
    reflection-padded Conv3x3 (layers.py:121-136); RuntimeError on anything else."""
    conv3 = getattr(mod, "conv", None)
    if not (isinstance(getattr(mod, "nonlin", None), nn.Module) and _is_reflect_conv3x3(conv3)):
        raise RuntimeError("fuse_decoder_stages: convs[%r] is not a ConvBlock with a reflection-padded Conv3x3: %s"
                           % (key, type(mod).__name__))
    return conv3.conv, mod.nonlin


def _is_reflect_conv3x3(m):
    conv = getattr(m, "conv", None)
    return (isinstance(getattr(m, "pad", None), nn.ReflectionPad2d) and tuple(m.pad.padding) == (1, 1, 1, 1)
            and isinstance(conv, nn.Conv2d) and tuple(conv.kernel_size) == (3, 3) and tuple(conv.padding) == (0, 0)
            and tuple(conv.stride) == (1, 1) and tuple(conv.dilation) == (1, 1) and conv.groups == 1)


def _check_head(mod, key):
    if not (isinstance(mod, DispConvSigmoid) or _is_reflect_conv3x3(mod)):
        raise RuntimeError("fuse_decoder_stages: convs[%r] is neither a DispConvSigmoid nor a reflection-padded "
                           "Conv3x3: %s" % (key, type(mod).__name__))


def _fused_decoder_forward(self, input_features):
    """DepthDecoder.forward (networks/depth_decoder.py:48-65) with every pad / upsample / cat done by upcat_pad."""
    self.outputs = {}
    x = input_features[-1]
    for i in range(4, -1, -1):
        conv, nonlin = _decoder_block(self.convs[("upconv", i, 0)], ("upconv", i, 0))
        x = nonlin(conv(upcat_pad(x, up=1)))
        skip = input_features[i - 1] if self.use_skips and i > 0 else None
        conv, nonlin = _decoder_block(self.convs[("upconv", i, 1)], ("upconv", i, 1))
        x = nonlin(conv(upcat_pad(x, skip, up=2)))
        if i in self.scales:
            head = self.convs[("dispconv", i)]
            _check_head(head, ("dispconv", i))
            y = head(x) if isinstance(head, DispConvSigmoid) else head.conv(upcat_pad(x, up=1))
            self.outputs[("disp", i)] = self.sigmoid(y)
    return self.outputs


def fuse_decoder_stages(depth_decoder):
    """Run every ConvBlock input of a reference DepthDecoder (networks/depth_decoder.py:17-65) through ``upcat_pad``:
    the forward installed on ``depth_decoder`` keeps the reference's dataflow (``use_skips``, ``scales``,
    ``num_output_channels``; it sets and returns ``self.outputs``) but runs each ConvBlock as
    ``nonlin(conv.conv(upcat_pad(...)))`` - one pass instead of upsample + torch.cat + ReflectionPad2d, and a backward
    without atomics.  A head fused by ``fuse_disp_heads`` is called as it is; a plain Conv3x3 head runs as
    ``conv.conv(upcat_pad(x, up=1))``.  Either fuse call may come first.  No module or Parameter is replaced, so
    ``state_dict`` keys and values are unchanged.  RuntimeError on a structure this does not recognise (no
    ``convs[("upconv", i, j)]``, a zero-padded Conv3x3).  Returns the decoder."""
    convs = getattr(depth_decoder, "convs", None)
    if convs is None or not hasattr(convs, "items"):
        raise RuntimeError("fuse_decoder_stages: %s has no convs dict of a reference DepthDecoder"
                           % type(depth_decoder).__name__)
    for i in range(4, -1, -1):
        for j in (0, 1):
            if ("upconv", i, j) not in convs:
                raise RuntimeError("fuse_decoder_stages: %s has no convs[('upconv', %d, %d)]"
                                   % (type(depth_decoder).__name__, i, j))
            _decoder_block(convs[("upconv", i, j)], ("upconv", i, j))
    for s in getattr(depth_decoder, "scales", ()):
        if ("dispconv", s) not in convs:
            raise RuntimeError("fuse_decoder_stages: scale %r has no convs[('dispconv', %r)]" % (s, s))
        _check_head(convs[("dispconv", s)], ("dispconv", s))
    for attr in ("use_skips", "scales", "sigmoid"):
        if not hasattr(depth_decoder, attr):
            raise RuntimeError("fuse_decoder_stages: %s has no %r attribute" % (type(depth_decoder).__name__, attr))
    depth_decoder.forward = types.MethodType(_fused_decoder_forward, depth_decoder)
    return depth_decoder


# ------------------------------------------------------------------ monitoring path (SURVEY.md 8f-5)
DEPTH_METRIC_NAMES = ["de/abs_rel", "de/sq_rel", "de/rms", "de/log_rms", "da/a1", "da/a2", "da/a3"]   # trainer.py:105-106


def depth_metrics(depth_pred, depth_gt, crop=(153, 371, 44, 1197)):
    """``Trainer.compute_depth_losses`` (/root/reference/trainer.py:498-526) as one fused call: bilinear up-sampling of
    ``outputs[("depth", 0, 0)]`` to the ground-truth size, clamp, gt > 0 and Garg/Eigen crop mask, median scaling and
    the seven metrics of ``compute_depth_errors`` (layers.py:251-269).  Returns a (7,) CUDA tensor in the order of
    ``DEPTH_METRIC_NAMES``; nothing is synchronised with the host."""
    d = _f32c(depth_pred.detach(), "depth_pred")
    g = _f32c(depth_gt, "depth_gt")
    B, _, H, W = d.shape
    Hg, Wg = g.shape[-2:]
    lib = _lib()
    n = C.c_size_t(0)
    _capi.check(lib, lib.md2_depth_metrics_scratch_bytes(B, Hg, Wg, C.byref(n)), "md2_depth_metrics_scratch_bytes")
    scratch = torch.empty(n.value, dtype=torch.uint8, device=d.device)
    out = torch.empty(7, dtype=torch.float32, device=d.device)
    _call("md2_depth_metrics", d.device, _p(d), _p(g), _p(out), _p(scratch), scratch.numel(), B, H, W, Hg, Wg,
          int(crop[0]), int(crop[1]), int(crop[2]), int(crop[3]), _stream(d))
    return out


# ------------------------------------------------------------------ off-path symbols kept importable
# (decoder building blocks / monitoring metric: OUT OF SCOPE per SURVEY.md 2.1 rows 3; stock PyTorch)
class Conv3x3(nn.Module):
    """Pad and convolve (layers.py:121-136); cuDNN, unchanged semantics."""

    def __init__(self, in_channels, out_channels, use_refl=True):
        super().__init__()
        self.pad = nn.ReflectionPad2d(1) if use_refl else nn.ZeroPad2d(1)
        self.conv = nn.Conv2d(int(in_channels), int(out_channels), 3)

    def forward(self, x):
        return self.conv(self.pad(x))


class ConvBlock(nn.Module):
    """Conv3x3 + ELU (layers.py:106-118)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv = Conv3x3(in_channels, out_channels)
        self.nonlin = nn.ELU(inplace=True)

    def forward(self, x):
        return self.nonlin(self.conv(x))


def upsample(x):
    """Nearest 2x up-sampling (layers.py:196-199)."""
    return F.interpolate(x, scale_factor=2, mode="nearest")


def compute_depth_errors(gt, pred):
    """Monitoring metrics (layers.py:251-269)."""
    thresh = torch.max(gt / pred, pred / gt)
    a1, a2, a3 = ((thresh < 1.25 ** k).float().mean() for k in (1, 2, 3))
    rmse = torch.sqrt(((gt - pred) ** 2).mean())
    rmse_log = torch.sqrt(((torch.log(gt) - torch.log(pred)) ** 2).mean())
    abs_rel = torch.mean(torch.abs(gt - pred) / gt)
    sq_rel = torch.mean((gt - pred) ** 2 / gt)
    return abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3
