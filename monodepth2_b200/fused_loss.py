"""Host side of the fused view-synthesis loss: a ``torch.autograd.Function`` over the
C ABI (include/md2_loss.h) and drop-in replacements for the two Trainer methods.

Replaces, in one call into libmd2loss.so,
``Trainer.generate_images_pred`` (/root/reference/trainer.py:341-391) and
``Trainer.compute_losses`` (/root/reference/trainer.py:407-496); gradients flow to
``outputs[("disp", s)]`` and ``outputs[("cam_T_cam", 0, f)]`` exactly where
``losses["loss"].backward()`` (trainer.py:208) would send them.  PyTorch is used for
device memory, streams and autograd plumbing only; there is no PyTorch or CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence

import torch

from . import _capi
from ._capi import MAX_SCALES, Md2Problem, Md2Tensors


def _check_f32_cuda(t: torch.Tensor, name: str, shape=None) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor (the fused loss has no CPU path)" % name)
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32, got %s" % (name, t.dtype))
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise RuntimeError("%s has shape %s, expected %s" % (name, tuple(t.shape), tuple(shape)))
    return t.contiguous()


# element types a differentiable leaf may have (md2_problem.disp_dtype / pose_dtype / pmask_dtype)
_LEAF_DTYPES = {torch.float32: _capi.DTYPE_F32, torch.bfloat16: _capi.DTYPE_BF16, torch.float16: _capi.DTYPE_F16}


def _check_leaf_cuda(t: torch.Tensor, name: str, shape=None) -> torch.Tensor:
    """A differentiable leaf: float32, bfloat16 or float16 (what the networks give under torch.autocast).  A narrower
    leaf is widened exactly inside the call; nothing here converts it."""
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor (the fused loss has no CPU path)" % name)
    if t.dtype not in _LEAF_DTYPES:
        raise RuntimeError("%s must be float32, bfloat16 or float16, got %s" % (name, t.dtype))
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise RuntimeError("%s has shape %s, expected %s" % (name, tuple(t.shape), tuple(shape)))
    return t.contiguous()


def _one_dtype(tensors: Sequence, names: Sequence[str], what: str) -> int:
    """The md2_dtype shared by ``tensors``; a mix raises, naming each tensor and its dtype."""
    dts = [t.dtype for t in tensors]
    if len(set(dts)) > 1 or any(d not in _LEAF_DTYPES for d in dts):
        raise RuntimeError("%s must share one dtype out of float32, bfloat16 and float16, got %s"
                           % (what, ", ".join("%s %s" % (n, d) for n, d in zip(names, dts))))
    return _LEAF_DTYPES[dts[0]] if dts else _capi.DTYPE_F32


def _check_u8_cuda(t: torch.Tensor, name: str, B: int, H: int, W: int, hwc: bool) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor (the fused loss has no CPU path)" % name)
    shape = (B, H, W, 3) if hwc else (B, 3, H, W)
    if t.dtype != torch.uint8 or tuple(t.shape) != shape:
        raise RuntimeError("%s must be uint8 of shape %s, got %s %s" % (name, shape, t.dtype, tuple(t.shape)))
    return t.contiguous()


class LossPlan:
    """Static description of one loss configuration (mirrors the ``opt`` flags the path reads)."""

    def __init__(self, batch_size: int, height: int, width: int, frame_ids: Sequence,
                 scales: Sequence[int] = (0, 1, 2, 3), min_depth: float = 0.1, max_depth: float = 100.0,
                 disparity_smoothness: float = 1e-3, avg_reprojection: bool = False,
                 disable_automasking: bool = False, align_corners: bool = False,
                 rows_per_segment: int = 0, no_ssim: bool = False, v1_multiscale: bool = False,
                 posecnn: bool = False, predictive_mask: bool = False):
        # --scales (options.py:64) is any list of pyramid levels: trainer.py:345,413 iterate it, the decoder emits
        # ("disp", s) for exactly those levels and the dataloader always holds levels 0..3 (trainer.py:127-135).  The
        # loss is a sum over the list, so the order does not matter: the plan keeps the levels ascending
        # (md2_problem.scale_level); slot i of every per-scale array is level self.scales[i].
        self.scales_given = [int(s) for s in scales]     # the order trainer.py:413 iterates (and draws the noise in)
        scales = sorted(self.scales_given)
        if not scales or len(set(scales)) != len(scales) or scales[0] < 0 or scales[-1] >= MAX_SCALES:
            raise RuntimeError("scales must be distinct pyramid levels in 0..%d, got %s" % (MAX_SCALES - 1, scales))
        if scales[0] != 0 and not v1_multiscale:
            # the reference warps at source_scale 0 with backproject_depth[0] / project_3d[0], which exist only when 0 is
            # in opt.scales (trainer.py:151-159,377: KeyError otherwise)
            raise RuntimeError("scales must contain level 0 (trainer.py:377 indexes backproject_depth[0]), got %s" % scales)
        self.batch_size, self.height, self.width = int(batch_size), int(height), int(width)
        self.frame_ids = list(frame_ids)
        self.src_ids = self.frame_ids[1:]
        self.scales = list(scales)
        self.min_depth, self.max_depth = float(min_depth), float(max_depth)
        self.disparity_smoothness = float(disparity_smoothness)
        self.avg_reprojection = bool(avg_reprojection)
        self.automask = not bool(disable_automasking)
        self.align_corners = bool(align_corners)
        self.rows_per_segment = int(rows_per_segment)
        self.no_ssim = bool(no_ssim)
        self.v1_multiscale = bool(v1_multiscale)
        # --pose_model_type posecnn (trainer.py:366-375) and --predictive_mask (trainer.py:447-459) are variants of
        # the fused kernels themselves (md2_problem.posecnn / .predictive_mask)
        self.posecnn = bool(posecnn)
        # --predictive_mask needs --disable_automasking (trainer.py:90-92)
        self.predictive_mask = bool(predictive_mask)
        if self.predictive_mask and self.automask:
            raise RuntimeError("When using predictive_mask, please disable automasking with --disable_automasking")
        self.n_src = len(self.src_ids)
        self.n_id = 0 if not self.automask else (1 if self.avg_reprojection else self.n_src)
        self.lib = _capi.load_library()
        self._workspace: Dict = {}
        # --v1_multiscale (trainer.py:347-352,417-420): every scale is an independent single-scale
        # problem at its own resolution, with its own K / inv_K / colour pyramid level
        self._scale_plans = None
        if self.v1_multiscale:
            self._scale_plans = [
                LossPlan(self.batch_size, self.height >> s, self.width >> s, self.frame_ids, [0], self.min_depth,
                         self.max_depth, self.disparity_smoothness / (2 ** s), self.avg_reprojection,
                         not self.automask, self.align_corners, self.rows_per_segment, self.no_ssim, False,
                         self.posecnn, self.predictive_mask)
                for s in self.scales]

    @classmethod
    def from_opt(cls, opt, **kw) -> "LossPlan":
        """Build from a reference ``options.py`` namespace (after trainer.py:51-52 appended "s")."""
        return cls(opt.batch_size, opt.height, opt.width, opt.frame_ids, opt.scales, opt.min_depth,
                   opt.max_depth, opt.disparity_smoothness, opt.avg_reprojection,
                   opt.disable_automasking, no_ssim=getattr(opt, "no_ssim", False),
                   v1_multiscale=getattr(opt, "v1_multiscale", False),
                   posecnn=(getattr(opt, "pose_model_type", "separate_resnet") == "posecnn"),
                   predictive_mask=getattr(opt, "predictive_mask", False), **kw)

    def problem(self, want_grad: bool, dtypes=None) -> Md2Problem:
        """``dtypes`` = (disp_dtype, (pose_dtype per source), pmask_dtype) of md2_problem; None = every leaf fp32."""
        disp_dt, pose_dt, pmask_dt = dtypes or (0, (), 0)
        pose = (C.c_int * _capi.MAX_SRC)(*pose_dt)
        return Md2Problem(disp_dtype=disp_dt, pose_dtype=pose, pmask_dtype=pmask_dt,batch=self.batch_size, height=self.height, width=self.width,
                          num_scales=len(self.scales), num_src=self.n_src, automask=int(self.automask),
                          avg_reprojection=int(self.avg_reprojection), align_corners=int(self.align_corners),
                          min_depth=self.min_depth, max_depth=self.max_depth,
                          disparity_smoothness=self.disparity_smoothness, want_grad=int(want_grad),
                          rows_per_segment=self.rows_per_segment, no_ssim=int(self.no_ssim),
                          posecnn=int(self.posecnn), predictive_mask=int(self.predictive_mask),
                          scale_level=self._levels())

    def _levels(self):
        """md2_problem.scale_level: all zero for the default 0..n-1, else the levels."""
        lv = (C.c_int * MAX_SCALES)()
        if self.scales != list(range(len(self.scales))):
            for i, s in enumerate(self.scales):
                lv[i] = s
        return lv

    def slot(self, level: int) -> int:
        """Index of pyramid level ``level`` in the per-scale arrays of the C ABI."""
        return self.scales.index(level)

    def workspace(self, device: torch.device, dtypes=None) -> torch.Tensor:
        """The call's device scratch; reduced-precision leaves (``dtypes``, see ``problem``) add their fp32 copies."""
        narrow = dtypes is not None and (dtypes[0] or any(dtypes[1]) or dtypes[2])
        key = (device.type, device.index) + ((dtypes,) if narrow else ())
        ws = self._workspace.get(key)
        if ws is None:
            n = C.c_size_t(0)
            p = self.problem(True, dtypes)
            _capi.check(self.lib, self.lib.md2_loss_workspace_bytes(C.byref(p), C.byref(n)), "md2_loss_workspace_bytes")
            ws = torch.empty(n.value, dtype=torch.uint8, device=device)
            self._workspace[key] = ws
        return ws


class _ViewSynthesisLossFn(torch.autograd.Function):
    """forward(plan, side, target, sources, K, inv_K, colors, noise, pose_grad, pose_invert, *leaves)

    leaves = S disparities, then per source the matrix T (B,4,4) *or* the axisangle leaf, then per source
    the translation leaf (None for a source given as a matrix), then (--predictive_mask) S masks.
    ``pose_invert[i]`` is None for a matrix source, else the ``invert`` flag of
    transformation_from_parameters (frame_id < 0)."""

    N_FIXED = 10

    @staticmethod
    def forward(ctx, plan: LossPlan, side: Optional[dict], target, sources, K, inv_K, colors, noise, pose_grad,
                pose_invert, *leaves):
        S, F = len(plan.scales), plan.n_src
        disps, firsts, seconds = leaves[:S], leaves[S:S + F], leaves[S + F:S + 2 * F]
        masks = leaves[S + 2 * F:S + 2 * F + S] if plan.predictive_mask else ()
        B, H, W = plan.batch_size, plan.height, plan.width
        dev = target.device
        want_grad = any(ctx.needs_input_grad[_ViewSynthesisLossFn.N_FIXED:])
        t = Md2Tensors()
        keep = []

        def ptr(x):
            keep.append(x)
            return x.data_ptr()

        def pose_leaf(x, name):
            # (B,3) / (B,1,3) view whose 3 components are adjacent; any batch stride (e.g. the [:, 0] view of
            # PoseDecoder's (B,2,1,3) output, pose_decoder.py:49-54)
            if not x.is_cuda or x.dtype not in _LEAF_DTYPES:
                raise RuntimeError("%s must be a CUDA float32, bfloat16 or float16 tensor, got %s" % (name, x.dtype))
            if x.numel() != B * 3 or x.shape[0] != B or x.shape[-1] != 3:
                raise RuntimeError("%s has shape %s, expected (%d,1,3)" % (name, tuple(x.shape), B))
            if x.stride(-1) != 1 or (B > 1 and x.stride(0) < 3):
                x = x.contiguous()
            return x, (x.stride(0) if B > 1 else 3)

        # uint8 frames (what the dataloader holds before ToTensor, mono_dataset.py:106-109): (B,H,W,3) or
        # (B,3,H,W); converted with x / 255 inside the kernels, a quarter of the host-to-device bytes
        u8 = target.dtype == torch.uint8
        hwc = u8 and target.dim() == 4 and target.shape[-1] == 3 and target.shape[1] != 3
        if u8:
            t.target_u8 = ptr(_check_u8_cuda(target, "target", B, H, W, hwc))
            t.u8_hwc = int(hwc)
        else:
            t.target = ptr(_check_f32_cuda(target, "target", (B, 3, H, W)))
        cam_T = [None] * F
        grad_first, grad_second = [None] * F, [None] * F
        # one dtype for all disparities, one for all masks, one per source (T, or the axisangle / translation pair)
        disp_dt = _one_dtype(disps, ["disp[%d]" % s for s in range(S)], "the disparities")
        mask_dt = _one_dtype(masks, ["predictive_mask[%d]" % s for s in range(S)], "the predictive masks")
        pose_dt = [_one_dtype([x for x in (firsts[i], seconds[i]) if x is not None],
                              ["axisangle[%d]" % i, "translation[%d]" % i] if pose_invert[i] is not None else ["T[%d]" % i],
                              "the pose leaves of source %d" % i) for i in range(F)]
        dtypes = (disp_dt, tuple(pose_dt), mask_dt)
        for i in range(F):
            if u8:
                t.source_u8[i] = ptr(_check_u8_cuda(sources[i], "source[%d]" % i, B, H, W, hwc))
            else:
                t.source[i] = ptr(_check_f32_cuda(sources[i], "source[%d]" % i, (B, 3, H, W)))
            t.pose_requires_grad[i] = int(bool(pose_grad[i]))
            if pose_invert[i] is None:
                t.T[i] = ptr(_check_leaf_cuda(firsts[i], "T[%d]" % i, (B, 4, 4)))
                if want_grad:
                    grad_first[i] = torch.empty((B, 4, 4), dtype=torch.float32, device=dev)
                    t.grad_T[i] = ptr(grad_first[i])
            else:
                aa, sa = pose_leaf(firsts[i], "axisangle[%d]" % i)
                tr, st_ = pose_leaf(seconds[i], "translation[%d]" % i)
                if sa != st_:
                    tr = tr.contiguous(); aa = aa.contiguous(); sa = 3
                t.axisangle[i], t.translation[i] = ptr(aa), ptr(tr)
                t.pose_stride[i], t.pose_invert[i] = int(sa), int(bool(pose_invert[i]))
                cam_T[i] = torch.empty((B, 4, 4), dtype=torch.float32, device=dev)
                t.cam_T_cam[i] = ptr(cam_T[i])
                if want_grad and pose_grad[i]:
                    grad_first[i] = torch.empty((B, 3), dtype=torch.float32, device=dev)
                    grad_second[i] = torch.empty((B, 3), dtype=torch.float32, device=dev)
                    t.grad_axisangle[i], t.grad_translation[i] = ptr(grad_first[i]), ptr(grad_second[i])
        t.K = ptr(_check_f32_cuda(K, "K", (B, 4, 4)))
        t.inv_K = ptr(_check_f32_cuda(inv_K, "inv_K", (B, 4, 4)))
        grad_disp = []
        grad_mask = [None] * S
        for s in range(S):
            hs, ws = H >> plan.scales[s], W >> plan.scales[s]
            t.disp[s] = ptr(_check_leaf_cuda(disps[s], "disp[%d]" % s, (B, 1, hs, ws)))
            if u8:
                t.color_u8[s] = ptr(_check_u8_cuda(colors[s], "color[%d]" % s, B, hs, ws, hwc))
            else:
                t.color[s] = ptr(_check_f32_cuda(colors[s], "color[%d]" % s, (B, 3, hs, ws)))
            if plan.n_id > 0:
                t.noise[s] = ptr(_check_f32_cuda(noise[s], "noise[%d]" % s, (B, plan.n_id, H, W)))
                ready = getattr(noise, "ready", None)
                if ready is not None:
                    keep.append(ready)
                    t.noise_ready_event = ready.cuda_event
            if want_grad:
                g = torch.empty((B, 1, hs, ws), dtype=torch.float32, device=dev)
                grad_disp.append(g)
                t.grad_disp[s] = ptr(g)
            if plan.predictive_mask:
                t.pmask[s] = ptr(_check_leaf_cuda(masks[s], "predictive_mask[%d]" % s, (B, F, hs, ws)))
                if want_grad and ctx.needs_input_grad[_ViewSynthesisLossFn.N_FIXED + S + 2 * F + s]:
                    g = torch.empty((B, F, hs, ws), dtype=torch.float32, device=dev)
                    grad_mask[s] = g
                    t.grad_pmask[s] = ptr(g)
        if side is not None:
            for s in side.get("depth_scales", []):
                d = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
                side[("depth", 0, s)] = d
                t.depth[plan.slot(s)] = ptr(d)
            for s in side.get("color_scales", []):
                for i, f in enumerate(plan.src_ids):
                    c = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
                    side[("color", f, s)] = c
                    t.warped[i][plan.slot(s)] = ptr(c)
            if plan.automask:
                for s in side.get("mask_scales", []):
                    m = torch.empty((B, H, W), dtype=torch.float32, device=dev)
                    side["identity_selection/{}".format(s)] = m
                    t.identity_selection[plan.slot(s)] = ptr(m)
            if want_grad:
                for s in side.get("grad_updisp_scales", []):
                    gd = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
                    side[("grad_updisp", s)] = gd
                    t.grad_depth_dbg[plan.slot(s)] = ptr(gd)
            side["_cam_T_cam"] = cam_T
        losses = torch.empty(MAX_SCALES + 1, dtype=torch.float32, device=dev)
        t.losses = ptr(losses)
        ws_buf = plan.workspace(dev, dtypes)
        p = plan.problem(want_grad, dtypes)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream().cuda_stream
            st = plan.lib.md2_view_synthesis_loss(C.byref(p), C.byref(t), ws_buf.data_ptr(), ws_buf.numel(),
                                                  C.c_void_p(stream))
        _capi.check(plan.lib, st, "md2_view_synthesis_loss")
        ctx.S, ctx.F = S, F
        ctx.lib = plan.lib
        ctx.pose_grad = list(pose_grad)
        ctx.first_shapes = [tuple(x.shape) for x in firsts]
        ctx.second_shapes = [tuple(x.shape) if x is not None else None for x in seconds]
        ctx.have = [(grad_first[i] is not None, grad_second[i] is not None) for i in range(F)]
        ctx.have_mask = [g is not None for g in grad_mask]
        ctx.n_leaves = len(leaves)
        ctx.leaf_dtypes = [x.dtype if x is not None else None for x in leaves]
        if want_grad:
            ctx.save_for_backward(*grad_disp, *[g for g in grad_first if g is not None],
                                  *[g for g in grad_second if g is not None],
                                  *[g for g in grad_mask if g is not None])
        total = losses[0]
        per_scale = losses[1:1 + S]
        ctx.mark_non_differentiable(per_scale)
        return total, per_scale

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_total, _g_scales):
        saved = list(ctx.saved_tensors)
        S, F = ctx.S, ctx.F
        n0 = _ViewSynthesisLossFn.N_FIXED
        # every stored gradient times the incoming scalar, all tensors in ONE launch (md2_scale_tensors); a bf16 / fp16
        # leaf gets the fp32 product rounded once to its dtype (md2_scale_tensors_typed): the scalar - a GradScaler
        # scale, a loss weight - is applied before the rounding, so scaled fp16 gradients do not flush to zero
        want = []           # (slot in the result tuple, stored gradient, shape)
        for s in range(S):
            if ctx.needs_input_grad[n0 + s]:
                want.append((n0 + s, saved[s], saved[s].shape))
        n1, n2 = sum(1 for h in ctx.have if h[0]), sum(1 for h in ctx.have if h[1])
        firsts = iter(saved[S:S + n1])
        seconds = iter(saved[S + n1:S + n1 + n2])
        gmasks = iter(saved[S + n1 + n2:])
        for i in range(F):
            a = next(firsts) if ctx.have[i][0] else None
            b = next(seconds) if ctx.have[i][1] else None
            if ctx.needs_input_grad[n0 + S + i] and ctx.pose_grad[i] and a is not None:
                want.append((n0 + S + i, a, ctx.first_shapes[i]))
            if ctx.needs_input_grad[n0 + S + F + i] and ctx.pose_grad[i] and b is not None:
                want.append((n0 + S + F + i, b, ctx.second_shapes[i]))
        for s, have in enumerate(ctx.have_mask):
            if have:
                gm = next(gmasks)
                want.append((n0 + S + 2 * F + s, gm, gm.shape))
        out = [None] * (n0 + ctx.n_leaves)
        if want:
            n = len(want)
            dts = [ctx.leaf_dtypes[w[0] - n0] for w in want]
            res = [torch.empty_like(w[1], dtype=d) for w, d in zip(want, dts)]
            g = g_total.detach().to(torch.float32).contiguous()
            src = (C.c_void_p * n)(*[w[1].data_ptr() for w in want])
            dst = (C.c_void_p * n)(*[r.data_ptr() for r in res])
            cnt = (C.c_longlong * n)(*[w[1].numel() for w in want])
            with torch.cuda.device(g.device):
                stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                if all(d == torch.float32 for d in dts):
                    name = "md2_scale_tensors"
                    st = ctx.lib.md2_scale_tensors(n, src, dst, cnt, g.data_ptr(), stream)
                else:
                    name = "md2_scale_tensors_typed"
                    dt = (C.c_int * n)(*[_LEAF_DTYPES[d] for d in dts])
                    st = ctx.lib.md2_scale_tensors_typed(n, src, dst, dt, cnt, g.data_ptr(), stream)
            _capi.check(ctx.lib, st, name)
            for w, r in zip(want, res):
                out[w[0]] = r.reshape(w[2])
        return tuple(out)


def bind_to_gpu_cpus(device) -> Optional[str]:
    """Restrict this process to the CPUs that are local to ``device`` (its PCI device's ``local_cpulist`` in sysfs), so
    that the pinned staging buffers allocated afterwards are first-touched on the GPU's NUMA node and the per-step
    host-to-device copy does not cross the socket interconnect.  What a one-process-per-GPU training loop does at
    start-up; it changes the process affinity, so it is an explicit call (bench.py makes it for its e2e leg), never
    made by the library on its own.  Returns the cpulist it bound to, or None when sysfs has nothing to say."""
    try:
        p = torch.cuda.get_device_properties(device)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        cpus = set()
        for part in txt.split(","):
            if part:
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return txt
    except Exception:
        return None


def _in_slot_order(plan: "LossPlan", drawn: list) -> list:
    """``drawn[i]`` belongs to ``plan.scales_given[i]`` (trainer.py:413,468-469: one draw per entry of opt.scales, in list
    order); the C ABI wants slot order = ascending levels.  The identity for a list given in ascending order."""
    if plan.scales_given == plan.scales:
        return drawn
    out = [None] * len(drawn)
    for i, s in enumerate(plan.scales_given):
        out[plan.slot(s)] = drawn[i]
    return out


class _Noise(list):
    """The tie-break draws of one call; ``ready`` is the torch.cuda.Event recorded after the last draw when they were
    made on the plan's side stream (handed to the library as md2_tensors.noise_ready_event)."""
    ready = None


_NOISE_STREAMS: Dict = {}


def _draw_noise(plan: LossPlan, dev) -> "_Noise":
    """trainer.py:468-469: one ``torch.randn`` per scale, in scale order, from the default CUDA generator - so the
    generator advances exactly as in the reference and the values are the ones a plain call would draw.  The four
    draws (~50 us at 640x192 x 12) do not depend on anything the call computes before the marching kernel, so they
    run on a side stream beside the prologue / identity pass; the library waits for ``ready`` right before the
    first kernel that reads them.  MD2_NOISE_STREAM=0: draw on the current stream."""
    shape = (plan.batch_size, plan.n_id, plan.height, plan.width)
    if os.environ.get("MD2_NOISE_STREAM", "1") == "0":
        return _Noise(_in_slot_order(plan, [torch.randn(shape, device=dev) for _ in plan.scales]))
    main = torch.cuda.current_stream(dev)
    key = (dev.index if dev.index is not None else torch.cuda.current_device())
    side_stream = _NOISE_STREAMS.get(key)
    if side_stream is None:
        side_stream = _NOISE_STREAMS[key] = torch.cuda.Stream(device=dev)
    # fork: everything already queued on the caller's stream - including the previous call's marching kernel, the
    # last reader of the previous draws, whose memory the allocator may hand out again - comes first
    side_stream.wait_stream(main)
    with torch.cuda.stream(side_stream):
        noise = _Noise(_in_slot_order(plan, [torch.randn(shape, device=dev) for _ in plan.scales]))
        noise.ready = torch.cuda.Event()
        noise.ready.record(side_stream)
    return noise


def view_synthesis_loss(plan: LossPlan, inputs: Dict, outputs: Dict,
                        noise: Optional[List[torch.Tensor]] = None,
                        side: Optional[dict] = None) -> Dict[str, torch.Tensor]:
    """Fused generate_images_pred + compute_losses on the reference's ``inputs``/``outputs`` dicts.

    ``noise`` (one (B,n_id,H,W) tensor per scale) replaces the ``torch.randn`` draws of
    trainer.py:468-469; when omitted they are drawn here, one call per scale in scale order, so the
    CUDA generator stream advances exactly as in the reference.
    ``side`` selects optional outputs: {"depth_scales": [...], "color_scales": [...], "mask_scales": [...]};
    the produced tensors are stored both in ``side`` and in ``outputs`` under the reference's keys.
    """
    if plan.v1_multiscale:
        return _view_synthesis_loss_v1_multiscale(plan, inputs, outputs, noise, side)
    S = len(plan.scales)
    target = inputs[("color", 0, 0)]
    dev = target.device
    sources = [inputs[("color", f, 0)] for f in plan.src_ids]
    colors = [inputs[("color", 0, s)] for s in plan.scales]
    disps = [outputs[("disp", s)] for s in plan.scales]
    firsts, seconds, pose_grad, pose_invert = [], [], [], []
    for f in plan.src_ids:
        if f == "s":
            firsts.append(inputs["stereo_T"]); seconds.append(None)
            pose_grad.append(False); pose_invert.append(None)
        elif ("cam_T_cam", 0, f) in outputs and not plan.posecnn:
            T = outputs[("cam_T_cam", 0, f)]
            firsts.append(T); seconds.append(None)
            pose_grad.append(bool(T.requires_grad) and torch.is_grad_enabled()); pose_invert.append(None)
        else:
            # pose leaves straight from the pose network (trainer.py:289-295): T is built inside the call
            # (SURVEY.md 8f rank 1) and handed back as outputs[("cam_T_cam", 0, f)]
            aa = outputs[("axisangle", 0, f)][:, 0]
            tr = outputs[("translation", 0, f)][:, 0]
            firsts.append(aa); seconds.append(tr)
            pose_grad.append(bool(aa.requires_grad or tr.requires_grad) and torch.is_grad_enabled())
            pose_invert.append(f < 0)
    if plan.n_id > 0 and noise is None:
        noise = _draw_noise(plan, dev)
    if side is None and any(pi is not None for pi in pose_invert):
        side = {}
    # --predictive_mask: outputs["predictive_mask"][("disp", s)] (trainer.py:449), (B, n_src, H>>s, W>>s)
    masks = [outputs["predictive_mask"][("disp", s)] for s in plan.scales] if plan.predictive_mask else []
    total, per_scale = _ViewSynthesisLossFn.apply(plan, side, target, sources, inputs[("K", 0)],
                                                  inputs[("inv_K", 0)], colors, noise, pose_grad, pose_invert,
                                                  *disps, *firsts, *seconds, *masks)
    if side is not None:
        for i, T in enumerate(side.pop("_cam_T_cam", [])):
            if T is not None and ("cam_T_cam", 0, plan.src_ids[i]) not in outputs:
                outputs[("cam_T_cam", 0, plan.src_ids[i])] = T
    losses = {"loss": total}
    for i, s in enumerate(plan.scales):
        losses["loss/{}".format(s)] = per_scale[i]
    if side is not None:
        for k, v in side.items():
            if isinstance(k, tuple) and k[0] in ("depth", "color") or (isinstance(k, str) and k.startswith("identity_selection/")):
                outputs[k] = v
    return losses


def _widened(x: torch.Tensor) -> torch.Tensor:
    return x.float() if x.dtype in (torch.bfloat16, torch.float16) else x


def _view_synthesis_loss_v1_multiscale(plan: LossPlan, inputs: Dict, outputs: Dict, noise, side):
    """--v1_multiscale: one single-scale fused call per pyramid level (source_scale = scale)."""
    losses: Dict[str, torch.Tensor] = {}
    total = 0
    # the pose tensors feed every per-level call: a bf16 / fp16 one is widened once, in the graph, so that autograd sums
    # the per-level gradients in fp32 and rounds the sum once to the leaf's dtype, as a single call would
    shared: Dict = {}
    for i, s in enumerate(plan.scales):
        sp = plan._scale_plans[i]
        ins = {("K", 0): inputs[("K", s)], ("inv_K", 0): inputs[("inv_K", s)]}
        if "stereo_T" in inputs:
            ins["stereo_T"] = inputs["stereo_T"]
        for f in plan.frame_ids:
            ins[("color", f, 0)] = inputs[("color", f, s)]
        outs = {("disp", 0): outputs[("disp", s)]}
        for f in plan.src_ids:
            if f != "s":       # the matrix if the caller built it, else the pose leaves (T is then built in the call)
                for key in (("cam_T_cam", 0, f), ("axisangle", 0, f), ("translation", 0, f)):
                    if key in outputs:
                        outs[key] = shared.setdefault(key, _widened(outputs[key]))
        if plan.predictive_mask:      # not up-sampled under --v1_multiscale (trainer.py:450)
            outs["predictive_mask"] = {("disp", 0): outputs["predictive_mask"][("disp", s)]}
        sub_side = None
        if side is not None:
            sub_side = {k: ([0] if s in side.get(k, []) else []) for k in
                        ("depth_scales", "color_scales", "mask_scales", "grad_updisp_scales")}
        ls = view_synthesis_loss(sp, ins, outs, [noise[i]] if noise is not None else None, sub_side)
        losses["loss/{}".format(s)] = ls["loss"]
        total = total + ls["loss"]
        if sub_side is not None:
            for k, v in sub_side.items():
                if isinstance(k, tuple):
                    key = (k[0], k[1], s) if len(k) == 3 else (k[0], s)
                    if k[0] == "grad_updisp":          # test hook: gradient of the averaged total loss
                        v = v / len(plan.scales)
                    side[key] = v
                    if k[0] in ("depth", "color"):
                        outputs[key] = v
                elif isinstance(k, str) and k.startswith("identity_selection/"):
                    side["identity_selection/{}".format(s)] = v
                    outputs["identity_selection/{}".format(s)] = v
    losses["loss"] = total / len(plan.scales)
    return losses


class GraphedLoss:
    """``view_synthesis_loss`` + ``backward()`` for a fixed plan, captured once in a CUDA graph over static device
    buffers - what a training loop with static shapes does to get rid of the launch and Python overhead of the
    eager call (the reference's own loop is eager; its ~2 100 launches per step are launch-bound, SURVEY.md 8d).

        g = GraphedLoss(plan, inputs, outputs)     # device tensors shaped like every later step's; captures
        g.load(inputs, outputs)                    # copies a step's tensors (pinned host or device) into the buffers
        loss = g.run()                             # replays; g.loss / g.grads[key] are the static results
        flat, ins, outs = g.staging()              # or: fill a pinned staging buffer (views per tensor) ...
        g.load_staged(flat)                        # ... and bring the whole step in with ONE host-to-device copy

    ``inputs`` holds the tensors the path reads (``("color", f, 0)`` float or uint8, ``("color", 0, s)``, ``("K", 0)``,
    ``("inv_K", 0)``, ``"stereo_T"``), ``outputs`` the leaves (``("disp", s)`` and ``("cam_T_cam", 0, f)`` or the pose
    leaves).  The tie-break noise is drawn inside the graph by ``torch.randn`` from the default CUDA generator
    (graph-safe), so every replay draws fresh noise as trainer.py:468-469 does.
    """

    def __init__(self, plan: LossPlan, inputs: Dict, outputs: Dict, warmup: int = 2):
        dev = inputs[("color", 0, 0)].device
        if dev.type != "cuda":
            raise RuntimeError("GraphedLoss needs CUDA tensors (there is no CPU path)")
        self.plan = plan
        # every static buffer is a view of ONE flat device allocation, so that a whole step's tensors can be brought
        # in by a single host-to-device copy from a pinned staging buffer of the same layout (staging / load_staged)
        self._layout = []          # (is_leaf, key, shape, dtype, offset, nbytes)
        off = 0
        for is_leaf, d in ((False, inputs), (True, outputs)):
            for k, v in d.items():
                if not torch.is_tensor(v):
                    continue
                n = v.numel() * v.element_size()
                self._layout.append((is_leaf, k, tuple(v.shape), v.dtype, off, n))
                off = (off + n + 255) // 256 * 256
        self._nbytes = off
        self._flat = torch.empty(off, dtype=torch.uint8, device=dev)
        self.inputs, self.leaves = self._views(self._flat)
        with torch.no_grad():
            for k, dst in self.inputs.items():
                dst.copy_(inputs[k])
            for k, dst in self.leaves.items():
                dst.copy_(outputs[k])
        for v in self.leaves.values():
            v.requires_grad_(True)
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                self._step()
        cur.wait_stream(side)
        torch.cuda.synchronize(dev)
        for v in self.leaves.values():
            v.grad = None
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.losses = self._step()
        self.loss = self.losses["loss"].detach()
        self.grads = {k: v.grad for k, v in self.leaves.items()}
        self._loss_host, self._loss_ev = None, None

    def _step(self):
        for v in self.leaves.values():
            v.grad = None
        losses = view_synthesis_loss(self.plan, self.inputs, dict(self.leaves))
        losses["loss"].backward()
        return losses

    def _views(self, flat: torch.Tensor):
        ins, leaves = {}, {}
        for is_leaf, k, shape, dtype, off, n in self._layout:
            (leaves if is_leaf else ins)[k] = flat[off:off + n].view(dtype).view(shape)
        return ins, leaves

    def staging(self):
        """A pinned host buffer laid out like the static device buffers, and its views ``(flat, inputs, outputs)``:
        what a dataloader's collate step fills.  ``load_staged(flat)`` then moves the whole step with one copy."""
        flat = torch.empty(self._nbytes, dtype=torch.uint8).pin_memory()
        ins, leaves = self._views(flat)
        return flat, ins, leaves

    def load_staged(self, flat: torch.Tensor) -> None:
        """One host-to-device copy of a staging buffer (see ``staging``) into the static buffers."""
        with torch.no_grad():
            self._flat.copy_(flat, non_blocking=True)

    def load(self, inputs: Dict, outputs: Dict) -> None:
        with torch.no_grad():
            for k, dst in self.inputs.items():
                dst.copy_(inputs[k], non_blocking=True)
            for k, dst in self.leaves.items():
                dst.copy_(outputs[k], non_blocking=True)

    def run(self) -> torch.Tensor:
        self.graph.replay()
        return self.loss

    def run_async(self) -> None:
        """Replay and put the device-to-host read of the loss in flight (pinned host slot + event) without blocking
        the host: ``read()`` returns the value later, e.g. after the next step has been enqueued - how a training
        loop reads its loss for logging without draining the GPU every step."""
        if self._loss_host is None:
            self._loss_host = torch.empty((), dtype=torch.float32).pin_memory()
            self._loss_ev = torch.cuda.Event()
        self.graph.replay()
        self._loss_host.copy_(self.loss, non_blocking=True)
        self._loss_ev.record()

    def read(self) -> float:
        """The loss of the last ``run_async()`` (waits for that step only)."""
        self._loss_ev.synchronize()
        return float(self._loss_host)


class FusedLossMixin:
    """Mix into (or bind onto) the reference ``Trainer``: overrides the two hot-path methods and makes the
    two consumers of their side outputs (``log`` and ``compute_depth_losses``, SURVEY.md 3.3) materialise
    what they read.

        class FusedTrainer(FusedLossMixin, Trainer): pass
        FusedTrainer(opts).train()

    ``self.opt`` must be the reference options namespace.  The training call itself produces no side outputs.
    ``Trainer.run_epoch`` decides to log only *after* ``process_batch`` (trainer.py:213-227), so the side outputs
    are produced on demand: when ``log`` / ``compute_depth_losses`` (also reached through ``val``) find
    ``outputs[("depth", 0, 0)]``, ``outputs[("color", f, 0)]`` or ``outputs["identity_selection/s"]`` missing,
    one extra forward-only fused call (same inputs, same tie-break noise as the training call) fills them in.
    Setting ``self.md2_side`` (e.g. ``{"depth_scales": [0], "color_scales": [0], "mask_scales": [0, 1, 2, 3]}``)
    makes every call produce them eagerly instead.
    """

    md2_side: Optional[dict] = None
    _md2_plan: Optional[LossPlan] = None

    def generate_images_pred(self, inputs, outputs):
        if self._md2_plan is None:
            self._md2_plan = LossPlan.from_opt(self.opt)
        plan = self._md2_plan
        side = dict(self.md2_side) if self.md2_side else None
        noise = None
        if plan.n_id > 0 and not plan.v1_multiscale:
            # drawn here exactly as view_synthesis_loss would (one torch.randn per scale, in scale order,
            # trainer.py:468-469) and kept so that a later on-demand side-output call sees the same masks
            shape = (plan.batch_size, plan.n_id, plan.height, plan.width)
            noise = _in_slot_order(plan, [torch.randn(shape, device=inputs[("color", 0, 0)].device) for _ in plan.scales])
            outputs["_md2_noise"] = noise
        outputs["_md2_losses"] = view_synthesis_loss(plan, inputs, outputs, noise=noise, side=side)

    def compute_losses(self, inputs, outputs):
        return outputs.pop("_md2_losses")

    def _md2_materialise(self, inputs, outputs, depth=False, color=False, masks=False):
        """Fill in the side outputs ``log`` / ``compute_depth_losses`` read, if the training call did not."""
        plan = self._md2_plan
        if plan is None:
            return
        scales = list(plan.scales)
        side = {}
        if depth and ("depth", 0, 0) not in outputs:
            side["depth_scales"] = [0]
        if color and any(("color", f, 0) not in outputs for f in plan.src_ids):
            side["color_scales"] = [0]
        if masks and plan.automask and any("identity_selection/{}".format(s) not in outputs for s in scales):
            side["mask_scales"] = scales
        if not side:
            return
        with torch.no_grad():
            outs = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in outputs.items()
                    if not (isinstance(k, str) and k.startswith("_md2"))}
            view_synthesis_loss(plan, inputs, outs, noise=outputs.get("_md2_noise"), side=side)
        for k, v in outs.items():
            if k not in outputs:
                outputs[k] = v

    def compute_depth_losses(self, inputs, outputs, losses):
        """trainer.py:498-526 through md2_depth_metrics (one fused call, SURVEY.md 8f-5); same keys, same value
        type (numpy scalars, trainer.py:526).  Set ``md2_fused_metrics = False`` to run the reference's own code."""
        self._md2_materialise(inputs, outputs, depth=True)
        if not getattr(self, "md2_fused_metrics", True):
            return super().compute_depth_losses(inputs, outputs, losses)
        import numpy as np
        from . import layers as L
        vals = L.depth_metrics(outputs[("depth", 0, 0)], inputs["depth_gt"]).cpu()
        for i, metric in enumerate(getattr(self, "depth_metric_names", L.DEPTH_METRIC_NAMES)):
            losses[metric] = np.array(vals[i])

    def log(self, mode, inputs, outputs, losses):
        self._md2_materialise(inputs, outputs, color=True, masks=True)
        return super().log(mode, inputs, outputs, losses)
