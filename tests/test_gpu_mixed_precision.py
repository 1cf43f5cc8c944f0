"""bfloat16 / float16 leaves of the fused loss and feature maps of the disparity head.

The rule under test: with reduced-precision operands every result equals the float32 entry point applied to the
operands widened exactly to float32; a result handed back in reduced precision is that float32 value rounded once
(nearest-even).  So each case rounds its leaves to the dtype, runs once with those leaves and once with their
.float(), and compares bit patterns.

The scalar sums of the fused call (losses, pose gradients, and under posecnn the mean-inverse-depth part of the
disparity gradient) go through fp64 atomics, whose order varies from run to run.  The float32 call is therefore run
twice: where its two runs agree bit for bit the reduced-precision run must match them exactly; where they do not,
it must lie within one unit in the last place of the compared dtype, the width of that run-to-run variation."""
from collections import OrderedDict

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from helpers import Golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
DT_IDS = ["bf16", "fp16"]
CASES = ["mono_iid", "stereo_iid", "avg_reprojection", "disable_automasking", "no_ssim", "posecnn", "predictive_mask",
         "scales_0_2", "v1_multiscale"]
_INT = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}


def _bits(t):
    return t.detach().contiguous().view(_INT[t.dtype]).to(torch.int64)


def _same(what, got, a, b, dtype=None):
    """``got`` == ``a`` rounded to ``dtype``, bit for bit when the two float32 runs ``a`` and ``b`` agree, else within one
    ulp of the compared dtype (a sign change between +-0 and the smallest subnormal counts as one step as well)."""
    ref = a.to(dtype) if dtype is not None else a
    assert got.dtype == ref.dtype and got.shape == ref.shape, (what, got.dtype, ref.dtype, got.shape, ref.shape)
    if torch.equal(_bits(a), _bits(b)):
        assert torch.equal(_bits(got), _bits(ref)), what
    else:
        near = (_bits(got) - _bits(ref)).abs() <= 1
        tiny = (_bits(got.abs()) <= 1) & (_bits(ref.abs()) <= 1)
        assert bool((near | tiny).all()), what


def _plan(g):
    from monodepth2_b200.fused_loss import LossPlan
    return LossPlan(g.B, g.H, g.W, g.frame_ids, avg_reprojection=g.avg_reprojection,
                    disable_automasking=g.disable_automasking, no_ssim=g.no_ssim, v1_multiscale=g.v1_multiscale,
                    posecnn=g.posecnn, predictive_mask=g.predictive_mask, scales=g.scales)


def _golden_leaves(g, pose_mode, rnd):
    """The fixture's leaves rounded to ``rnd`` (still in ``rnd``): disparities, masks, and per network source either
    cam_T_cam or the PoseDecoder-shaped (B,2,1,3) axisangle / translation pair."""
    lv = {("disp", s): g.t("disp__%d" % s).to(rnd) for s in g.scales}
    if g.predictive_mask:
        for s in g.scales:
            lv[("mask", s)] = g.t("mask__%d" % s).to(rnd)
    for f in g.frame_ids[1:]:
        if f == "s":
            continue
        if pose_mode == "cam_T_cam":
            lv[("cam_T_cam", f)] = g.t("cam_T_cam__%s" % f).to(rnd)
        else:
            for name in ("axisangle", "translation"):
                x = torch.zeros(g.B, 2, 1, 3, dtype=rnd)
                x[:, 0] = g.t("%s__%s" % (name, f)).reshape(g.B, 1, 3).to(rnd)
                lv[(name, f)] = x
    return lv


def _run_golden(g, plan, lv, dtype, scale=None):
    """One fused call + backward with the leaves ``lv`` cast to ``dtype``; returns losses, side outputs and grads."""
    from monodepth2_b200.fused_loss import view_synthesis_loss
    leaves = {k: v.to(DEV).to(dtype).requires_grad_(True) for k, v in lv.items()}
    outs = {}
    for k, v in leaves.items():
        if k[0] == "disp":
            outs[k] = v
        elif k[0] == "cam_T_cam":
            outs[("cam_T_cam", 0, k[1])] = v
        elif k[0] in ("axisangle", "translation"):
            outs[(k[0], 0, k[1])] = v
    if g.predictive_mask:
        outs["predictive_mask"] = {("disp", s): leaves[("mask", s)] for s in g.scales}
    inputs = {k: v.to(DEV) for k, v in g.inputs().items()}
    noise = [n.to(DEV) for n in g.noise()] if g.n_id > 0 else None
    side = {"depth_scales": list(g.scales), "color_scales": list(g.scales),
            "mask_scales": list(g.scales) if g.n_id > 0 else []}
    given = set(outs)
    losses = view_synthesis_loss(plan, inputs, outs, noise, side)
    (losses["loss"] if scale is None else scale * losses["loss"]).backward()
    torch.cuda.synchronize()
    # what the call produced: cam_T_cam built from pose leaves, depth, warped colours, identity selection
    extra = {k: v.detach() for k, v in outs.items()
             if k not in given and isinstance(k, tuple) and k[0] in ("cam_T_cam", "depth", "color")}
    extra.update({k: v for k, v in outs.items() if isinstance(k, str) and k.startswith("identity_selection/")})
    return ({k: v.detach() for k, v in losses.items()}, extra, {k: v.grad for k, v in leaves.items()})


@pytest.mark.parametrize("pose_mode", ["cam_T_cam", "pose_leaves"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("name", CASES)
def test_reduced_precision_leaves_equal_the_fp32_call_on_the_upcast_leaves(name, dtype, pose_mode):
    g = Golden(name)
    if g.posecnn and pose_mode == "cam_T_cam":
        pytest.skip("posecnn builds T per scale from the pose leaves; it takes no cam_T_cam")
    plan = _plan(g)
    lv = _golden_leaves(g, pose_mode, dtype)
    l32a, x32a, g32a = _run_golden(g, plan, lv, torch.float32)
    l32b, x32b, g32b = _run_golden(g, plan, lv, torch.float32)
    ln, xn, gn = _run_golden(g, plan, lv, dtype)
    for k in l32a:
        _same("losses[%s]" % k, ln[k], l32a[k], l32b[k])
        assert ln[k].dtype == torch.float32
    assert set(xn) == set(x32a) and len(xn) >= len(g.scales)
    for k in x32a:
        assert xn[k].dtype == torch.float32, k
        _same(str(k), xn[k], x32a[k], x32b[k])
    if pose_mode == "pose_leaves" and not g.v1_multiscale:     # (the per-level calls of v1 keep theirs)
        assert any(isinstance(k, tuple) and k[0] == "cam_T_cam" for k in xn)
    for k in g32a:
        assert gn[k] is not None and gn[k].dtype == dtype, k
        _same("grad %s" % (k,), gn[k], g32a[k], g32b[k], dtype)


@pytest.mark.parametrize("pose_mode", ["cam_T_cam", "pose_leaves"])
def test_scaled_fp16_backward_rounds_after_the_scale(pose_mode):
    """GradScaler's pattern, (65536 * loss).backward(): the fp16 gradient is (65536 * g32) rounded once, including
    elements whose unscaled value underflows fp16; a scale that overflows fp16 gives +-inf, never a saturated value."""
    g = Golden("mono_iid")
    plan = _plan(g)
    lv = _golden_leaves(g, pose_mode, torch.float16)
    _, _, g32a = _run_golden(g, plan, lv, torch.float32)
    _, _, g32b = _run_golden(g, plan, lv, torch.float32)
    underflow_rescued = False
    for scale in (65536.0, 2.0 ** 40):
        _, _, gn = _run_golden(g, plan, lv, torch.float16, scale=scale)
        any_inf = False
        for k in g32a:
            # scale is a power of two: scale * g32 is exact in float32, so the comparison is the unscaled one's
            _same("grad %s x %g" % (k, scale), gn[k], scale * g32a[k], scale * g32b[k], torch.float16)
            any_inf |= bool(torch.isinf(gn[k]).any())
            if scale == 65536.0:
                underflow_rescued |= bool(((g32a[k].half() == 0) & (g32a[k] != 0) & (gn[k] != 0)).any())
        if scale == 2.0 ** 40:
            assert any_inf
    assert underflow_rescued


def _stand_in(B, H, W, fids, seed):
    from benchmarks.train_step import Nets
    from monodepth2_b200.synthetic import make_batch
    torch.manual_seed(seed)
    nets = Nets(fids, 18).to(DEV)
    inputs, _, _, _ = make_batch(B, H, W, fids, 4, seed, "structured")
    return nets, {k: v.to(DEV) for k, v in inputs.items()}


@pytest.mark.parametrize("pose_mode", ["pose_leaves", "cam_T_cam"])
def test_autocast_bf16_training_step_gives_finite_fp32_gradients(pose_mode):
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from oracle import view_synthesis as O
    B, H, W, fids = 2, 64, 96, [0, -1, 1]
    nets, inputs = _stand_in(B, H, W, fids, 5)
    plan = LossPlan(B, H, W, fids)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        outputs = nets({f: inputs[("color", f, 0)] for f in fids})
        assert outputs[("disp", 0)].dtype == torch.bfloat16
        assert outputs[("axisangle", 0, -1)].dtype == torch.bfloat16
        if pose_mode == "cam_T_cam":        # predict_poses as the reference runs it under autocast (trainer.py:294-295)
            for f in fids[1:]:
                outputs[("cam_T_cam", 0, f)] = O.transformation_from_parameters(
                    outputs[("axisangle", 0, f)][:, 0], outputs[("translation", 0, f)][:, 0], invert=(f < 0))
                assert outputs[("cam_T_cam", 0, f)].dtype == torch.bfloat16
        losses = view_synthesis_loss(plan, inputs, outputs)
    assert losses["loss"].dtype == torch.float32 and bool(torch.isfinite(losses["loss"]))
    losses["loss"].backward()
    for n, p in nets.named_parameters():
        assert p.grad is not None and p.grad.dtype == torch.float32, n
        assert bool(torch.isfinite(p.grad).all()), n
    assert float(nets.depth.heads["0"][1].weight.grad.abs().sum()) > 0
    assert float(nets.pose.c2.weight.grad.abs().sum()) > 0


def test_autocast_fp16_gradscaler_step_is_not_skipped():
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    B, H, W, fids = 2, 64, 96, [0, -1, 1]
    nets, inputs = _stand_in(B, H, W, fids, 6)
    plan = LossPlan(B, H, W, fids)
    opt = torch.optim.Adam(nets.parameters(), 1e-4)
    # The pose leaves' gradients are sums over every pixel, of order 1: times the default initial scale of 65536 they
    # overflow fp16 on the first step (to inf, and GradScaler backs off as designed).  2^10 keeps them finite, while
    # the per-pixel disparity gradients (~1e-6 here) would still underflow fp16 without the scale.
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 10)
    before = {n: p.detach().clone() for n, p in nets.named_parameters()}
    with torch.autocast("cuda", dtype=torch.float16):
        outputs = nets({f: inputs[("color", f, 0)] for f in fids})
        assert outputs[("disp", 0)].dtype == torch.float16
        losses = view_synthesis_loss(plan, inputs, outputs)
    scale0 = scaler.get_scale()
    scaler.scale(losses["loss"]).backward()
    scaler.step(opt)
    scaler.update()
    assert scaler.get_scale() == scale0           # a found inf would have halved the scale and skipped the step
    assert any(not torch.equal(before[n], p.detach()) for n, p in nets.named_parameters())


def test_graphed_loss_with_bf16_leaves_replays_the_eager_call():
    """--disable_automasking: no tie-break noise, so replay and eager call compute on the same values."""
    from monodepth2_b200.fused_loss import GraphedLoss, LossPlan, view_synthesis_loss
    from monodepth2_b200.synthetic import make_batch
    B, H, W, fids = 2, 64, 96, [0, -1, 1]
    plan = LossPlan(B, H, W, fids, disable_automasking=True)
    inputs, outputs, pose, _ = make_batch(B, H, W, fids, 4, 73, "structured")
    ins = {k: v.to(DEV) for k, v in inputs.items() if k in [("color", f, 0) for f in fids]
           + [("color", 0, s) for s in range(1, 4)] + [("K", 0), ("inv_K", 0)]}
    leaves = {("disp", s): outputs[("disp", s)].to(DEV, torch.bfloat16) for s in range(4)}
    for f in fids[1:]:
        for i, name in enumerate(("axisangle", "translation")):
            x = torch.zeros(B, 2, 1, 3, device=DEV, dtype=torch.bfloat16)
            x[:, 0, 0] = pose[f][i].to(DEV, torch.bfloat16)
            leaves[(name, 0, f)] = x
    gl = GraphedLoss(plan, ins, leaves)
    gl.load(ins, leaves)
    loss = gl.run().clone()
    torch.cuda.synchronize()
    for k, v in gl.grads.items():
        assert v is not None and v.dtype == torch.bfloat16, k
    runs = []
    for _ in range(2):
        outs = {k: v.clone().requires_grad_(True) for k, v in leaves.items()}
        ref = view_synthesis_loss(plan, ins, outs)
        ref["loss"].backward()
        runs.append((ref["loss"].detach(), {k: v.grad for k, v in outs.items()}))
    torch.cuda.synchronize()
    _same("loss", loss, runs[0][0], runs[1][0])
    for k in leaves:
        _same("grad %s" % (k,), gl.grads[k], runs[0][1][k], runs[1][1][k])


def test_reduced_precision_refusals():
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from monodepth2_b200.synthetic import make_batch
    B, H, W, fids = 2, 32, 48, [0, -1, 1]
    plan = LossPlan(B, H, W, fids)
    inputs, outputs, _, _ = make_batch(B, H, W, fids, 4, 9, "structured")
    ins = {k: v.to(DEV) for k, v in inputs.items()}
    outs = {k: v.to(DEV) for k, v in outputs.items()}

    def but(d, key, value):
        d = dict(d)
        d[key] = value
        return d
    with pytest.raises(RuntimeError, match=r"disp\[0\].*float64"):
        view_synthesis_loss(plan, ins, but(outs, ("disp", 0), outs[("disp", 0)].double()))
    with pytest.raises(RuntimeError, match=r"disp\[0\] torch.float32, disp\[1\] torch.bfloat16"):
        view_synthesis_loss(plan, ins, but(outs, ("disp", 1), outs[("disp", 1)].bfloat16()))
    with pytest.raises(RuntimeError, match=r"T\[0\].*float64"):
        view_synthesis_loss(plan, ins, but(outs, ("cam_T_cam", 0, -1), outs[("cam_T_cam", 0, -1)].double()))
    with pytest.raises(RuntimeError, match="target must be float32"):
        view_synthesis_loss(plan, but(ins, ("color", 0, 0), ins[("color", 0, 0)].bfloat16()), outs)
    from monodepth2_b200 import layers as L
    head = L.DispConvSigmoid(4).to(DEV)
    with pytest.raises(RuntimeError, match="float64"):
        head(torch.zeros(1, 4, 8, 8, device=DEV, dtype=torch.float64))


# ------------------------------------------------------------------ disparity head on bf16 / fp16 feature maps
HEAD_SHAPES = {16: (2, 96, 160), 32: (2, 48, 80), 64: (2, 24, 40), 128: (2, 12, 20)}
F32_ULP = 2.0 ** -23


def _fp32_head_backward(g32, d32, x32, w):
    """md2_dispconv_sigmoid_backward (the float32 kernels) on float32 operands."""
    import ctypes as C
    from monodepth2_b200 import layers as L
    B, Cc, H, W = x32.shape
    gx, gw, gb = torch.empty_like(x32), torch.empty_like(w), torch.empty(1, device=DEV)
    L._call("md2_dispconv_sigmoid_backward", x32.device, L._p(g32), L._p(d32), L._p(x32), L._p(w), L._p(gx), L._p(gw),
            L._p(gb), C.c_int(B), C.c_int(Cc), C.c_int(H), C.c_int(W), L._stream(x32))
    return gx


def _weight_grad_ref(gd, d, x, dtype):
    """grad_weight, grad_bias of conv(pad(x)) with the pre-activation gradient gd * d * (1 - d), in ``dtype`` on the
    CPU, from the widened operands the kernel reads."""
    gd, d, x = (t.detach().cpu().to(dtype) for t in (gd, d, x))
    gpre = gd * d * (1 - d)
    xp = F.pad(x, (1, 1, 1, 1), mode="reflect")
    gw = torch.nn.grad.conv2d_weight(xp, (1, x.shape[1], 3, 3), gpre)
    return gw, gpre.sum().reshape(1)


@pytest.mark.parametrize("shape", ["typical", "h2w3", "h3w2"])
@pytest.mark.parametrize("Cc", [16, 32, 64, 128])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_disparity_head_on_reduced_precision_maps(dtype, Cc, shape):
    from monodepth2_b200 import layers as L
    B, H, W = {"typical": HEAD_SHAPES[Cc], "h2w3": (2, 2, 3), "h3w2": (3, 3, 2)}[shape]
    gen = torch.Generator().manual_seed(Cc * 7 + H)
    x = torch.randn(B, Cc, H, W, generator=gen).to(DEV, dtype)
    up = torch.randn(B, 1, H, W, generator=gen).to(DEV, dtype)
    head = L.DispConvSigmoid(Cc).to(DEV)
    xd = x.clone().requires_grad_(True)
    y = head(xd)
    assert y.dtype == dtype
    y.backward(up)
    assert xd.grad.dtype == dtype and head.conv.weight.grad.dtype == torch.float32
    w, b = head.conv.weight.detach(), head.conv.bias.detach()
    with torch.no_grad():
        y32 = L._DispHead.apply(x.float(), w, b)
    assert torch.equal(_bits(y), _bits(y32.to(dtype)))
    gx32 = _fp32_head_backward(up.float(), y.float(), x.float(), w)
    assert torch.equal(_bits(xd.grad), _bits(gx32.to(dtype)))
    # weight / bias gradients: float32 atomics, against float64 within the bound of the float32 head's edge tests
    r32w, r32b = _weight_grad_ref(up, y, x, torch.float32)
    r64w, r64b = _weight_grad_ref(up, y, x, torch.float64)
    for got, r32, r64 in ((head.conv.weight.grad, r32w, r64w), (head.conv.bias.grad, r32b, r64b)):
        got, r32 = got.cpu().double(), r32.double()
        bound = 1.5 * (r32 - r64).abs() + 32 * F32_ULP * r64.abs() + 1e-5 * float(r64.abs().max())
        assert bool(((got - r64).abs() <= bound).all()), (float((got - r64).abs().max()), float(bound.min()))


def test_fused_heads_under_autocast_feed_the_fused_loss():
    from monodepth2_b200 import layers as L
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from monodepth2_b200.synthetic import make_batch

    class Dec(nn.Module):       # laid out like networks/depth_decoder.py:17-65: convs dict + ModuleList + sigmoid
        def __init__(self):
            super().__init__()
            self.convs = OrderedDict()
            self.convs[("upconv", 0, 0)] = L.ConvBlock(3, 16)
            for s in range(4):
                self.convs[("dispconv", s)] = L.Conv3x3(16, 1)
            self.decoder = nn.ModuleList(list(self.convs.values()))
            self.sigmoid = nn.Sigmoid()

        def forward(self, x):
            x = self.convs[("upconv", 0, 0)](x)
            return {("disp", s): self.sigmoid(self.convs[("dispconv", s)](F.avg_pool2d(x, 2 ** s) if s else x))
                    for s in range(4)}

    B, H, W, fids = 2, 64, 96, [0, -1, 1]
    torch.manual_seed(1)
    dec = L.fuse_disp_heads(Dec().to(DEV))
    inputs, outputs, _, _ = make_batch(B, H, W, fids, 4, 11, "structured")
    ins = {k: v.to(DEV) for k, v in inputs.items()}
    with torch.autocast("cuda", dtype=torch.bfloat16):
        outs = dec(ins[("color", 0, 0)])
        for f in fids[1:]:
            outs[("cam_T_cam", 0, f)] = outputs[("cam_T_cam", 0, f)].to(DEV)
        assert all(outs[("disp", s)].dtype == torch.bfloat16 for s in range(4))
        losses = view_synthesis_loss(LossPlan(B, H, W, fids), ins, outs)
    losses["loss"].backward()
    assert bool(torch.isfinite(losses["loss"]))
    for n, p in dec.named_parameters():
        assert p.grad is not None and p.grad.dtype == torch.float32 and bool(torch.isfinite(p.grad).all()), n
