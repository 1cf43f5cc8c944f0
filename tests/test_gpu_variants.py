"""--pose_model_type posecnn (trainer.py:366-375) and --predictive_mask (trainer.py:447-459) as variants of the fused
kernels (md2_problem.posecnn / .predictive_mask), alone, together, with --avg_reprojection / --no_ssim / a stereo source
and under --v1_multiscale, against the live oracle on seeded inputs larger than the committed golden fixtures.
Loss parity 1e-5 (north_star); aggregated gradients no worse than 1.5 x the reference's own fp32-vs-fp64 noise on the
same case plus the weight of a few discrete-decision flips (protocol P3, SURVEY.md 8c), several of them sharp."""
import pytest
import torch

from helpers import rel_l2
from oracle import view_synthesis as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

CASES = [
    # name, B, H, W, frame_ids, flags
    ("posecnn", 3, 96, 160, [0, -1, 1], dict(posecnn=True)),
    ("posecnn_noauto_avg", 2, 64, 96, [0, -1, 1], dict(posecnn=True, disable_automasking=True, avg_reprojection=True)),
    ("posecnn_one_source", 2, 64, 96, [0, 1], dict(posecnn=True)),
    ("posecnn_v1", 2, 64, 96, [0, -1, 1], dict(posecnn=True, v1_multiscale=True)),
    ("pmask", 3, 96, 160, [0, -1, 1], dict(predictive_mask=True, disable_automasking=True)),
    ("pmask_avg", 2, 64, 96, [0, -1, 1], dict(predictive_mask=True, disable_automasking=True, avg_reprojection=True)),
    ("pmask_l1", 2, 64, 96, [0, -1, 1], dict(predictive_mask=True, disable_automasking=True, no_ssim=True)),
    ("pmask_stereo3", 2, 64, 96, [0, -1, 1, "s"], dict(predictive_mask=True, disable_automasking=True)),
    ("pmask_one_source", 2, 64, 96, [0, "s"], dict(predictive_mask=True, disable_automasking=True)),
    ("pmask_v1", 2, 64, 96, [0, -1, 1], dict(predictive_mask=True, disable_automasking=True, v1_multiscale=True)),
    ("pmask_posecnn", 2, 64, 96, [0, -1, 1], dict(predictive_mask=True, disable_automasking=True, posecnn=True)),
    # four sources with pose leaves and masks: 4 disparities + 4 x (axisangle, translation) + 4 masks = 16 autograd
    # leaves, the most md2_scale_tensors takes in its one launch
    ("pmask_posecnn_4src", 2, 64, 96, [0, -2, -1, 1, 2], dict(predictive_mask=True, disable_automasking=True,
                                                              posecnn=True)),
]


def _leaves(B, H, W, fids, flags, seed, dtype):
    from monodepth2_b200.synthetic import make_batch
    v1 = flags.get("v1_multiscale", False)
    inputs, outputs, pose, noise = make_batch(B, H, W, fids, 4, seed, "structured", all_scale_K=v1, multiscale_noise=v1)
    g = torch.Generator().manual_seed(seed + 1)
    outs = {k: v.to(dtype).clone().requires_grad_(True) for k, v in outputs.items() if k[0] == "disp"}
    leaves = dict(outs)
    for f in fids[1:]:
        if f == "s":
            continue
        aa, tr = pose[f]
        # what PoseDecoder emits (pose_decoder.py:49-54): (B, 2, 1, 3), only [:, 0] is used
        a4 = torch.zeros(B, 2, 1, 3, dtype=dtype)
        t4 = torch.zeros(B, 2, 1, 3, dtype=dtype)
        a4[:, 0, 0] = aa.reshape(B, 3).to(dtype)
        t4[:, 0, 0] = tr.reshape(B, 3).to(dtype)
        a4.requires_grad_(True); t4.requires_grad_(True)
        outs[("axisangle", 0, f)], outs[("translation", 0, f)] = a4, t4
        leaves[("axisangle", f)], leaves[("translation", f)] = a4, t4
    if flags.get("predictive_mask"):
        outs["predictive_mask"] = {}
        for s in range(4):
            m = (0.05 + 0.9 * torch.rand(B, len(fids) - 1, H >> s, W >> s, generator=g)).to(dtype).requires_grad_(True)
            outs["predictive_mask"][("disp", s)] = m
            leaves[("mask", s)] = m
    return inputs, outs, leaves, noise


def _oracle(B, H, W, fids, flags, seed, dtype):
    inputs, outs, leaves, noise = _leaves(B, H, W, fids, flags, seed, dtype)
    cfg = O.OracleConfig(height=H, width=W, frame_ids=tuple(fids), **flags)
    for f in fids[1:]:
        if f != "s":   # predict_poses (trainer.py:294-295)
            outs[("cam_T_cam", 0, f)] = O.transformation_from_parameters(
                outs[("axisangle", 0, f)][:, 0], outs[("translation", 0, f)][:, 0], invert=(f < 0))
    n_id = 0 if flags.get("disable_automasking") else (1 if flags.get("avg_reprojection") else len(fids) - 1)
    nz = [n[:, :n_id].to(dtype) for n in noise] if n_id else None
    losses = O.view_synthesis_loss({k: v.to(dtype) for k, v in inputs.items()}, outs, cfg, nz)
    losses["loss"].backward()
    return losses, leaves, nz


@pytest.mark.parametrize("name,B,H,W,fids,flags", CASES, ids=[c[0] for c in CASES])
def test_kernel_variant_matches_oracle(name, B, H, W, fids, flags):
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    seed = 300 + len(name)
    o_losses, o_leaves, nz = _oracle(B, H, W, fids, flags, seed, torch.float32)
    d_losses, d_leaves, _ = _oracle(B, H, W, fids, flags, seed, torch.float64)

    inputs, outs, leaves, _ = _leaves(B, H, W, fids, flags, seed, torch.float32)
    plan = LossPlan(B, H, W, fids, **flags)

    def dev(v):
        return v.detach().to(DEV).requires_grad_(True)
    c_leaves = {k: dev(v) for k, v in leaves.items()}
    c_outs = {k: c_leaves[k] for k in leaves if k[0] == "disp"}
    for f in fids[1:]:
        if f != "s":
            c_outs[("axisangle", 0, f)], c_outs[("translation", 0, f)] = c_leaves[("axisangle", f)], c_leaves[("translation", f)]
    if flags.get("predictive_mask"):
        c_outs["predictive_mask"] = {("disp", s): c_leaves[("mask", s)] for s in range(4)}
    losses = view_synthesis_loss(plan, {k: v.to(DEV) for k, v in inputs.items()}, c_outs,
                                 [n.to(DEV) for n in nz] if nz else None)
    losses["loss"].backward()
    torch.cuda.synchronize()

    for key in ["loss"] + ["loss/%d" % s for s in range(4)]:
        ref = float(o_losses[key].detach())
        assert abs(float(losses[key].detach()) - ref) <= 1e-5 * abs(ref), (key, float(losses[key].detach()), ref)
    # Gradients are flip-limited (SURVEY.md 7.3-1): on a case this small a single bilinear-cell / argmin flip moves an
    # aggregated gradient by ~1e-2 in relative L2 - for the kernel and for the reference's own fp32 run alike, and not
    # in the same leaves (measured: every leaf sits either at ~2e-5..5e-4 or at ~1e-2, scripts/variant_probe.py).  So:
    # every leaf within 1.5 x the reference's own noise plus a few flips, AND several leaves sharp - among them a
    # disparity and (where the variant has them) a pose leaf and every mask: a wrong term in the new code paths (the
    # mean-inverse-depth constant, the translation rescale, the mask weights) would leave no leaf of its kind sharp.
    errs, noise = {}, {}
    for k, leaf in c_leaves.items():
        assert leaf.grad is not None and torch.isfinite(leaf.grad).all(), k
        truth = d_leaves[k].grad
        ref_noise = rel_l2(o_leaves[k].grad, truth)
        errs[k] = rel_l2(leaf.grad.cpu(), truth)
        noise[k] = ref_noise
        # (masks: one flipped bilinear cell moves a mask leaf of this size by ~2e-3 - the reference's own fp32 run shows
        # exactly that on ("mask", 2): scripts/variant_leaf_probe.py - so the cap allows a couple of flips and the sharpness
        # requirement below does the real work)
        bound = (5e-3 + 1.5 * ref_noise) if k[0] == "mask" else 1.5 * ref_noise + 5e-2
        assert errs[k] <= bound, (k, errs[k], ref_noise, bound)
    masks = [k for k in errs if k[0] == "mask"]
    if masks:
        assert sum(1 for k in masks if errs[k] < 1e-4) >= 2, errs          # flip-free mask leaves are exact to rounding
    # sharp: flip-free, or sitting on the reference's own fp32 result - flips included (scripts/variant_leaf_probe.py:
    # with the up-sampling blend spelled out as the reference's kernel contracts it, posecnn_one_source reproduces the
    # one flip of the reference's fp32 run, and its two pose leaves then carry exactly the reference's 5.6e-3 / 3.4e-3)
    sharp = [k for k, e in errs.items() if e < 2e-3 or e <= 1.05 * noise[k] + 1e-5]
    assert len(sharp) >= 3 and any(k[0] == "disp" for k in sharp), errs
    if any(k[0] == "axisangle" for k in errs):
        assert any(k[0] in ("axisangle", "translation") for k in sharp), errs


def test_scaled_loss_scales_every_gradient_bitwise():
    """(w * loss).backward() hands w to the call's backward, which multiplies every stored gradient by it in one
    md2_scale_tensors launch: every leaf kind (disparity, axisangle, translation, mask) of the 16-leaf configuration
    gets exactly w x the plain gradient."""
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    name, B, H, W, fids, flags = next(c for c in CASES if c[0] == "pmask_posecnn_4src")
    inputs, _, leaves, _ = _leaves(B, H, W, fids, flags, 300 + len(name), torch.float32)
    c_leaves = {k: v.detach().to(DEV).requires_grad_(True) for k, v in leaves.items()}
    c_outs = {k: c_leaves[k] for k in leaves if k[0] == "disp"}
    for f in fids[1:]:
        c_outs[("axisangle", 0, f)], c_outs[("translation", 0, f)] = c_leaves[("axisangle", f)], c_leaves[("translation", f)]
    c_outs["predictive_mask"] = {("disp", s): c_leaves[("mask", s)] for s in range(4)}
    losses = view_synthesis_loss(LossPlan(B, H, W, fids, **flags), {k: v.to(DEV) for k, v in inputs.items()}, c_outs)
    keys = list(c_leaves)
    assert len(keys) == 16 and {k[0] for k in keys} == {"disp", "axisangle", "translation", "mask"}
    plain = torch.autograd.grad(losses["loss"], [c_leaves[k] for k in keys], retain_graph=True)
    w = torch.tensor(-0.7071067811865476, device=DEV)
    scaled = torch.autograd.grad(w * losses["loss"], [c_leaves[k] for k in keys])
    for k, a, b in zip(keys, plain, scaled):
        # bit patterns where the call wrote a gradient; the unused half of a PoseDecoder leaf is autograd's +0 fill
        # in both runs (w x +0 would be -0 for negative w, an equal value with another bit pattern)
        nz = a != 0
        assert bool(nz.any()), k
        assert torch.equal(b[nz].view(torch.int32), (a[nz] * w).view(torch.int32)), k
        assert bool((b[~nz] == 0).all()), k
