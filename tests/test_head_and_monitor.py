"""The two components either side of the loss path that SURVEY.md 8f ranks next:
8f-4  the disparity head of DepthDecoder, sigmoid(Conv3x3(C -> 1)(x))  (networks/depth_decoder.py:60-63,
      layers.py:119-136) as one fused forward pass + a two-pass backward, against torch's own conv / pad / sigmoid;
8f-5  Trainer.compute_depth_losses (trainer.py:498-526, layers.py:251-269) as a fused metrics call, against the
      oracle restatement, which is pinned against the reference's own method on stored values
      (tests/golden/reference_interface.json, recorded by tests/golden/make_reference_interface.py)."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from helpers import GOLDEN_DIR
from oracle import view_synthesis as O


def test_oracle_depth_metrics_equal_the_reference_method():
    """Trainer.compute_depth_losses of the reference on these seeded inputs, as make_reference_interface.py stores it."""
    with open(os.path.join(GOLDEN_DIR, "reference_interface.json")) as f:
        losses = json.load(f)["depth_metrics"]
    g = torch.Generator().manual_seed(0)
    depth = torch.rand(3, 1, 48, 160, generator=g) * 40 + 0.5
    gt = torch.rand(3, 1, 375, 1242, generator=g) * 60
    gt[torch.rand(gt.shape, generator=g) < 0.7] = 0            # sparse LiDAR ground truth
    mine = O.depth_metrics(depth, gt)
    for i, k in enumerate(["de/abs_rel", "de/sq_rel", "de/rms", "de/log_rms", "da/a1", "da/a2", "da/a3"]):
        assert abs(float(mine[i]) - float(losses[k])) <= 1e-6 * abs(float(losses[k])), k


KITTI_GT, EIGEN_CROP = (375, 1242), (153, 371, 44, 1197)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,sparsity,seed,gt_hw,crop", [
    pytest.param((2, 48, 160), 0.7, 1, KITTI_GT, EIGEN_CROP, id="shape0-0.7-1"),
    pytest.param((3, 192, 640), 0.95, 2, KITTI_GT, EIGEN_CROP, id="shape1-0.95-2"),
    pytest.param((1, 24, 80), 0.0, 3, KITTI_GT, EIGEN_CROP, id="shape2-0.0-3"),
    pytest.param((4, 96, 320), 0.5, 4, KITTI_GT, EIGEN_CROP, id="shape3-0.5-4"),
    # gt smaller than the prediction (bilinear down-sampling), gt of odd size, crops reaching past the gt
    pytest.param((2, 96, 320), 0.3, 5, (48, 160), (10, 40, 20, 150), id="gt_below_pred"),
    pytest.param((2, 48, 160), 0.5, 6, (37, 123), (20, 375, 50, 1242), id="crop_past_gt"),
    pytest.param((1, 24, 80), 0.0, 7, (24, 80), (0, 24, 0, 80), id="same_size_full_crop"),
    pytest.param((3, 12, 40), 0.9, 8, (1, 1242), (0, 1, 44, 1197), id="one_gt_row")])
def test_cuda_depth_metrics_match_oracle(shape, sparsity, seed, gt_hw, crop):
    from monodepth2_b200 import layers as L
    B, H, W = shape
    g = torch.Generator().manual_seed(seed)
    depth = torch.rand(B, 1, H, W, generator=g) * 60 + 0.05
    gt = torch.rand(B, 1, *gt_hw, generator=g) * 70 + 0.5
    gt[torch.rand(gt.shape, generator=g) < sparsity] = 0
    ref = O.depth_metrics(depth, gt, crop)
    got = L.depth_metrics(depth.cuda(), gt.cuda(), crop).cpu()
    for i, k in enumerate(L.DEPTH_METRIC_NAMES):
        assert abs(float(got[i]) - float(ref[i])) <= 2e-5 * abs(float(ref[i])) + 1e-7, (k, float(got[i]), float(ref[i]))


class _RefConv3x3(nn.Module):          # layers.py:119-136, restated for the comparison
    def __init__(self, cin, cout):
        super().__init__()
        self.pad = nn.ReflectionPad2d(1)
        self.conv = nn.Conv2d(cin, cout, 3)

    def forward(self, x):
        return self.conv(self.pad(x))


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,H,W", [(2, 16, 48, 80), (3, 32, 24, 40), (1, 64, 12, 20), (2, 128, 6, 10), (1, 16, 5, 7), (12, 16, 192, 640),
                                     (2, 1, 3, 3), (1, 3, 2, 5), (2, 17, 3, 2), (1, 17, 7, 3), (3, 1, 2, 2)])
def test_cuda_disparity_head_matches_torch(B, C, H, W):
    from monodepth2_b200 import layers as L
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(C + H)
    ref = _RefConv3x3(C, 1).cuda()
    head = L.DispConvSigmoid(C).cuda()
    head.load_state_dict(ref.state_dict())               # same parameter names: conv.weight / conv.bias
    x = torch.randn(B, C, H, W, device="cuda")
    x0 = x.clone().requires_grad_(True)
    x1 = x.clone().requires_grad_(True)
    y0 = torch.sigmoid(ref(x0))                          # depth_decoder.py:62-63
    y1 = head(x1)
    assert torch.allclose(y0, y1, rtol=1e-5, atol=1e-6)
    up = torch.randn_like(y0)
    y0.backward(up)
    y1.backward(up)
    scale = float(x0.grad.abs().max())
    assert float((x0.grad - x1.grad).abs().max()) <= 2e-5 * scale + 1e-7
    for a, b in ((ref.conv.weight.grad, head.conv.weight.grad), (ref.conv.bias.grad, head.conv.bias.grad)):
        assert float((a - b).abs().max()) <= 1e-4 * float(a.abs().max()) + 1e-6


@pytest.mark.gpu
def test_fuse_disp_heads_keeps_the_decoder_interface():
    """A decoder laid out like networks/depth_decoder.py:17-65 (convs dict + ModuleList + sigmoid): after
    fuse_disp_heads its forward returns the same disparities, its state_dict keys are unchanged and the parameters
    are the same objects (an optimiser built before the swap keeps working)."""
    from collections import OrderedDict
    from monodepth2_b200 import layers as L

    class Dec(nn.Module):
        def __init__(self):
            super().__init__()
            self.convs = OrderedDict()
            self.convs[("upconv", 0, 0)] = L.ConvBlock(8, 16)
            for s in range(2):
                self.convs[("dispconv", s)] = L.Conv3x3(16, 1)
            self.decoder = nn.ModuleList(list(self.convs.values()))
            self.sigmoid = nn.Sigmoid()

        def forward(self, x):
            x = self.convs[("upconv", 0, 0)](x)
            return {("disp", s): self.sigmoid(self.convs[("dispconv", s)](x)) for s in range(2)}
    torch.manual_seed(0)
    dec = Dec().cuda()
    keys = list(dec.state_dict().keys())
    params = [id(p) for p in dec.parameters()]
    x = torch.randn(2, 8, 16, 24, device="cuda")
    before = {k: v.detach().clone() for k, v in dec(x).items()}
    L.fuse_disp_heads(dec)
    after = dec(x)
    assert list(dec.state_dict().keys()) == keys and [id(p) for p in dec.parameters()] == params
    for k in before:
        assert torch.allclose(before[k], after[k], rtol=1e-5, atol=1e-6)
    sum(v.sum() for v in after.values()).backward()
    assert all(p.grad is not None for p in dec.parameters())
