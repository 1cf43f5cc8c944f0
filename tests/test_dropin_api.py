"""The drop-in boundary against the reference's own definitions (CPU): same public names in layers.py, same
constructor / call signatures, the two Trainer methods the mixin overrides, and LossPlan.from_opt on the options the
reference's parser produces for each flag set - as stored in tests/golden/reference_interface.json, which
tests/golden/make_reference_interface.py records from the reference.  The run_epoch test drives the reference's own
Trainer and runs where MD2_REFERENCE_DIR names a checkout of the reference."""
import copy
import inspect
import json
import os
import sys
import types

import pytest

from helpers import GOLDEN_DIR

REF = os.environ.get("MD2_REFERENCE_DIR", "")
with open(os.path.join(GOLDEN_DIR, "reference_interface.json")) as f:
    GOLD = json.load(f)


@pytest.fixture(scope="module")
def ref():
    if not os.path.isdir(REF):
        pytest.skip("MD2_REFERENCE_DIR does not name a checkout of the reference")
    for name, attrs in (("tensorboardX", {"SummaryWriter": object}), ("IPython", {"embed": lambda *a, **k: None}),
                        ("skimage", {}), ("skimage.transform", {})):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules.setdefault(name, m)
    sys.modules["skimage"].transform = sys.modules["skimage.transform"]
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF)
    try:
        import layers as ref_layers
        import trainer as ref_trainer
        from options import MonodepthOptions
    finally:
        sys.path.remove(REF)
    return types.SimpleNamespace(layers=ref_layers, trainer=ref_trainer, Options=MonodepthOptions)


def _params(fn):
    return [p.name for p in inspect.signature(fn).parameters.values()]


def _reference_options(flags):
    """The namespace the reference's MonodepthOptions().parse() returns for `train.py <flags>` (the fields the loss
    path reads)."""
    return types.SimpleNamespace(**copy.deepcopy(GOLD["options"][" ".join(flags)]))


def test_layers_exports_every_public_name_of_the_reference():
    from monodepth2_b200 import layers as L
    ref_public = GOLD["layers_public"]
    assert ref_public, "nothing found in the reference's layers.py"
    missing = [n for n in ref_public if not hasattr(L, n)]
    assert missing == []
    assert set(ref_public) <= set(L.__all__) | {"grid_sample_border"}


@pytest.mark.parametrize("name", ["BackprojectDepth", "Project3D", "SSIM", "ConvBlock", "Conv3x3"])
def test_module_signatures_match(name):
    from monodepth2_b200 import layers as L
    a, b = GOLD["modules"][name], getattr(L, name)
    assert a["__init__"] == _params(b.__init__), name
    assert a["forward"] == _params(b.forward), name


@pytest.mark.parametrize("name", ["disp_to_depth", "transformation_from_parameters", "get_translation_matrix",
                                  "rot_from_axisangle", "get_smooth_loss", "upsample", "compute_depth_errors"])
def test_function_signatures_match(name):
    from monodepth2_b200 import layers as L
    assert GOLD["functions"][name] == _params(getattr(L, name)), name


def test_mixin_overrides_exactly_the_two_hot_path_methods():
    from monodepth2_b200.fused_loss import FusedLossMixin
    for m in ("generate_images_pred", "compute_losses"):
        assert GOLD["trainer_methods"][m] == _params(getattr(FusedLossMixin, m)), m

    class T:                  # stand-in for the reference's Trainer: the methods the mixin leaves to it
        def process_batch(self, inputs):
            pass

        def predict_poses(self, inputs, features):
            pass

    class FusedTrainer(FusedLossMixin, T):
        pass
    assert FusedTrainer.generate_images_pred is FusedLossMixin.generate_images_pred
    assert FusedTrainer.compute_losses is FusedLossMixin.compute_losses
    assert FusedTrainer.process_batch is T.process_batch            # the caller stays the reference's
    assert FusedTrainer.predict_poses is T.predict_poses
    # the two consumers of the side outputs are wrapped (they materialise what they read, then delegate)
    for m in ("log", "compute_depth_losses"):
        assert GOLD["trainer_methods"][m] == _params(getattr(FusedLossMixin, m)), m
    overridden = [n for n, v in vars(FusedLossMixin).items() if callable(v) and not n.startswith("_")]
    assert sorted(overridden) == ["compute_depth_losses", "compute_losses", "generate_images_pred", "log"]


def test_reference_run_epoch_drives_the_mixin_through_logging_and_val(ref, monkeypatch):
    """ADVICE r1: the documented `FusedTrainer(opts).train()` must survive the first logging step.  The real
    Trainer.run_epoch (trainer.py:193-231) logs at batch_idx == 0 and calls val(); log() and
    compute_depth_losses() read outputs[("depth",0,0)], ("color",f,0) and "identity_selection/s".  No GPU here:
    the fused call is replaced by the CPU oracle behind the same signature, which only produces side outputs
    when `side` asks for them - exactly the contract of the CUDA call."""
    import torch
    from monodepth2_b200 import _capi, fused_loss
    from monodepth2_b200.fused_loss import FusedLossMixin
    from monodepth2_b200.synthetic import make_batch
    from oracle import view_synthesis as O
    if not os.path.exists(_capi.LIB_PATH):
        pytest.skip("libmd2loss.so not built")
    monkeypatch.setattr(sys, "argv", ["train.py", "--batch_size", "2", "--height", "32", "--width", "64",
                                      "--log_frequency", "1"])
    opt = ref.Options().parse()
    B, H, W, fids = opt.batch_size, opt.height, opt.width, opt.frame_ids
    calls = []

    def fake_fused(plan, inputs, outputs, noise=None, side=None):
        calls.append((torch.is_grad_enabled(), dict(side) if side else None))
        cfg = O.OracleConfig(height=plan.height, width=plan.width, frame_ids=tuple(plan.frame_ids))
        outs = dict(outputs)
        losses = O.view_synthesis_loss(dict(inputs), outs, cfg, noise)
        if side:
            want = [("depth", 0, s) for s in side.get("depth_scales", [])]
            want += [("color", f, s) for s in side.get("color_scales", []) for f in plan.src_ids]
            want += ["identity_selection/{}".format(s) for s in side.get("mask_scales", [])]
            for k in want:
                outputs[k] = outs[k].detach()
        return losses
    monkeypatch.setattr(fused_loss, "view_synthesis_loss", fake_fused)
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self, raising=False)

    class Enc(torch.nn.Module):
        def __init__(self, cin):
            super().__init__()
            self.c = torch.nn.Conv2d(cin, 4, 3, padding=1)

        def forward(self, x):
            return [self.c(x)]

    class Depth(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.c = torch.nn.Conv2d(4, 1, 3, padding=1)

        def forward(self, feats):
            d = torch.sigmoid(self.c(feats[0]))
            return {("disp", s): torch.nn.functional.avg_pool2d(d, 2 ** s) if s else d for s in range(4)}

    class Pose(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.l = torch.nn.Linear(4, 12)

        def forward(self, feats):
            o = 0.01 * self.l(feats[0][-1].mean((2, 3))).view(-1, 2, 1, 6)
            return o[..., :3], o[..., 3:]

    class Writer:
        def __init__(self):
            self.scalars, self.images = [], []

        def add_scalar(self, name, v, step):
            self.scalars.append(name)

        def add_image(self, name, img, step):
            self.images.append((name, tuple(img.shape)))

    class Loader(list):
        """val_iter.next() is how the reference pulls validation batches (trainer.py:325)"""
        def __iter__(self):
            it = super().__iter__()

            class It:
                def __iter__(s):
                    return s

                def __next__(s):
                    return next(it)
                next = __next__
            return It()

    def batch(seed):
        inputs, _, _, _ = make_batch(B, H, W, fids, 4, seed, "structured")
        for f in fids:
            inputs[("color_aug", f, 0)] = inputs[("color", f, 0)]
        inputs["depth_gt"] = torch.rand(B, 1, 375, 1242) * 50 + 1
        return inputs

    class FusedTrainer(FusedLossMixin, ref.trainer.Trainer):
        def __init__(self):          # Trainer.__init__ needs KITTI on disk (trainer.py:118-139): build the state by hand
            pass
    t = FusedTrainer()
    t.md2_fused_metrics = False       # no GPU here: compute_depth_losses runs the reference's own code
    t.opt, t.device = opt, torch.device("cpu")
    t.models = {"encoder": Enc(3), "depth": Depth(), "pose_encoder": Enc(6), "pose": Pose()}
    params = [p for m in t.models.values() for p in m.parameters()]
    t.model_optimizer = torch.optim.Adam(params, 1e-4)
    t.model_lr_scheduler = torch.optim.lr_scheduler.StepLR(t.model_optimizer, 15, 0.1)
    t.use_pose_net, t.num_pose_frames, t.num_input_frames, t.num_scales = True, 2, len(fids), 4
    t.train_loader, t.val_loader = [batch(1), batch(2)], Loader([batch(3)])
    t.val_iter = iter(t.val_loader)
    t.writers = {"train": Writer(), "val": Writer()}
    t.depth_metric_names = ["de/abs_rel", "de/sq_rel", "de/rms", "de/log_rms", "da/a1", "da/a2", "da/a3"]
    t.epoch, t.step, t.start_time, t.num_total_steps = 0, 0, 0.0, 100
    t.run_epoch()                                            # two training steps, each followed by log + val
    assert t.step == 2
    # training calls never ask for side outputs; every logging step costs forward-only calls under no_grad
    train_calls = [c for c in calls if c[0]]
    assert len(train_calls) == 2 and all(c[1] is None for c in train_calls)
    lazy = [c[1] for c in calls if not c[0] and c[1]]
    assert any("depth_scales" in c for c in lazy) and any("mask_scales" in c for c in lazy)
    for mode in ("train", "val"):
        names = [n for n, _ in t.writers[mode].images]
        assert "color_pred_-1_0/0" in names and "automask_3/1" in names and "disp_0/0" in names
        assert "de/abs_rel" in t.writers[mode].scalars and "loss" in t.writers[mode].scalars


@pytest.mark.parametrize("flags", [[], ["--use_stereo"], ["--avg_reprojection"], ["--disable_automasking"],
                                   ["--no_ssim"], ["--v1_multiscale"], ["--pose_model_type", "posecnn"],
                                   ["--disable_automasking", "--predictive_mask"],
                                   ["--height", "320", "--width", "1024"], ["--frame_ids", "0", "--use_stereo"]])
def test_plan_from_the_reference_option_parser(flags):
    from monodepth2_b200 import _capi
    from monodepth2_b200.fused_loss import LossPlan
    if not os.path.exists(_capi.LIB_PATH):
        pytest.skip("libmd2loss.so not built")
    opt = _reference_options(flags)
    if opt.use_stereo:
        opt.frame_ids.append("s")                                    # trainer.py:51-52
    plan = LossPlan.from_opt(opt)
    assert (plan.batch_size, plan.height, plan.width) == (opt.batch_size, opt.height, opt.width)
    assert plan.frame_ids == opt.frame_ids and plan.scales == opt.scales
    assert plan.automask == (not opt.disable_automasking)
    assert plan.avg_reprojection == opt.avg_reprojection and plan.no_ssim == opt.no_ssim
    assert plan.v1_multiscale == opt.v1_multiscale and plan.predictive_mask == opt.predictive_mask
    assert plan.posecnn == (opt.pose_model_type == "posecnn")
    assert (plan.min_depth, plan.max_depth, plan.disparity_smoothness) == (opt.min_depth, opt.max_depth,
                                                                          opt.disparity_smoothness)


def test_predictive_mask_without_disable_automasking_raises_like_the_reference():
    from monodepth2_b200 import _capi
    from monodepth2_b200.fused_loss import LossPlan
    if not os.path.exists(_capi.LIB_PATH):
        pytest.skip("libmd2loss.so not built")
    opt = _reference_options(["--predictive_mask"])
    with pytest.raises(RuntimeError):                                # trainer.py:90-92 asserts the same
        LossPlan.from_opt(opt)
