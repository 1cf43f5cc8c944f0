"""Record the original monodepth2's drop-in interface as tests/golden/reference_interface.json.

    python tests/golden/make_reference_interface.py <directory of the original monodepth2 sources>

It imports the original's layers.py, trainer.py and options.py (after stubbing the three absent, irrelevant modules
tensorboardX / IPython / skimage, SURVEY.md App. B.1) and stores what tests/test_dropin_api.py and
tests/test_head_and_monitor.py compare with: the public names of layers.py, the parameter lists of its modules and
functions and of the Trainer methods the mixin replaces or wraps, the options MonodepthOptions parses for each flag
set the tests use, and Trainer.compute_depth_losses on seeded inputs.
"""
import inspect
import json
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "reference_interface.json")

MODULES = ["BackprojectDepth", "Project3D", "SSIM", "ConvBlock", "Conv3x3"]
FUNCTIONS = ["disp_to_depth", "transformation_from_parameters", "get_translation_matrix", "rot_from_axisangle",
             "get_smooth_loss", "upsample", "compute_depth_errors"]
TRAINER_METHODS = ["generate_images_pred", "compute_losses", "log", "compute_depth_losses"]
FLAG_SETS = [[], ["--use_stereo"], ["--avg_reprojection"], ["--disable_automasking"], ["--no_ssim"], ["--v1_multiscale"],
             ["--pose_model_type", "posecnn"], ["--disable_automasking", "--predictive_mask"],
             ["--height", "320", "--width", "1024"], ["--frame_ids", "0", "--use_stereo"], ["--predictive_mask"]]
OPTION_FIELDS = ["batch_size", "height", "width", "frame_ids", "scales", "min_depth", "max_depth",
                 "disparity_smoothness", "use_stereo", "avg_reprojection", "disable_automasking", "no_ssim",
                 "v1_multiscale", "predictive_mask", "pose_model_type"]
DEPTH_METRIC_NAMES = ["de/abs_rel", "de/sq_rel", "de/rms", "de/log_rms", "da/a1", "da/a2", "da/a3"]


def depth_metric_inputs():
    """The seeded inputs of test_oracle_depth_metrics_equal_the_reference_method."""
    g = torch.Generator().manual_seed(0)
    depth = torch.rand(3, 1, 48, 160, generator=g) * 40 + 0.5
    gt = torch.rand(3, 1, 375, 1242, generator=g) * 60
    gt[torch.rand(gt.shape, generator=g) < 0.7] = 0            # sparse LiDAR ground truth
    return depth, gt


def _params(fn):
    return [p.name for p in inspect.signature(fn).parameters.values()]


def _import_reference(ref_dir):
    for name, attrs in (("tensorboardX", {"SummaryWriter": object}), ("IPython", {"embed": lambda *a, **k: None}),
                        ("skimage", {}), ("skimage.transform", {})):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules.setdefault(name, m)
    sys.modules["skimage"].transform = sys.modules["skimage.transform"]
    sys.dont_write_bytecode = True
    sys.path.insert(0, ref_dir)
    try:
        import layers
        import trainer
        from options import MonodepthOptions
    finally:
        sys.path.remove(ref_dir)
    return layers, trainer, MonodepthOptions


def record(ref_dir):
    layers, trainer, MonodepthOptions = _import_reference(ref_dir)
    out = {
        "source": "recorded from the original monodepth2 sources with make_reference_interface.py",
        "layers_public": sorted(n for n, v in vars(layers).items()
                                if not n.startswith("_") and getattr(v, "__module__", None) == layers.__name__),
        "modules": {n: {"__init__": _params(getattr(layers, n).__init__), "forward": _params(getattr(layers, n).forward)}
                    for n in MODULES},
        "functions": {n: _params(getattr(layers, n)) for n in FUNCTIONS},
        "trainer_methods": {m: _params(getattr(trainer.Trainer, m)) for m in TRAINER_METHODS},
        "options": {},
    }
    for flags in FLAG_SETS:
        sys.argv = ["train.py"] + flags
        opt = MonodepthOptions().parse()
        out["options"][" ".join(flags)] = {k: getattr(opt, k) for k in OPTION_FIELDS}
    depth, gt = depth_metric_inputs()
    me = types.SimpleNamespace(depth_metric_names=DEPTH_METRIC_NAMES)
    losses = {}
    trainer.Trainer.compute_depth_losses(me, {"depth_gt": gt}, {("depth", 0, 0): depth}, losses)
    out["depth_metrics"] = {k: float(losses[k]) for k in DEPTH_METRIC_NAMES}
    return out


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(sys.argv[1]):
        sys.exit(__doc__)
    data = record(os.path.abspath(sys.argv[1]))
    with open(OUT, "w") as f:
        json.dump(data, f, indent=1)
        f.write("\n")
    print("wrote", OUT)
