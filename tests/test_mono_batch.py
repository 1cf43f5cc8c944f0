"""The training batch of MonoDataset on the GPU (SURVEY.md 8f-3): monodepth2_b200.mono_batch against oracle/mono_batch.py.
CPU: the oracle against a direct Pillow / torchvision run (and against the reference's KITTIRAWDataset where
MD2_REFERENCE_DIR names a checkout), the mixin's draws, the packing and the ABI's validation.  GPU: MonoBatch against
the oracle, byte for byte, and the fused loss, a CUDA graph and a multi-worker DataLoader fed by it."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from monodepth2_b200.mono_batch import NativeFramesMixin
from oracle import mono_batch as OM

Image = pytest.importorskip("PIL.Image")
T = pytest.importorskip("torchvision.transforms")
F = pytest.importorskip("torchvision.transforms.functional")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KITTI_SIZES = [(375, 1242), (376, 1241), (374, 1238), (370, 1226), (370, 1224)]     # (h, w) of the raw drives


def _frame(seed, h, w):
    """Smooth colour fields plus noise: a contrast mean away from 128, every hue, a few saturated pixels."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    base = np.stack([120 + 90 * np.sin(x / (17.0 + seed % 7) + c) * np.cos(y / 11.0 - c) for c in (0.0, 1.3, 2.6)], -1)
    return np.clip(base + rng.normal(0, 14, (h, w, 3)) + 15, 0, 255).astype(np.uint8)


def _params(seed, order=None, none=()):
    torch.manual_seed(seed)
    fn_idx, b, c, s, h = T.ColorJitter.get_params(OM.BRIGHTNESS, OM.CONTRAST, OM.SATURATION, OM.HUE)
    if order is not None:
        fn_idx = torch.tensor(order)
    fac = [b, c, s, h]
    for i in none:
        fac[i] = None
    return (fn_idx,) + tuple(fac)


# ------------------------------------------------------------------ CPU: the oracle
ORDERS = [None, [0, 1, 2, 3], [3, 2, 1, 0], [1, 3, 0, 2], [2, 0, 3, 1]]


@pytest.mark.parametrize("flip", [False, True])
@pytest.mark.parametrize("aug", range(len(ORDERS) + 2))
def test_oracle_equals_pillow_and_torchvision(flip, aug):
    """The oracle's item against the chain written out directly: flip, LANCZOS scale i from scale i-1, ToTensor, and the
    jitter (every order, a None factor, no augmentation) after each resize."""
    H, W, S = 32, 64, 4
    if aug == 0:
        p = None
    elif aug <= len(ORDERS) - 1:
        p = _params(aug, ORDERS[aug])
    else:
        p = _params(aug, [2, 1, 3, 0], none=(1,) if aug == len(ORDERS) else (0, 3))
    frames = {0: _frame(1, 50, 90), -1: _frame(2, 50, 90), 1: _frame(3, 20, 40)}
    got = OM.get_item(frames, flip, p, "l", H, W, S)
    for f, a in frames.items():
        cur = Image.fromarray(a)
        if flip:
            cur = cur.transpose(Image.FLIP_LEFT_RIGHT)
        for s in range(S):
            cur = cur.resize((W >> s, H >> s), Image.LANCZOS)
            aug_img = cur
            if p is not None:
                fn_idx, b, c, sa, h = p
                for i in fn_idx:
                    fac = [b, c, sa, h][int(i)]
                    if fac is not None:
                        aug_img = [F.adjust_brightness, F.adjust_contrast, F.adjust_saturation, F.adjust_hue][int(i)](aug_img, fac)
            want = torch.from_numpy(np.array(cur)).permute(2, 0, 1).float().div(255)
            assert torch.equal(got[("color", f, s)], want), (f, s)
            want_aug = torch.from_numpy(np.array(aug_img)).permute(2, 0, 1).float().div(255)
            assert torch.equal(got[("color_aug", f, s)], want_aug), (f, s)
    assert sorted(k for k in got if k[0] in ("K", "inv_K")) == sorted([("K", s) for s in range(S)] + [("inv_K", s) for s in range(S)])
    assert "stereo_T" not in got and ("color", 0, -1) not in got


def _write_png_drive(root, folder, sizes_by_side, n_frames):
    for side, (h, w) in sizes_by_side.items():
        d = os.path.join(root, folder, "image_0%d" % {"l": 2, "r": 3}[side], "data")
        os.makedirs(d, exist_ok=True)
        for i in range(n_frames):
            Image.fromarray(_frame(100 * i + ord(side), h, w)).save(os.path.join(d, "%010d.png" % i))


def _reference_module(name):
    ref = os.environ.get("MD2_REFERENCE_DIR", "")
    if not ref or not os.path.exists(os.path.join(ref, "datasets", "mono_dataset.py")):
        pytest.skip("MD2_REFERENCE_DIR does not name a checkout of the reference")
    sys.path.insert(0, ref)
    try:
        import importlib
        return importlib.import_module(name)
    finally:
        sys.path.remove(ref)


def test_oracle_equals_reference_kittirawdataset(tmp_path, monkeypatch):
    """The reference's own KITTIRAWDataset.__getitem__ on PNG frames, with Image.ANTIALIAS = Image.LANCZOS and the
    get_params tuple made callable, against the oracle fed the same frames and draws."""
    monkeypatch.setattr(Image, "ANTIALIAS", Image.LANCZOS, raising=False)
    datasets = _reference_module("datasets")
    orig = T.ColorJitter.get_params
    monkeypatch.setattr(T.ColorJitter, "get_params", staticmethod(lambda *a: OM.jitter_fn(orig(*a))))
    _write_png_drive(str(tmp_path), "drive", {"l": (375, 1242), "r": (375, 1242)}, 4)
    fids = [0, -1, 1, "s"]
    ds = datasets.KITTIRAWDataset(str(tmp_path), ["drive 1 l", "drive 2 r"], 192, 640, fids, 4, is_train=True,
                                  img_ext=".png")
    for index in range(2):
        for seed in range(4):
            random.seed(seed); torch.manual_seed(seed)
            want = ds[index]
            random.seed(seed); torch.manual_seed(seed)
            do_aug, do_flip, p = OM.draw(True)
            folder, fi, side = ds.filenames[index].split()
            frames = {f: np.array(ds.get_color(folder, int(fi) + (0 if f == "s" else f),
                                               {"l": "r", "r": "l"}[side] if f == "s" else side, False)) for f in fids}
            got = OM.get_item(frames, do_flip, p, side, 192, 640, 4)
            assert sorted(map(str, got)) == sorted(map(str, want))
            for k in want:
                assert torch.equal(got[k], want[k]), (index, seed, k)


class _PngDataset:
    """The part of the reference's MonoDataset / KITTIRAWDataset interface NativeFramesMixin uses, on PNG files."""

    def __init__(self, root, filenames, frame_idxs, is_train=True):
        self.data_path, self.filenames, self.frame_idxs, self.is_train = root, filenames, frame_idxs, is_train
        self.brightness, self.contrast, self.saturation, self.hue = OM.BRIGHTNESS, OM.CONTRAST, OM.SATURATION, OM.HUE
        self.load_depth = False

    def __len__(self):
        return len(self.filenames)

    def get_color(self, folder, frame_index, side, do_flip):
        p = os.path.join(self.data_path, folder, "image_0%d" % {"l": 2, "r": 3}[side], "data", "%010d.png" % frame_index)
        with open(p, "rb") as f:
            color = Image.open(f).convert("RGB")
        if do_flip:
            color = color.transpose(Image.FLIP_LEFT_RIGHT)
        return color


class _GpuPng(NativeFramesMixin, _PngDataset):
    pass


def _mixin_dataset(root, filenames, fids):
    return _GpuPng(root, filenames, fids)


def test_mixin_makes_the_oracles_draws(tmp_path):
    _write_png_drive(str(tmp_path), "d", {"l": (40, 60), "r": (40, 60)}, 3)
    ds = _mixin_dataset(str(tmp_path), ["d 1 l", "d 1 r"], [0, -1, 1, "s"])
    seen = set()
    for seed in range(24):
        random.seed(seed); torch.manual_seed(seed)
        item = ds[seed % 2]
        after = (random.random(), float(torch.rand(1)))
        random.seed(seed); torch.manual_seed(seed)
        do_aug, do_flip, p = OM.draw(True)
        assert (item["do_color_aug"], item["do_flip"]) == (do_aug, do_flip)
        if p is None:
            assert item["color_aug"] is None
        else:
            assert torch.equal(item["color_aug"][0], p[0]) and item["color_aug"][1:] == p[1:]
        assert after == (random.random(), float(torch.rand(1)))     # no draw more, no draw less
        assert item["side"] == ("l" if seed % 2 == 0 else "r")
        assert item["frames"][-1].shape == (40, 60, 3) and item["frames"][-1].dtype == np.uint8
        seen.add((do_aug, do_flip))
    assert len(seen) == 4


def test_collate_native_packs_frames_draws_and_jobs():
    from monodepth2_b200.mono_batch import JOB_DTYPE, collate_native
    from monodepth2_b200.pyramid import ColorAug
    items = []
    for b in range(3):
        p = _params(b) if b != 1 else None
        items.append({"frames": {0: _frame(b, 30 + b, 50), "s": _frame(9 + b, 30 + b, 50)}, "do_color_aug": p is not None,
                      "do_flip": b == 2, "color_aug": p, "side": "lr"[b % 2], "depth_gt": torch.full((1, 4, 5), float(b))})
    nb = collate_native(items, pin_memory=False)
    assert nb.n_images == 6 and nb.frame_ids == [0, "s"]
    jobs = nb.jobs()
    assert jobs.dtype.itemsize == 32 and JOB_DTYPE.itemsize == 32
    h = nb.buffer.numpy()
    for i in range(6):
        f, b = nb.frame_ids[i // 3], i % 3
        j = jobs[i]
        assert (j["height"], j["width"], j["flip"], j["sample"]) == (30 + b, 50, int(b == 2), b)
        a = nb.frames_offset + int(j["offset"])
        assert np.array_equal(h[a:a + 3 * 30 * 50 + 3 * b * 50].reshape(30 + b, 50, 3), items[b]["frames"][f])
    rows = ColorAug.pack_params([it["color_aug"] or ((), None, None, None, None) for it in items]).numpy()
    assert np.array_equal(h[:3 * 32].view(np.int32).reshape(3, 8), rows)
    st = h[nb.stereo_offset:nb.stereo_offset + 3 * 64].view(np.float32).reshape(3, 4, 4)
    for b in range(3):
        want = OM.get_item({0: items[b]["frames"][0][:8, :8], "s": items[b]["frames"]["s"][:8, :8]}, b == 2, None,
                           "lr"[b % 2], 8, 8, 1)["stereo_T"].numpy()
        assert np.array_equal(st[b], want)
    assert torch.equal(nb.extra["depth_gt"][:, 0, 0, 0], torch.tensor([0.0, 1.0, 2.0]))


def test_job_layout_matches_header(tmp_path):
    from monodepth2_b200.mono_batch import JOB_DTYPE
    src = tmp_path / "job.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "md2_loss.h"', 'int main(void) {',
             'printf("sizeof %zu\\n", sizeof(md2_batch_job));']
    lines += ['printf("%s %%zu\\n", offsetof(md2_batch_job, %s));' % (n, n) for n in JOB_DTYPE.names]
    src.write_text("\n".join(lines + ['return 0; }']))
    exe = tmp_path / "job"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["sizeof"]) == JOB_DTYPE.itemsize
    for n in JOB_DTYPE.names:
        assert int(got[n]) == JOB_DTYPE.fields[n][1], n


@pytest.fixture(scope="module")
def lib():
    from monodepth2_b200 import _capi, build
    build.build()
    return _capi.load_library()


def test_batch_abi_validation_without_gpu(lib):
    from monodepth2_b200.mono_batch import JOB_DTYPE
    p = C.c_void_p()
    assert lib.md2_batch_plan_create(192, 640, 5, C.byref(p)) == -1           # more than MD2_MAX_SCALES
    assert lib.md2_batch_plan_create(192, 640, 0, C.byref(p)) == -1
    assert lib.md2_batch_plan_create(4, 640, 4, C.byref(p)) == -1             # level 3 would be empty
    assert lib.md2_batch_plan_create(192, 640, 4, None) == -1
    assert lib.md2_batch_plan_create(192, 640, 4, C.byref(p)) == 0            # no device work until a size is added
    n = C.c_size_t(0)
    assert lib.md2_batch_scratch_bytes(p, 0, 0, C.byref(n)) == -1
    assert lib.md2_batch_scratch_bytes(p, 36, 1, C.byref(n)) == 0
    planes = sum((192 >> s) * (640 >> s) for s in range(4))
    assert n.value == 1280 + 36 * 3 * 192 * 320 + 36 * 3 * planes     # sums (256-aligned) | level-1 temporary | uint8 levels
    idx = C.c_int(0)
    assert lib.md2_batch_plan_add_native_size(p, 0, 1242, C.byref(idx)) == -1
    jobs = np.zeros(2, JOB_DTYPE)
    jobs["height"], jobs["width"] = 375, 1242
    jobs["offset"] = [0, 375 * 1242 * 3]
    frames = np.zeros(2 * 375 * 1242 * 3, np.uint8)
    dummy = np.zeros(1 << 20, np.uint8).ctypes.data
    args = lambda jp, ni, ns: (p, frames.ctypes.data, frames.nbytes, jp, dummy, ni, dummy, ns, dummy, 0, dummy, dummy,
                               1 << 20, None)
    assert lib.md2_batch_build_u8(*args(jobs.ctypes.data, 2, 1)) == -1        # the plan holds no size
    assert lib.md2_batch_build_u8(*args(None, 2, 1)) == -1
    assert lib.md2_batch_build_u8(*args(jobs.ctypes.data, 0, 1)) == -1
    assert lib.md2_batch_build_u8(*args(jobs.ctypes.data, 2, 0)) == -1
    assert lib.md2_batch_build_u8(None, frames.ctypes.data, frames.nbytes, jobs.ctypes.data, dummy, 2, dummy, 1, dummy, 0,
                                  dummy, dummy, 1 << 20, None) == -1
    lib.md2_batch_plan_destroy(p)


# ------------------------------------------------------------------ GPU: MonoBatch against the oracle
def _items(fids, B, sizes, seed):
    """B items: sample b flipped when b is odd, augmented when b // 2 is odd, side "l" for b < B / 2 (every flip x side
    sign of stereo_T), native size sizes[b % len(sizes)]; sample 0's frame 1 has another size than its other frames."""
    items = []
    for b in range(B):
        h, w = sizes[b % len(sizes)]
        frames = {}
        for k, f in enumerate(fids):
            hh, ww = (sizes[(b + 1) % len(sizes)] if (b == 0 and f == 1) else (h, w))
            frames[f] = _frame(seed * 1000 + b * 10 + k, hh, ww)
        aug = (b // 2) % 2 == 1
        items.append({"frames": frames, "do_color_aug": aug, "do_flip": b % 2 == 1,
                      "color_aug": _params(seed * 100 + b, none=(3,) if b == 3 else ()) if aug else None,
                      "side": "l" if b < B // 2 else "r"})
    return items


def _oracle_batch(native, height, width, S):
    items = []
    for b in range(native.batch_size):
        fr = {}
        jobs = native.jobs()
        h = native.buffer.numpy()
        for fi, f in enumerate(native.frame_ids):
            j = jobs[fi * native.batch_size + b]
            a = native.frames_offset + int(j["offset"])
            fr[f] = h[a:a + 3 * int(j["height"]) * int(j["width"])].reshape(int(j["height"]), int(j["width"]), 3)
        items.append(OM.get_item(fr, bool(native.do_flip[b]), native.color_aug[b], native.side[b], height, width, S))
    return OM.collate(items)


def _assert_equal_batch(got, want, color_dtype):
    assert sorted(map(str, got)) == sorted(map(str, want))
    for k, w in want.items():
        g = got[k].cpu()
        assert g.shape == w.shape, (k, g.shape, w.shape)
        if k[0] == "color" and color_dtype == torch.uint8:
            assert g.dtype == torch.uint8
            assert torch.equal(g, (w * 255).round().to(torch.uint8)), k             # the bytes
            assert torch.equal(g.float().div(255), w), k                           # and ToTensor of them
        else:
            assert g.dtype == w.dtype and torch.equal(g.view(torch.int32), w.view(torch.int32)), k    # bitwise


CASES = [((192, 640), [0, -1, 1], 4), ((192, 640), [0, -1, 1, "s"], 4), ((192, 640), [0, -2, -1, 1, 2], 4),
         ((192, 640), [0, -1, 1, "s"], 1), ((320, 1024), [0, -1, 1], 4), ((320, 1024), [0, -1, 1, "s"], 1),
         ((320, 1024), [0, -2, -1, 1, 2], 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%dx%d-%s-S%d" % (c[0][1], c[0][0], "".join(map(str, c[1])), c[2]))
@pytest.mark.parametrize("color_dtype", [torch.uint8, torch.float32], ids=["u8", "f32"])
def test_mono_batch_equals_oracle(case, color_dtype):
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    (H, W), fids, S = case
    sizes = KITTI_SIZES + [(H * 3 // 4, W * 3 // 4 + 3), (H - 7, W // 2)]       # the raw drives, and up-sampling
    native = collate_native(_items(fids, 8, sizes, seed=H + len(fids) + S))
    got = MonoBatch(H, W, fids, S, color_dtype=color_dtype)(native)
    _assert_equal_batch(got, _oracle_batch(native, H, W, S), color_dtype)


@pytest.mark.gpu
def test_batch_abi_rejects_bad_jobs_on_gpu():
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    fids = [0, -1]
    native = collate_native(_items(fids, 2, [(60, 100)], seed=5))
    mb = MonoBatch(32, 64, fids, 2)
    flat = mb.upload(native)
    mb.build(native, flat)
    jobs = native.jobs()
    for field, value in (("width", 99), ("size", 7), ("offset", native.buffer.numel()), ("sample", 2)):
        keep = jobs[field][1].copy()
        jobs[field][1] = value
        with pytest.raises(RuntimeError, match="invalid argument"):
            mb.build(native, flat)
        jobs[field][1] = keep
    jobs["offset"][1] = native.buffer.numel() - native.frames_offset - 60 * 100 * 3 + 1     # one byte past the end
    with pytest.raises(RuntimeError, match="invalid argument"):
        mb.build(native, flat)


@pytest.mark.gpu
def test_fused_loss_fed_mono_batch_equals_fed_oracle():
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    from monodepth2_b200.synthetic import make_batch
    B, H, W, fids = 4, 192, 640, [0, -1, 1]
    native = collate_native(_items(fids, B, KITTI_SIZES, seed=21))
    dev = torch.device("cuda:0")
    ins_u8 = MonoBatch(H, W, fids, 4)(native)
    ins_f = {k: v.to(dev) for k, v in _oracle_batch(native, H, W, 4).items()}
    _, outputs, _, noise = make_batch(B, H, W, fids, 4, 11, "structured")
    plan = LossPlan(B, H, W, fids)
    res = []
    for ins in (ins_u8, ins_f):
        outs = {k: v.to(dev).clone().requires_grad_(True) for k, v in outputs.items()}
        losses = view_synthesis_loss(plan, ins, outs, [n.to(dev) for n in noise])
        losses["loss"].backward()
        res.append((losses, outs))
    for k in res[1][0]:
        assert torch.equal(res[0][0][k], res[1][0][k]), k
    for k, v in res[1][1].items():
        if v.grad is not None:
            assert torch.equal(res[0][1][k].grad, v.grad), k


@pytest.mark.gpu
def test_cuda_graph_replay_equals_eager():
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    fids, H, W = [0, -1, 1, "s"], 192, 640
    natives = [collate_native(_items(fids, 6, KITTI_SIZES[:3], seed=s)) for s in (31, 32)]
    for nb in natives[1:]:                 # the same layout: the second batch can be copied into the first's buffer
        assert nb.buffer.numel() == natives[0].buffer.numel()
    mb = MonoBatch(H, W, fids, 4)
    eager = [{k: v.clone() for k, v in mb(nb).items()} for nb in natives]
    flat = mb.upload(natives[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        mb.build(natives[0], flat)          # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = mb.build(natives[0], flat)
    for i, nb in enumerate(natives + natives[:1]):
        flat.copy_(nb.buffer)               # the eager call wrote the size indices into nb's job table
        g.replay()
        torch.cuda.synchronize()
        for k, v in eager[i % len(natives)].items():
            assert torch.equal(out[k], v), (i, k)


@pytest.mark.gpu
def test_dataloader_with_workers_end_to_end(tmp_path):
    from torch.utils.data import DataLoader
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    _write_png_drive(str(tmp_path), "a", {"l": (375, 1242), "r": (375, 1242)}, 5)
    _write_png_drive(str(tmp_path), "b", {"l": (370, 1226), "r": (370, 1226)}, 5)
    fids = [0, -1, 1, "s"]
    names = ["%s %d %s" % (d, i, s) for d in "ab" for i in (1, 2, 3) for s in "lr"]
    ds = _mixin_dataset(str(tmp_path), names, fids)
    torch.manual_seed(0)
    loader = DataLoader(ds, batch_size=4, shuffle=True, num_workers=2, pin_memory=True, collate_fn=collate_native,
                        drop_last=False)
    mb = MonoBatch(192, 640, fids, 4)
    n = 0
    for native in loader:
        assert native.buffer.is_pinned()
        got = mb(native)
        _assert_equal_batch(got, _oracle_batch(native, 192, 640, 4), torch.uint8)
        n += native.batch_size
    assert n == len(names)
