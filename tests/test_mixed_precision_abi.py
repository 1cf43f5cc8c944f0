"""CPU-side checks of the reduced-precision (bf16 / fp16) fields of the C ABI and of the Python refusals.

The workspace of an all-fp32 problem must not change when the dtype fields exist: the size at the default workload
(640x192, batch 12, two sources, 4 scales, automasking, with gradients) is pinned to the value of the library before
they were added."""
import ctypes as C

import pytest
import torch

BASELINE_WORKSPACE_BYTES = 196493312


@pytest.fixture(scope="module")
def lib():
    from monodepth2_b200 import build, _capi
    build.build()
    return _capi.load_library()


def _baseline(**kw):
    from monodepth2_b200._capi import Md2Problem
    return Md2Problem(batch=12, height=192, width=640, num_scales=4, num_src=2, automask=1, min_depth=0.1,
                      max_depth=100.0, disparity_smoothness=1e-3, want_grad=1, **kw)


def _ws(lib, p):
    n = C.c_size_t(0)
    st = lib.md2_loss_workspace_bytes(C.byref(p), C.byref(n))
    return st, n.value


def test_version_and_dtype_codes(lib):
    from monodepth2_b200 import _capi
    assert lib.md2_version() == 101
    assert (_capi.DTYPE_F32, _capi.DTYPE_BF16, _capi.DTYPE_F16) == (0, 1, 2)


def test_all_fp32_workspace_is_unchanged(lib):
    assert _ws(lib, _baseline()) == (0, BASELINE_WORKSPACE_BYTES)


def test_reduced_precision_leaves_reserve_their_fp32_copies(lib):
    B, H, W = 12, 192, 640
    disp = sum(B * (H >> s) * (W >> s) * 4 for s in range(4))
    st, n = _ws(lib, _baseline(disp_dtype=1))
    assert st == 0 and n >= BASELINE_WORKSPACE_BYTES + disp
    st, n2 = _ws(lib, _baseline(disp_dtype=2))
    assert st == 0 and n2 == n
    pose = (C.c_int * 4)(1, 0, 0, 0)
    st, n3 = _ws(lib, _baseline(pose_dtype=pose))
    assert st == 0 and BASELINE_WORKSPACE_BYTES < n3 < BASELINE_WORKSPACE_BYTES + 4096
    # a mask dtype without --predictive_mask has nothing to widen
    assert _ws(lib, _baseline(pmask_dtype=1)) == (0, BASELINE_WORKSPACE_BYTES)
    pm = _baseline(pmask_dtype=1, predictive_mask=1)
    pm.automask = 0
    pm0 = _baseline(predictive_mask=1)
    pm0.automask = 0
    assert _ws(lib, pm)[1] > _ws(lib, pm0)[1]


@pytest.mark.parametrize("field", ["disp_dtype", "pose_dtype", "pmask_dtype"])
@pytest.mark.parametrize("bad", [3, -1])
def test_unknown_dtype_is_refused(lib, field, bad):
    from monodepth2_b200._capi import Md2Tensors
    p = _baseline()
    if field == "pose_dtype":
        p.pose_dtype[3] = bad            # checked for every slot, used or not
    else:
        setattr(p, field, bad)
    assert _ws(lib, p)[0] == -1
    t = Md2Tensors()
    assert lib.md2_view_synthesis_loss(C.byref(p), C.byref(t), None, 0, None) == -1


def test_typed_entry_points_refuse_bad_arguments_without_a_gpu(lib):
    one = (C.c_void_p * 1)(16)
    cnt = (C.c_longlong * 1)(4)
    for bad in (3, -1):
        dt = (C.c_int * 1)(bad)
        assert lib.md2_scale_tensors_typed(1, one, one, dt, cnt, C.c_void_p(16), None) == -1
    dt = (C.c_int * 1)(1)
    assert lib.md2_scale_tensors_typed(0, one, one, dt, cnt, C.c_void_p(16), None) == -1
    assert lib.md2_scale_tensors_typed(17, one, one, dt, cnt, C.c_void_p(16), None) == -1
    assert lib.md2_scale_tensors_typed(1, one, one, None, cnt, C.c_void_p(16), None) == -1
    assert lib.md2_dispconv_sigmoid_typed(16, 16, 16, 16, 3, 1, 4, 8, 8, None) == -1
    assert lib.md2_dispconv_sigmoid_backward_typed(16, 16, 16, 16, 16, 16, 16, 3, 1, 4, 8, 8, None) == -1
    assert lib.md2_dispconv_sigmoid_typed(None, 16, 16, 16, 1, 1, 4, 8, 8, None) == -1


def test_leaf_dtype_rules():
    from monodepth2_b200.fused_loss import _one_dtype
    f, b, h = (torch.zeros(2, dtype=d) for d in (torch.float32, torch.bfloat16, torch.float16))
    assert _one_dtype([f, f], ["a", "b"], "x") == 0
    assert _one_dtype([b, b], ["a", "b"], "x") == 1
    assert _one_dtype([h], ["a"], "x") == 2
    assert _one_dtype([], [], "x") == 0
    with pytest.raises(RuntimeError, match=r"disp\[0\] torch.float32, disp\[1\] torch.bfloat16"):
        _one_dtype([f, b], ["disp[0]", "disp[1]"], "the disparities")
    with pytest.raises(RuntimeError, match=r"disp\[0\] torch.float64"):
        _one_dtype([f.double()], ["disp[0]"], "the disparities")
