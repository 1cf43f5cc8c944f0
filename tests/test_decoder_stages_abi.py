"""CPU-side checks of the fused decoder stages: the argument refusals of md2_upcat_pad / md2_upcat_pad_backward (they
run before any CUDA call), and what fuse_decoder_stages does to a reference DepthDecoder's module tree - the same
Parameter objects and state_dict keys, either order with fuse_disp_heads, and a RuntimeError on a structure it does not
recognise."""
import ctypes as C

import pytest
import torch

ENC18 = [64, 64, 128, 256, 512]
P = C.c_void_p(256)            # never dereferenced: every call below is refused before it reaches the device


@pytest.fixture(scope="module")
def lib():
    from monodepth2_b200 import build, _capi
    build.build()
    return _capi.load_library()


def _fwd(lib, dtype=0, batch=2, cx=4, cs=3, h=5, w=6, up=2, x=P, skip=P, out=P):
    return lib.md2_upcat_pad(x, skip, out, dtype, batch, cx, cs, h, w, up, None)


def _bwd(lib, dtype=0, batch=2, cx=4, cs=3, h=5, w=6, up=2, g=P, gx=P, gs=P):
    return lib.md2_upcat_pad_backward(g, gx, gs, dtype, batch, cx, cs, h, w, up, None)


@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("bad", [
    dict(dtype=3), dict(dtype=-1),
    dict(up=0), dict(up=3), dict(up=-2),
    dict(h=1, up=1), dict(w=1, up=1), dict(h=0), dict(w=0),          # ReflectionPad2d(1) needs 2 values an axis
    dict(cx=0), dict(cs=-1), dict(batch=0),
])
def test_argument_refusals(lib, call, bad):
    assert call(lib, **bad) == -1


def test_pointer_refusals(lib):
    assert _fwd(lib, x=None) == -1
    assert _fwd(lib, out=None) == -1
    assert _fwd(lib, skip=None) == -1                 # Cs > 0 needs a skip
    assert _bwd(lib, g=None) == -1


def test_too_many_elements_is_unsupported(lib):
    # out would hold 2^31 or more values: the kernels index with 32 bits
    assert _fwd(lib, batch=128, cx=512, cs=512, h=64, w=64) == -2
    assert _bwd(lib, batch=128, cx=512, cs=512, h=64, w=64) == -2


def test_upcat_pad_refuses_cpu_tensors():
    from monodepth2_b200.layers import upcat_pad
    with pytest.raises(RuntimeError, match="x must be a CUDA tensor"):
        upcat_pad(torch.zeros(1, 2, 3, 3))


def _oracle(**kw):
    from oracle.depth_decoder import DepthDecoder
    torch.manual_seed(0)
    return DepthDecoder(ENC18, **kw)


@pytest.mark.parametrize("kw", [{}, dict(scales=[0, 2]), dict(use_skips=False), dict(num_output_channels=2)])
def test_fuse_keeps_parameters_and_state_dict(kw):
    from monodepth2_b200.layers import fuse_decoder_stages
    dec = _oracle(**kw)
    keys = list(dec.state_dict().keys())
    params = [(n, p) for n, p in dec.named_parameters()]
    mods = dict(dec.convs)
    assert fuse_decoder_stages(dec) is dec
    assert list(dec.state_dict().keys()) == keys
    assert [(n, id(p)) for n, p in dec.named_parameters()] == [(n, id(p)) for n, p in params]
    assert all(dec.convs[k] is m for k, m in mods.items())
    assert dec.forward.__func__.__name__ == "_fused_decoder_forward"


@pytest.mark.parametrize("heads_first", [False, True])
def test_either_order_with_fuse_disp_heads(heads_first):
    from monodepth2_b200.layers import DispConvSigmoid, fuse_decoder_stages, fuse_disp_heads
    dec = _oracle()
    keys = list(dec.state_dict().keys())
    ids = [id(p) for p in dec.parameters()]
    for f in ((fuse_disp_heads, fuse_decoder_stages) if heads_first else (fuse_decoder_stages, fuse_disp_heads)):
        assert f(dec) is dec
    assert list(dec.state_dict().keys()) == keys
    assert [id(p) for p in dec.parameters()] == ids
    assert all(isinstance(dec.convs[("dispconv", s)], DispConvSigmoid) for s in range(4))
    assert isinstance(dec.sigmoid, torch.nn.Identity)
    assert dec.forward.__func__.__name__ == "_fused_decoder_forward"


def test_refuses_the_stand_in_decoder():
    from benchmarks.train_step import DepthDecoder as StandIn
    from monodepth2_b200.layers import fuse_decoder_stages
    with pytest.raises(RuntimeError, match="convs"):
        fuse_decoder_stages(StandIn(ENC18))


def test_refuses_a_zero_padded_head():
    from monodepth2_b200.layers import Conv3x3, fuse_decoder_stages
    dec = _oracle()
    dec.convs[("dispconv", 1)] = Conv3x3(32, 1, use_refl=False)
    with pytest.raises(RuntimeError, match=r"dispconv', 1"):
        fuse_decoder_stages(dec)


def test_refuses_a_zero_padded_block_and_a_missing_stage():
    from monodepth2_b200.layers import Conv3x3, fuse_decoder_stages
    dec = _oracle()
    dec.convs[("upconv", 2, 1)].conv = Conv3x3(128, 64, use_refl=False)
    with pytest.raises(RuntimeError, match=r"upconv', 2, 1"):
        fuse_decoder_stages(dec)
    dec = _oracle()
    del dec.convs[("upconv", 3, 0)]
    with pytest.raises(RuntimeError, match=r"'upconv', 3, 0"):
        fuse_decoder_stages(dec)
    dec = _oracle(scales=[0])
    del dec.convs[("dispconv", 0)]
    with pytest.raises(RuntimeError, match=r"dispconv', 0"):
        fuse_decoder_stages(dec)


def test_refused_decoder_is_left_unchanged():
    from monodepth2_b200.layers import Conv3x3, fuse_decoder_stages
    dec = _oracle()
    dec.convs[("dispconv", 3)] = Conv3x3(128, 1, use_refl=False)
    with pytest.raises(RuntimeError):
        fuse_decoder_stages(dec)
    assert "forward" not in vars(dec)
