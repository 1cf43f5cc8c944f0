"""The fused decoder stages on the GPU: upcat_pad = ReflectionPad2d(1)(cat([nearest_up(x, up), skip], 1)) against
torch's chain, and fuse_decoder_stages on the reference DepthDecoder (oracle/depth_decoder.py) against the unfused one.

- Forward is pure data movement: bitwise torch's chain in every dtype.
- Backward (fp32): bitwise torch's chain wherever every fold that feeds an element has at most two terms (torch's
  zero-initialised atomic adds of two terms are exact in any order); every element within 2^-24 (n - 1) sum|terms| of
  the float64 chain on the CPU, n the element's term count.  bf16 / fp16: bitwise the fp32 path on grad_out.float(),
  rounded once.  Two runs are bitwise equal.
- The decoder: disparities bitwise equal (fp32 and autocast bf16), gradients as close to a float64 run as the unfused
  chain's (1.5x its relL2 error + 1e-6) and within relL2 2e-5 of them; under
  torch.use_deterministic_algorithms(True) the fused decoder runs, reproducibly; its forward + backward launch none of
  torch's pad / up-sample / cat kernels; one CUDA-graph capture of forward + backward replays to the eager result.
"""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DT = [torch.float32, torch.bfloat16, torch.float16]
ENC = {18: [64, 64, 128, 256, 512], 50: [64, 256, 512, 1024, 2048]}
DEC = [16, 32, 64, 128, 256]
B, H, W = 12, 192, 640


def block_inputs(layers):
    """(Cx, Cs, h, w, up) of the 10 ConvBlock inputs of the reference decoder at 640x192 (depth_decoder.py:48-65)."""
    enc, out = ENC[layers], []
    for i in range(4, -1, -1):
        h, w = H >> (i + 1), W >> (i + 1)
        out.append((enc[-1] if i == 4 else DEC[i + 1], 0, h, w, 1))            # ("upconv", i, 0): pad only
        out.append((DEC[i], enc[i - 1] if i > 0 else 0, h, w, 2))               # ("upconv", i, 1): up + cat + pad
    return out


FULL = sorted(set(block_inputs(18) + block_inputs(50)))
EDGE = [  # (B, Cx, Cs, h, w, up)
    (2, 3, 2, 1, 5, 2), (2, 3, 2, 4, 1, 2), (3, 2, 0, 1, 1, 2),      # h or w of 1, up-sampled to 2
    (2, 4, 0, 2, 3, 1), (2, 4, 0, 3, 2, 1), (2, 3, 0, 3, 3, 1),      # 2 and 3 after "up-sampling" by 1
    (2, 5, 3, 5, 7, 2), (1, 3, 0, 7, 9, 1), (2, 2, 5, 3, 3, 2),      # odd sizes
    (2, 1, 0, 4, 6, 2), (2, 1, 0, 5, 4, 1), (2, 1, 1, 6, 5, 2),      # Cx = 1, Cs = 0
]


def ref_chain(x, skip, up):
    y = F.interpolate(x, scale_factor=2, mode="nearest") if up == 2 else x
    if skip is not None:
        y = torch.cat([y, skip], 1)
    return F.pad(y, (1, 1, 1, 1), mode="reflect")


def make(b, cx, cs, h, w, up, dtype=torch.float32, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(b, cx, h, w, device="cuda", generator=g).to(dtype)
    skip = torch.randn(b, cs, up * h, up * w, device="cuda", generator=g).to(dtype) if cs else None
    return x, skip


def bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def assert_bitwise(a, b, what=""):
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    eq = bits(a.contiguous()) == bits(b.contiguous())
    assert bool(eq.all()), "%s: %d of %d elements differ" % (what, int((~eq).sum()), eq.numel())


# ------------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("dtype", DT, ids=str)
@pytest.mark.parametrize("shape", FULL, ids=lambda s: "Cx%d_Cs%d_%dx%d_up%d" % s)
def test_forward_decoder_shapes_bitwise(shape, dtype):
    from monodepth2_b200.layers import upcat_pad
    cx, cs, h, w, up = shape
    x, skip = make(B, cx, cs, h, w, up, dtype)
    assert_bitwise(upcat_pad(x, skip, up), ref_chain(x, skip, up))


@pytest.mark.parametrize("dtype", DT, ids=str)
@pytest.mark.parametrize("shape", EDGE, ids=lambda s: "B%d_Cx%d_Cs%d_%dx%d_up%d" % s)
def test_forward_edge_shapes_bitwise(shape, dtype):
    from monodepth2_b200.layers import upcat_pad
    b, cx, cs, h, w, up = shape
    x, skip = make(b, cx, cs, h, w, up, dtype, seed=1)
    assert_bitwise(upcat_pad(x, skip, up), ref_chain(x, skip, up))


@pytest.mark.parametrize("xd,sd", [(torch.bfloat16, torch.float32), (torch.float32, torch.float16),
                                   (torch.bfloat16, torch.float16), (torch.float16, torch.bfloat16)], ids=str)
def test_mixed_dtypes_follow_torch_cat(xd, sd):
    from monodepth2_b200.layers import upcat_pad
    x = torch.randn(2, 3, 5, 6, device="cuda").to(xd).requires_grad_(True)
    skip = torch.randn(2, 4, 10, 12, device="cuda").to(sd).requires_grad_(True)
    out = upcat_pad(x, skip)
    ref = ref_chain(x, skip, 2)
    assert out.dtype == ref.dtype == torch.promote_types(xd, sd)
    assert_bitwise(out, ref)
    g = torch.randn_like(out)
    gx, gs = torch.autograd.grad(out, (x, skip), g)
    assert gx.dtype == xd and gs.dtype == sd
    # the gradients are the promoted-dtype path's, cast back to each input's dtype
    xp, sp = x.detach().to(out.dtype).requires_grad_(True), skip.detach().to(out.dtype).requires_grad_(True)
    gxp, gsp = torch.autograd.grad(upcat_pad(xp, sp), (xp, sp), g)
    assert_bitwise(gx, gxp.to(xd), "grad_x")
    assert_bitwise(gs, gsp.to(sd), "grad_skip")


@pytest.mark.parametrize("dtype", DT, ids=str)
def test_channels_last_and_sliced_inputs(dtype):
    from monodepth2_b200.layers import upcat_pad
    x, skip = make(2, 6, 5, 7, 9, 2, dtype, seed=2)
    xs = x[:, 1:4]                                              # non-contiguous slices
    ss = skip[:, ::2]
    assert_bitwise(upcat_pad(xs, ss), ref_chain(xs, ss, 2), "sliced")
    xc, sc = x.to(memory_format=torch.channels_last), skip.to(memory_format=torch.channels_last)
    assert not xc.is_contiguous()
    assert_bitwise(upcat_pad(xc, sc), ref_chain(x, skip, 2), "channels_last")
    assert_bitwise(upcat_pad(xc, up=1), ref_chain(x, None, 1), "channels_last, up=1")
    # gradients of a sliced input land in the right place
    leaf = x.clone().requires_grad_(True)
    g = torch.randn(2, 3 + 3, 16, 20, device="cuda").to(dtype)
    (gl,) = torch.autograd.grad(upcat_pad(leaf[:, 1:4], ss), (leaf,), g)
    assert bool((gl[:, [0, 4, 5]] == 0).all())
    xx = x[:, 1:4].contiguous().requires_grad_(True)
    (gxx,) = torch.autograd.grad(upcat_pad(xx, ss), (xx,), g)
    assert_bitwise(gl[:, 1:4].contiguous(), gxx)


def test_refusals_on_the_gpu():
    from monodepth2_b200.layers import upcat_pad
    x = torch.zeros(1, 2, 3, 3, device="cuda")
    with pytest.raises(RuntimeError, match="x must be float32, bfloat16 or float16"):
        upcat_pad(x.double())
    with pytest.raises(RuntimeError, match="skip must be float32, bfloat16 or float16"):
        upcat_pad(x, torch.zeros(1, 1, 6, 6, device="cuda", dtype=torch.int32))
    with pytest.raises(RuntimeError, match="skip must be a CUDA tensor"):
        upcat_pad(x, torch.zeros(1, 1, 6, 6))
    with pytest.raises(RuntimeError, match="does not fit"):
        upcat_pad(x, torch.zeros(1, 1, 5, 6, device="cuda"))
    with pytest.raises(RuntimeError, match="up must be 1 or 2"):
        upcat_pad(x, up=3)
    with pytest.raises(RuntimeError):                              # ReflectionPad2d refuses a 1-value axis too
        upcat_pad(torch.zeros(1, 2, 1, 3, device="cuda"), up=1)


# ------------------------------------------------------------------------------------------------------ backward
def fold_counts(n):
    """Per up-sampled index of an axis of length n: how many padded positions fold onto it."""
    c = torch.ones(n, dtype=torch.int64)
    c[1] += 1
    c[n - 2] += 1
    return c


def max_fold_terms(h, w, up, for_x):
    """Largest fold term count that feeds each element of grad_x (for_x) or grad_skip, as an (h', w') map."""
    f = fold_counts(up * h)[:, None] * fold_counts(up * w)[None, :]
    if for_x and up == 2:
        f = F.max_pool2d(f[None, None].double(), 2)[0, 0].long()
    return f


def f64_chain_grads(x, skip, up, g):
    xd = x.detach().double().cpu().requires_grad_(True)
    sd = skip.detach().double().cpu().requires_grad_(True) if skip is not None else None
    leaves = (xd,) + ((sd,) if sd is not None else ())
    return torch.autograd.grad(ref_chain(xd, sd, up), leaves, g.double().cpu())


def check_backward_fp32(b, cx, cs, h, w, up, seed):
    from monodepth2_b200.layers import upcat_pad
    x, skip = make(b, cx, cs, h, w, up, seed=seed)
    x.requires_grad_(True)
    if skip is not None:
        skip.requires_grad_(True)
    leaves = (x,) + ((skip,) if skip is not None else ())
    out = upcat_pad(x, skip, up)
    g = torch.randn(out.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed + 7))
    ours = torch.autograd.grad(out, leaves, g)
    torch_ = torch.autograd.grad(ref_chain(x, skip, up), leaves, g)
    exact = f64_chain_grads(x, skip, up, g)
    n_terms = f64_chain_grads(x, skip, up, torch.ones_like(g))
    abs_sum = f64_chain_grads(x, skip, up, g.abs())
    for k, (o, t, e, n, s) in enumerate(zip(ours, torch_, exact, n_terms, abs_sum)):
        name = "grad_x" if k == 0 else "grad_skip"
        mask = max_fold_terms(h, w, up, k == 0).cuda() <= 2
        mask = mask.expand_as(o)
        assert bool((bits(o[mask]) == bits(t[mask])).all()), "%s differs from torch where every fold has <= 2 terms" % name
        bound = 2.0 ** -24 * (n - 1).clamp_min(0) * s * (1 + 1e-6)
        err = (o.double().cpu() - e).abs()
        assert bool((err <= bound).all()), "%s: max excess %g" % (name, float((err - bound).max()))
    # two runs are bitwise equal
    again = torch.autograd.grad(upcat_pad(x, skip, up), leaves, g)
    for a, o in zip(again, ours):
        assert_bitwise(a, o, "rerun")
    return x, skip, g, ours


@pytest.mark.parametrize("shape", EDGE, ids=lambda s: "B%d_Cx%d_Cs%d_%dx%d_up%d" % s)
def test_backward_edge_shapes(shape):
    check_backward_fp32(*shape, seed=3)


@pytest.mark.parametrize("shape", sorted(set(block_inputs(18))), ids=lambda s: "Cx%d_Cs%d_%dx%d_up%d" % s)
def test_backward_resnet18_shapes(shape):
    cx, cs, h, w, up = shape
    check_backward_fp32(2, cx, cs, h, w, up, seed=4)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=str)
@pytest.mark.parametrize("shape", EDGE[:9] + [(B, 32, 64, 48, 160, 2), (B, 16, 0, 96, 320, 2)],
                         ids=lambda s: "B%d_Cx%d_Cs%d_%dx%d_up%d" % s)
def test_backward_reduced_precision_is_the_rounded_fp32_path(shape, dtype):
    from monodepth2_b200.layers import upcat_pad
    b, cx, cs, h, w, up = shape
    x, skip = make(b, cx, cs, h, w, up, dtype, seed=5)
    x.requires_grad_(True)
    leaves = (x,)
    if skip is not None:
        skip.requires_grad_(True)
        leaves += (skip,)
    out = upcat_pad(x, skip, up)
    g = torch.randn(out.shape, device="cuda").to(dtype)
    ours = torch.autograd.grad(out, leaves, g)
    x32 = x.detach().float().requires_grad_(True)
    s32 = skip.detach().float().requires_grad_(True) if skip is not None else None
    leaves32 = (x32,) + ((s32,) if s32 is not None else ())
    ref = torch.autograd.grad(upcat_pad(x32, s32, up), leaves32, g.float())
    for o, r in zip(ours, ref):
        assert o.dtype == dtype
        assert_bitwise(o, r.to(dtype))
    again = torch.autograd.grad(upcat_pad(x, skip, up), leaves, g)
    for a, o in zip(again, ours):
        assert_bitwise(a, o, "rerun")


def test_backward_skip_only_and_x_only():
    from monodepth2_b200.layers import upcat_pad
    x, skip = make(2, 3, 4, 5, 6, 2, seed=6)
    g = torch.randn(2, 7, 12, 14, device="cuda")
    xa, sa = x.clone().requires_grad_(True), skip.clone().requires_grad_(True)
    gx_both, gs_both = torch.autograd.grad(upcat_pad(xa, sa), (xa, sa), g)
    (gx,) = torch.autograd.grad(upcat_pad(xa, skip), (xa,), g)
    (gs,) = torch.autograd.grad(upcat_pad(x, sa), (sa,), g)
    assert_bitwise(gx, gx_both)
    assert_bitwise(gs, gs_both)


# ------------------------------------------------------------------------------------------------------ the decoder
def features(layers, b, dtype=torch.float32, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(b, c, H >> (i + 1), W >> (i + 1), device="cuda", generator=g).to(dtype)
            for i, c in enumerate(ENC[layers])]


def decoders(heads_fused, **kw):
    from monodepth2_b200.layers import fuse_decoder_stages, fuse_disp_heads
    from oracle.depth_decoder import DepthDecoder
    torch.manual_seed(0)
    ref = DepthDecoder(ENC[18], **kw).cuda()
    fused = copy.deepcopy(ref)
    if heads_fused:
        fuse_disp_heads(ref)
        fuse_disp_heads(fused)
    fuse_decoder_stages(fused)
    return ref, fused


def run(dec, feats, seed=0):
    """Forward, then the gradients of a fixed random projection of the disparities w.r.t. the parameters and the
    features."""
    feats = [f.detach().clone().requires_grad_(True) for f in feats]
    outs = dec(feats)
    keys = sorted(outs)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    loss = sum((outs[k].double() * torch.randn(outs[k].shape, device="cuda", generator=gen).double()).sum()
               for k in keys)
    params = [p for p in dec.parameters()]
    grads = torch.autograd.grad(loss, params + feats, allow_unused=True)      # use_skips=False leaves features unused
    return [outs[k].detach() for k in keys], list(grads)


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


@pytest.fixture
def cudnn_deterministic():
    """Both arms pick the same convolution algorithms, in full fp32: with TF32 a last-bit difference in a gradient can
    round differently to 10 mantissa bits and hide the fold-order differences the comparison is about."""
    c = torch.backends.cudnn
    prev = c.deterministic, c.benchmark, c.allow_tf32
    c.deterministic, c.benchmark, c.allow_tf32 = True, False, False
    yield
    c.deterministic, c.benchmark, c.allow_tf32 = prev


def float64_arm(feats, **kw):
    """The unfused reference decoder in float64, same initial parameters as decoders()."""
    from oracle.depth_decoder import DepthDecoder
    torch.manual_seed(0)
    return run(DepthDecoder(ENC[18], **kw).cuda().double(), [f.double() for f in feats])


def assert_gradients_as_accurate(g_fus, g_ref, g_64, names):
    """The fused and unfused gradients differ only by the order of the sums at 3- and 4-term folds.  Through ten
    ConvBlocks such rounding differences reach a weight gradient that cancels strongly (the deepest block's, a sum over
    all pixels of terms of both signs) amplified to a few 1e-6 relL2, so the bound is relative to the error the unfused
    chain makes itself: against float64 the fused gradient may be at most 1.5x as far off, plus 1e-6 relL2."""
    for n, a, b, r in zip(names, g_fus, g_ref, g_64):
        if b is None:                                  # a feature the decoder does not read (use_skips=False)
            assert a is None and r is None, n
            continue
        e_f, e_u = rel_l2(a, r), rel_l2(b, r)
        assert e_f <= 1.5 * e_u + 1e-6, (n, e_f, e_u)
        assert rel_l2(a, b) <= 2e-5, (n, rel_l2(a, b))


@pytest.mark.parametrize("heads_fused", [False, True], ids=["heads_unfused", "heads_fused"])
@pytest.mark.parametrize("kw", [{}, dict(scales=(0, 2)), dict(use_skips=False)], ids=["default", "scales02", "no_skips"])
def test_decoder_matches_unfused(kw, heads_fused, cudnn_deterministic):
    ref, fused = decoders(heads_fused, **kw)
    feats = features(18, 2)
    d_ref, g_ref = run(ref, feats)
    d_fus, g_fus = run(fused, feats)
    assert len(d_ref) == len(d_fus) == len(kw.get("scales", range(4)))
    assert set(fused.outputs) == set(ref.outputs)
    for a, b in zip(d_fus, d_ref):
        assert_bitwise(a, b, "disp")
    names = [n for n, _ in ref.named_parameters()] + ["feature%d" % i for i in range(5)]
    assert_gradients_as_accurate(g_fus, g_ref, float64_arm(feats, **kw)[1], names)


@pytest.mark.parametrize("heads_fused", [False, True], ids=["heads_unfused", "heads_fused"])
def test_decoder_autocast_bf16_disparities_bitwise(heads_fused, cudnn_deterministic):
    ref, fused = decoders(heads_fused)
    feats = features(18, 2)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        d_ref = ref(feats)
        d_fus = fused(feats)
    assert set(d_ref) == set(d_fus)
    for k in d_ref:
        assert d_fus[k].dtype == d_ref[k].dtype == torch.bfloat16
        assert_bitwise(d_fus[k], d_ref[k], str(k))
    # and the backward runs, with gradients close to the unfused chain's (which rounds to bf16 between its ops)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        _, g_ref = run(ref, feats)
        _, g_fus = run(fused, feats)
    for a, b in zip(g_fus, g_ref):
        assert a.dtype == b.dtype and bool(torch.isfinite(a).all())
        assert rel_l2(a, b) <= 2e-2


def test_decoder_num_output_channels(cudnn_deterministic):
    ref, fused = decoders(False, num_output_channels=2)
    feats = features(18, 1)
    d_ref, g_ref = run(ref, feats)
    d_fus, g_fus = run(fused, feats)
    for a, b in zip(d_fus, d_ref):
        assert a.shape[1] == 2
        assert_bitwise(a, b)
    names = [n for n, _ in ref.named_parameters()] + ["feature%d" % i for i in range(5)]
    assert_gradients_as_accurate(g_fus, g_ref, float64_arm(feats, num_output_channels=2)[1], names)


@pytest.fixture
def deterministic_mode(cudnn_deterministic):
    prev = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def test_deterministic_mode(deterministic_mode):
    """The fused decoder runs under torch.use_deterministic_algorithms(True) and gives bitwise-equal results twice.
    (The installed torch does not refuse the unfused decoder there: it switches reflection_pad2d's backward to a
    deterministic kernel of its own, see test_kernels_launched.)"""
    assert torch.utils.deterministic.fill_uninitialized_memory      # unwritten output elements would read NaN
    feats = features(18, 2)
    _, fused = decoders(False)
    d1, g1 = run(fused, feats)
    d2, g2 = run(fused, feats)
    for a, b in zip(d1 + g1, d2 + g2):
        assert bool(torch.isfinite(a).all())
        assert_bitwise(a, b, "rerun")
    _, fused_heads = decoders(True)
    d, g = run(fused_heads, feats)
    assert all(bool(torch.isfinite(t).all()) for t in d + g)


def kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def test_kernels_launched(cudnn_deterministic):
    """The fused decoder's forward + backward launch md2_decoder's two kernels and none of torch's pad, up-sample or
    cat kernels; the unfused one runs reflection_pad2d's atomic backward, or its deterministic variant in deterministic
    mode."""
    feats = features(18, 1)
    ref, fused = decoders(False)
    torch_ops = ("reflection_pad", "upsample_nearest", "CatArray")
    names = kernel_names(lambda: run(fused, feats))
    assert any("k_upcat_pad<" in n or "k_upcat_pad(" in n or "k_upcat_padI" in n for n in names), sorted(names)
    assert any("k_upcat_pad_bwd" in n for n in names), sorted(names)
    assert not [n for n in names if any(t in n for t in torch_ops)]
    names = kernel_names(lambda: run(ref, feats))
    pad_bwd = [n for n in names if "reflection_pad2d_backward" in n]
    assert pad_bwd and not [n for n in pad_bwd if "det" in n], pad_bwd
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        names = kernel_names(lambda: run(ref, feats))
    finally:
        torch.use_deterministic_algorithms(prev)
    assert [n for n in names if "reflection_pad2d_backward_det" in n], sorted(names)


def test_cuda_graph_replay_equals_eager(cudnn_deterministic):
    _, fused = decoders(False)
    feats = [f.requires_grad_(True) for f in features(18, 2, seed=1)]
    params = list(fused.parameters())
    with torch.no_grad():
        gout = [torch.randn_like(d) for d in (fused(feats)[("disp", s)] for s in range(4))]

    def step():
        outs = fused(feats)
        disp = [outs[("disp", s)] for s in range(4)]
        return disp, list(torch.autograd.grad(disp, params + feats, gout))

    # everything on one side stream: autograd runs each backward node on the stream of its forward
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eager_d, eager_g = step()
        eager_d, eager_g = [t.clone() for t in eager_d], [t.clone() for t in eager_g]
        for _ in range(2):
            step()
    side.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        static_d, static_g = step()
    torch.cuda.current_stream().wait_stream(side)
    for t in static_d + static_g:
        t.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(static_d + static_g, eager_d + eager_g):
        assert_bitwise(a, b, "graph replay")
