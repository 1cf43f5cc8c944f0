"""Edge shapes and branches of the per-layer kernels (md2_ops.cu, md2_head.cu, md2_monitor.cu, md2::pose_to_matrix)
against the same operation in float64 on the CPU.

Every comparison follows protocol P3 (SURVEY.md 8c) element by element:
    |kernel - fp64| <= 1.5 |fp32 reference - fp64| + floor,
where the fp32 reference is the same oracle / torch function run in float32 on the CPU and the floor is
rel * |fp64| + abs.  The inputs are built so that fp32 and fp64 take the same discrete decisions (dyadic grid
coordinates, exact zero angles, depths away from the 1.25^k thresholds, image differences whose sign is exact), so
no gradient here can flip a bilinear cell, a clamp or a sign, and every gradient is checked per element.  Each floor
says where it comes from.

Branches that layers.py never takes (one output or one incoming gradient NULL) are driven through the C ABI with
ctypes.  The CPU-only checks at the end show that the discriminating inputs discriminate."""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import view_synthesis as O

DEV = "cuda:0"
gpu = pytest.mark.gpu
F32_ULP = 2.0 ** -23


def _lib():
    from monodepth2_b200 import _capi
    return _capi.load_library()


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _d(t):
    return torch.as_tensor(t).detach().to("cpu", torch.float64)


def p3(what, got, r32, r64, rel=0.0, abs_=0.0):
    """P3 per element: |got - r64| <= 1.5 |r32 - r64| + rel |r64| + abs_."""
    got, r32, r64 = _d(got), _d(r32), _d(r64)
    assert got.shape == r64.shape, (what, tuple(got.shape), tuple(r64.shape))
    assert bool(torch.isfinite(got).all()), (what, "non-finite kernel output")
    err, own = (got - r64).abs(), (r32 - r64).abs()
    bound = 1.5 * own + rel * r64.abs() + abs_
    bad = err > bound
    if bool(bad.any()):
        i = int(torch.argmax(err - bound))
        raise AssertionError("%s: %d of %d elements over the P3 bound; worst at flat index %d: kernel %r fp64 %r "
                             "(error %.3e, fp32 reference error %.3e, floor %.3e)"
                             % (what, int(bad.sum()), bad.numel(), i, float(got.flatten()[i]), float(r64.flatten()[i]),
                                float(err.flatten()[i]), float(own.flatten()[i]),
                                float((rel * r64.abs() + abs_).flatten()[i])))


def _leaf(t, dtype, requires_grad=True):
    return t.detach().to(dtype, copy=True).requires_grad_(requires_grad)


def _amax(t):
    return float(_d(t).abs().max())


# ------------------------------------------------------------------ SSIM (k_ssim / k_ssim_bwd)
# H or W = 2 or 3: the reflection multiplicity of k_ssim_bwd gets both end rules on one row / column
SSIM_SHAPES = [(1, 1, 2, 2), (2, 3, 3, 3), (1, 2, 2, 7), (1, 1, 3, 9), (2, 1, 6, 2), (1, 3, 7, 3), (1, 2, 4, 5)]


def _ssim_inputs(shape):
    g = torch.Generator().manual_seed(sum(shape) * 7 + shape[2])
    x = torch.rand(shape, generator=g)
    y = 0.6 * x + 0.4 * torch.rand(shape, generator=g)
    up = torch.randn(shape, generator=g)
    return x, y, up


def _ssim_ref(x, y, up, dtype, grads="xy"):
    a, b = _leaf(x, dtype, "x" in grads), _leaf(y, dtype, "y" in grads)
    s = O.ssim_dissimilarity(a, b)
    s.backward(up.to(dtype))
    return s.detach(), a.grad, b.grad


def ssim_conditioning(x, y):
    """Per output pixel, how much the kernel's one-pass window statistics amplify one ulp of their inputs.  ssim_at
    (md2_ops.cu) works on 9-pixel sums: n2 = 2 (9 Sxy - Sx Sy) + C2 and d2 = 9 (Sxx + Syy) - Sx^2 - Sy^2 + C2
    cancel terms of size 18 |Sxy| + 2 |Sx Sy| and 9 (Sxx + Syy) + Sx^2 + Sy^2, so Q = n1 n2 / (d1 d2) and the output
    (1 - Q) / 2 carry kappa = |Q| / 2 (those sizes / |n2| and / d2) ulp (computed in fp64)."""
    xp, yp = (F.pad(t.double(), (1, 1, 1, 1), mode="reflect") for t in (x, y))
    S = lambda t: 9 * F.avg_pool2d(t, 3, 1)                                        # noqa: E731
    sx, sy, sxx, syy, sxy = S(xp), S(yp), S(xp * xp), S(yp * yp), S(xp * yp)
    pxy, pp = sx * sy, sx * sx + sy * sy
    c1, c2 = 81 * 0.01 ** 2, 81 * 0.03 ** 2
    n1, n2 = 2 * pxy + c1, 2 * (9 * sxy - pxy) + c2
    d1, d2 = pp + c1, 9 * (sxx + syy) - pp + c2
    q = n1 * n2 / (d1 * d2)
    return 0.5 * q.abs() * ((18 * sxy.abs() + 2 * pxy.abs()) / n2.abs() + (9 * (sxx + syy) + pp) / d2)


def ssim_grad_floor(x, y, up, wrt):
    """32 ulp x sum over the windows q that reach pixel j of kappa_q |up_q d s_q / d wrt_j|: each window's share of
    the gradient carries that window's conditioning (fp64 Jacobian; the planes here have at most 126 pixels).  The
    derivative coefficients of ssim_at cancel once more (n2 - n1, d2 - d1, a + b x_j + c y_j): k_ssim_bwd's float32
    arithmetic restated on the CPU reaches 18 such ulp on these shapes (four seeds each), hence 32."""
    xd, yd = x.double(), y.double()
    fn = (lambda t: O.ssim_dissimilarity(t, yd)) if wrt == "x" else (lambda t: O.ssim_dissimilarity(xd, t))
    J = torch.autograd.functional.jacobian(fn, xd if wrt == "x" else yd).reshape(x.numel(), x.numel())
    w = (ssim_conditioning(x, y) * up.double().abs()).reshape(1, -1)
    return 32 * F32_ULP * (w @ J.abs()).reshape(x.shape)


@gpu
@pytest.mark.parametrize("grads", ["xy", "x", "y"])
@pytest.mark.parametrize("shape", SSIM_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_ssim_small_planes_match_fp64(shape, grads):
    """grad_x alone / grad_y alone is what SSIM(pred, target) asks for when only one side needs a gradient."""
    from monodepth2_b200 import layers as L
    x, y, up = _ssim_inputs(shape)
    s32, gx32, gy32 = _ssim_ref(x, y, up, torch.float32, grads)
    s64, gx64, gy64 = _ssim_ref(x, y, up, torch.float64, grads)
    a = x.to(DEV).requires_grad_("x" in grads)
    b = y.to(DEV).requires_grad_("y" in grads)
    s = L.SSIM()(a, b)
    s.backward(up.to(DEV))
    # forward floor: 4 ulp x the conditioning of the one-pass statistics, per pixel (ssim_conditioning).  ssim_at's
    # float32 arithmetic restated on the CPU stays within 0.84 kappa ulp on every shape here; the oracle's
    # two-pass avg_pool form is better conditioned, so its own fp32 error can be far smaller on a pixel
    p3("ssim forward", s, s32, s64, abs_=4 * F32_ULP * ssim_conditioning(x, y))
    for want, got, r32, r64, name in (("x", a.grad, gx32, gx64, "grad_x"), ("y", b.grad, gy32, gy64, "grad_y")):
        if want in grads:
            p3("ssim " + name, got, r32, r64, abs_=ssim_grad_floor(x, y, up, want))
        else:
            assert got is None


# ------------------------------------------------------------------ disparity head (md2_head.cu)
def _head_inputs(B, Cc, H, W, bias=None, seed=0):
    g = torch.Generator().manual_seed(seed + 31 * Cc + H)
    k = 1.0 / math.sqrt(9 * Cc)                              # nn.Conv2d's default init range
    x = torch.randn(B, Cc, H, W, generator=g)
    w = (2 * torch.rand(1, Cc, 3, 3, generator=g) - 1) * k
    b = (2 * torch.rand(1, generator=g) - 1) * k
    if bias is not None:                                    # saturated head: pre-activation bias +- O(1)
        x = 0.3 * x
        b = torch.full((1,), float(bias))
    up = torch.randn(B, 1, H, W, generator=g)
    return x, w, b, up


def _head_ref(x, w, b, up, dtype, need):
    xr, wr, br = (_leaf(t, dtype, n) for t, n in zip((x, w, b), need))
    y = torch.sigmoid(F.conv2d(F.pad(xr, (1, 1, 1, 1), mode="reflect"), wr, br))
    y.backward(up.to(dtype))
    return y.detach(), xr.grad, wr.grad, br.grad


HEAD_CASES = [
    # B, C, H, W, bias (None: random), : H or W = 3 puts y == 1 and y == H-2 on one pixel; C not a multiple of 16
    (2, 1, 3, 3, None), (1, 3, 3, 5, None), (2, 17, 4, 3, None), (1, 17, 2, 3, None), (3, 5, 2, 2, None),
    (1, 1365, 3, 4, None),                     # the largest C whose 9 C weights fit the 48 KB of shared memory
    (2, 3, 6, 7, -20.0),                       # pre-activation in [-25, -15]: sigmoid through __expf, saturated
]
NEEDS = {"all": (True, True, True), "frozen_head": (True, False, False), "input_frozen": (False, True, True),
         "bias_only": (False, False, True)}


@gpu
@pytest.mark.parametrize("need", list(NEEDS))
@pytest.mark.parametrize("B,Cc,H,W,bias", HEAD_CASES, ids=lambda v: "n" if v is None else str(v))
def test_disparity_head_edges_match_fp64(B, Cc, H, W, bias, need):
    from monodepth2_b200 import layers as L
    x, w, b, up = _head_inputs(B, Cc, H, W, bias)
    nx, nw, nb = NEEDS[need]
    y32, gx32, gw32, gb32 = _head_ref(x, w, b, up, torch.float32, NEEDS[need])
    y64, gx64, gw64, gb64 = _head_ref(x, w, b, up, torch.float64, NEEDS[need])
    head = L.DispConvSigmoid(Cc).to(DEV)
    with torch.no_grad():
        head.conv.weight.copy_(w)
        head.conv.bias.copy_(b)
    head.conv.weight.requires_grad_(nw)
    head.conv.bias.requires_grad_(nb)
    xd = x.to(DEV).requires_grad_(nx)
    y = head(xd)
    y.backward(up.to(DEV))
    # forward floor: __expf is within 2 + 1.173 |x| ulp (CUDA C Programming Guide, intrinsic functions), 31 ulp =
    # 3.7e-6 relative at |x| = 25; plus 1e-6 absolute for the C*9-term dot product summed in another order
    p3("head forward", y, y32, y64, rel=32 * F32_ULP, abs_=1e-6)
    # gradients: the same __expf error (relative, per term) and re-ordered sums, against the largest element
    for n, got, r32, r64, name in ((nx, xd.grad, gx32, gx64, "grad_x"), (nw, head.conv.weight.grad, gw32, gw64, "grad_w"),
                                   (nb, head.conv.bias.grad, gb32, gb64, "grad_b")):
        if n:
            p3("head " + name, got, r32, r64, rel=32 * F32_ULP, abs_=1e-5 * _amax(r64))
        else:
            assert got is None, name


@gpu
def test_disparity_head_rejects_channels_beyond_shared_memory():
    """C = 1366 needs 49176 bytes of weights: both entry points refuse it before any launch."""
    from monodepth2_b200 import layers as L
    B, Cc, H, W = 1, 1366, 3, 4
    x = torch.randn(B, Cc, H, W, device=DEV)
    with pytest.raises(RuntimeError, match="unsupported"):
        L.DispConvSigmoid(Cc).to(DEV)(x)
    lib = _lib()
    w = torch.zeros(1, Cc, 3, 3, device=DEV)
    disp, g = torch.full((B, 1, H, W), 0.5, device=DEV), torch.ones(B, 1, H, W, device=DEV)
    gx, gw, gb = torch.empty_like(x), torch.empty_like(w), torch.empty(1, device=DEV)
    st = lib.md2_dispconv_sigmoid_backward(_p(g), _p(disp), _p(x), _p(w), _p(gx), _p(gw), _p(gb), B, Cc, H, W,
                                           _stream())
    assert st == -2                                               # MD2_ERR_UNSUPPORTED


# ------------------------------------------------------------------ Project3D (k_project3d / k_project3d_bwd)
def _project_full_inputs(B=2, H=192, W=640):
    g = torch.Generator().manual_seed(5)
    K = torch.tensor([[0.58 * W, 0, 0.5 * W, 0], [0, 1.92 * H, 0.5 * H, 0], [0, 0, 1, 0], [0, 0, 0, 1]]).expand(B, 4, 4)
    depth = 1.0 + 30.0 * torch.rand(B, 1, H, W, generator=g)
    pts = O.backproject(depth, torch.linalg.inv(K)).contiguous()
    T = O.transformation_from_parameters(0.02 * torch.randn(B, 1, 3, generator=g),
                                         0.1 * torch.randn(B, 1, 3, generator=g)).contiguous()
    up = torch.randn(B, H, W, 2, generator=g)
    return pts, K.contiguous(), T, up


def _project_near_plane_inputs(B, H, W):
    """Depths on and behind the camera plane with a camera row that makes the depth coordinate exact in fp32:
    K's last rows are [0 0 1 0], [0 0 0 1] and T only translates in x and y by dyadic steps, so c2 = Z."""
    g = torch.Generator().manual_seed(H * 13 + W)
    n = H * W
    X = torch.randint(-64, 65, (B, 1, n), generator=g) / 16.0
    Y = torch.randint(-64, 65, (B, 1, n), generator=g) / 16.0
    choices = torch.tensor([2.0 ** -10, -(2.0 ** -10), 2.0 ** -7, -0.5, 1.0, 1.5, 2.25, 3.0, -4.0])
    Z = choices[torch.randint(0, len(choices), (B, 1, n), generator=g)]
    pts = torch.cat([X, Y, Z, torch.ones(B, 1, n)], 1).contiguous()
    K = torch.tensor([[8.0, 0, 4.0, 0], [0, 8.0, 2.0, 0], [0, 0, 1, 0], [0, 0, 0, 1]]).expand(B, 4, 4).contiguous()
    T = torch.eye(4).repeat(B, 1, 1)
    T[:, 0, 3], T[:, 1, 3] = 0.25, -0.125
    up = torch.randn(B, H, W, 2, generator=g)
    return pts, K, T, up


def _project_ref(pts, K, T, up, H, W, dtype):
    p, t = _leaf(pts, dtype), _leaf(T, dtype)
    grid = O.project(p, K.to(dtype), t, H, W)
    grid.backward(up.to(dtype))
    return grid.detach(), p.grad, t.grad


def _project_check(pts, K, T, up, H, W, tag, grid_abs, gp_abs, gT_rel):
    from monodepth2_b200 import layers as L
    B = pts.shape[0]
    g32, gp32, gT32 = _project_ref(pts, K, T, up, H, W, torch.float32)
    g64, gp64, gT64 = _project_ref(pts, K, T, up, H, W, torch.float64)
    p = pts.to(DEV).requires_grad_(True)
    t = T.to(DEV).requires_grad_(True)
    grid = L.Project3D(B, H, W)(p, K.to(DEV), t)
    grid.backward(up.to(DEV))
    p3(tag + " grid", grid, g32, g64, rel=4 * F32_ULP, abs_=grid_abs)
    p3(tag + " grad_points", p.grad, gp32, gp64, rel=4 * F32_ULP, abs_=gp_abs * _amax(gp64))
    p3(tag + " grad_T", t.grad, gT32, gT64, abs_=gT_rel * _amax(gT64))


@gpu
def test_project3d_full_size_grad_T_matches_fp64():
    """192 x 640: 480 blocks per sample reduce grad_T with a block sum and one float atomic each."""
    pts, K, T, up = _project_full_inputs()
    # floors: the grid carries ~1 ulp of |u| <= ~1e3 pixels (normalised: 1e-6 absolute); grad_T sums 122880
    # products per entry in float blocks and float atomics, ~sqrt(480) ulp of the largest entry
    _project_check(pts, K, T, up, 192, 640, "full size", grid_abs=1e-6, gp_abs=1e-6, gT_rel=1e-5)


@gpu
@pytest.mark.parametrize("B,H,W", [(2, 2, 5), (1, 8, 2), (2, 16, 24)])
def test_project3d_near_and_behind_camera_plane_match_fp64(B, H, W):
    pts, K, T, up = _project_near_plane_inputs(B, H, W)
    # Z = 2^-10 puts |u| near 1e4 and |d grid / d Z| near 1e11: the relative floor of a few ulp carries that; the
    # grid's "- 0.5" cancels for points near the image centre: 8 ulp of 1 absolute; the gradient floors are 1e-6 of
    # each tensor's largest element (re-ordered 4-term dot products)
    _project_check(pts, K, T, up, H, W, "near plane %dx%d" % (H, W), grid_abs=8 * F32_ULP, gp_abs=1e-6, gT_rel=1e-6)


@gpu
def test_project3d_backward_single_output_branches():
    """md2_project3d_backward with only grad_points or only grad_T: each equals that output of the full call
    (one block per sample, so the grad_T reduction order is the same)."""
    B, H, W = 2, 8, 16
    pts, K, T, up = (t.to(DEV) for t in _project_near_plane_inputs(B, H, W))
    lib = _lib()

    def run(want_p, want_T):
        gp = torch.full_like(pts, float("nan")) if want_p else None
        gT = torch.full_like(T, float("nan")) if want_T else None
        st = lib.md2_project3d_backward(_p(up), _p(pts), _p(K), _p(T), C.c_float(1e-7), _p(gp), _p(gT), B, H, W,
                                        _stream())
        assert st == 0
        return gp, gT
    gp, gT = run(True, True)
    gp_only, _ = run(True, False)
    _, gT_only = run(False, True)
    torch.cuda.synchronize()
    assert torch.equal(gp_only, gp) and torch.equal(gT_only, gT)
    _, gp64, gT64 = _project_ref(pts.cpu(), K.cpu(), T.cpu(), up.cpu(), H, W, torch.float64)
    _, gp32, gT32 = _project_ref(pts.cpu(), K.cpu(), T.cpu(), up.cpu(), H, W, torch.float32)
    p3("grad_points only", gp_only, gp32, gp64, rel=4 * F32_ULP, abs_=1e-6 * _amax(gp64))
    p3("grad_T only", gT_only, gT32, gT64, abs_=1e-6 * _amax(gT64))


# ------------------------------------------------------------------ grid_sample, border padding
def lattice(n, align_corners):
    """Normalised coordinates of the texel centres 0 .. n-1 (exact in fp32 when n, or n-1 with align_corners, is a
    power of two)."""
    u = torch.arange(n, dtype=torch.float64)
    if align_corners:
        return 2 * u / (n - 1) - 1 if n > 1 else torch.zeros(1, dtype=torch.float64)
    return (2 * u + 1) / n - 1


def unnormalize(g, n, align_corners):
    """The kernel's (and torch's) map from a normalised coordinate to texel units, in g's dtype."""
    return (g + 1) * 0.5 * (n - 1) if align_corners else ((g + 1) * n - 1) * 0.5


GS_CASES = [
    # B, C, IH, IW, OH, OW, align_corners: sizes (IW, or IW-1 with align_corners) powers of two for the lattice
    (2, 3, 4, 8, 4, 8, False), (1, 5, 5, 9, 3, 7, True), (2, 1, 1, 8, 2, 6, False), (1, 2, 5, 1, 5, 3, True),
    (1, 4, 1, 1, 2, 2, False), (2, 3, 8, 16, 11, 13, False), (1, 6, 9, 17, 16, 8, True),
]


def _gs_inputs(B, Cc, IH, IW, OH, OW, ac):
    """Grid = both borders exactly, then texel centres, half-texels and random multiples of 1/64 in [-1.25, 1.25]:
    every coordinate and every bilinear weight is exact in fp32, so fp32 and fp64 take the same cells and clamps."""
    g = torch.Generator().manual_seed(IH * 100 + IW * 10 + OW)
    img = torch.rand(B, Cc, IH, IW, generator=g)

    def axis(n):
        lat = lattice(n, ac)
        half = (lat[:-1] + lat[1:]) / 2
        dy = torch.randint(-80, 81, (64,), generator=g).double() / 64
        return torch.cat([lat[:1], lat[-1:], lat, half, dy]).float()
    ax, ay = axis(IW), axis(IH)
    n = OH * OW
    gx = ax[torch.randint(0, len(ax), (B, n), generator=g)]
    gy = ay[torch.randint(0, len(ay), (B, n), generator=g)]
    k = min(n, 4)                                   # the four border combinations come first in every sample
    gx[:, :k] = torch.tensor([ax[0], ax[1], ax[0], ax[1]])[:k]
    gy[:, :k] = torch.tensor([ay[0], ay[0], ay[1], ay[1]])[:k]
    grid = torch.stack([gx, gy], -1).reshape(B, OH, OW, 2).contiguous()
    up = torch.randn(B, Cc, OH, OW, generator=g)
    return img, grid, up


def _gs_ref(img, grid, up, ac, dtype):
    gr = _leaf(grid, dtype)
    out = F.grid_sample(img.to(dtype), gr, mode="bilinear", padding_mode="border", align_corners=ac)
    out.backward(up.to(dtype))
    return out.detach(), gr.grad


@gpu
@pytest.mark.parametrize("B,Cc,IH,IW,OH,OW,ac", GS_CASES, ids=lambda v: str(v))
def test_grid_sample_border_lattice_and_edges_match_fp64(B, Cc, IH, IW, OH, OW, ac):
    """The clamp-gradient mask is 0 exactly on the border (torch treats ux == 0 and ux == IW-1 as outside)."""
    from monodepth2_b200 import layers as L
    img, grid, up = _gs_inputs(B, Cc, IH, IW, OH, OW, ac)
    o32, gg32 = _gs_ref(img, grid, up, ac, torch.float32)
    o64, gg64 = _gs_ref(img, grid, up, ac, torch.float64)
    gd = grid.to(DEV).requires_grad_(True)
    out = L.grid_sample_border(img.to(DEV), gd, align_corners=ac)
    out.backward(up.to(DEV))
    # floors: a bilinear blend of values in [0, 1] with exact weights: a couple of ulp of 1; the grid gradient sums
    # C products of such differences with the upstream gradient: a few ulp of the largest element
    p3("grid_sample forward", out, o32, o64, abs_=4 * F32_ULP)
    p3("grid_sample grad_grid", gd.grad, gg32, gg64, abs_=4 * F32_ULP * Cc * _amax(gg64))
    on_border = torch.zeros(grid.shape, dtype=torch.bool)
    for j, n in ((0, IW), (1, IH)):
        u = unnormalize(grid[..., j].double(), n, ac)
        on_border[..., j] = (u == 0) | (u == n - 1)
    assert bool((gd.grad.cpu()[on_border] == 0).all())


# ------------------------------------------------------------------ get_smooth_loss (k_smooth_*)
SMOOTH_CASES = [
    # B, C, H, W, levels (0: continuous disparity; n: n levels, so many neighbours are equal and their sign is 0)
    (2, 1, 5, 7, 0), (1, 3, 2, 9, 0), (2, 2, 6, 2, 4), (1, 1, 2, 2, 2), (3, 3, 16, 24, 3), (12, 3, 192, 640, 0),
]


def _smooth_inputs(B, Cc, H, W, levels):
    g = torch.Generator().manual_seed(B * 1000 + H + W + levels)
    d = torch.rand(B, 1, H, W, generator=g)
    if levels:
        d = torch.floor(d * levels) / levels
    img = torch.rand(B, Cc, H, W, generator=g)
    return d, img


def _smooth_ref(d, img, dtype):
    dr = _leaf(d, dtype)
    loss = O.smooth_loss(dr, img.to(dtype))
    (3.0 * loss).backward()
    return loss.detach(), dr.grad


@gpu
@pytest.mark.parametrize("B,Cc,H,W,levels", SMOOTH_CASES, ids=lambda v: str(v))
def test_smooth_loss_edges_match_fp64(B, Cc, H, W, levels):
    from monodepth2_b200 import layers as L
    d, img = _smooth_inputs(B, Cc, H, W, levels)
    l32, g32 = _smooth_ref(d, img, torch.float32)
    l64, g64 = _smooth_ref(d, img, torch.float64)
    dd = d.to(DEV).requires_grad_(True)
    loss = L.get_smooth_loss(dd, img.to(DEV))
    (3.0 * loss).backward()
    # floors: the loss is a mean of positive terms, summed in float per block and in double across blocks: a few ulp
    # relative; each gradient element is 4 signed, weighted terms of one size (1 / element count): a few ulp of it
    p3("smooth loss", loss, l32, l64, rel=8 * F32_ULP)
    p3("smooth grad", dd.grad, g32, g64, abs_=8 * F32_ULP * _amax(g64))
    if levels:                                          # equal neighbours, where the sign (and its gradient) is 0
        assert bool((d[..., 1:] == d[..., :-1]).any()) and bool((d[..., 1:, :] == d[..., :-1, :]).any())


# ------------------------------------------------------------------ pose (md2::pose_to_matrix and its backward)
def _pose_batch(B=300):
    """300 samples (two blocks of 256 threads): zero angles in both blocks, tiny angles, angles at and near pi, and
    0.3 randn elsewhere."""
    g = torch.Generator().manual_seed(11)
    aa = 0.3 * torch.randn(B, 1, 3, generator=g)
    u = torch.randn(B, 1, 3, generator=g)
    u = u / u.norm(dim=2, keepdim=True)
    special = [0.0, 0.0, 1e-8, 3e-8, 1e-7, 1e-6, 1e-5, math.pi - 1e-3, math.pi - 1e-6, math.pi]
    for i, m in enumerate(special):
        aa[i] = m * u[i]
    aa[280:284] = 0.0
    tr = torch.randn(B, 1, 3, generator=g)
    up = torch.randn(B, 4, 4, generator=g)
    return aa, tr, up


def _pose_ref(fn, args, up, dtype):
    a = [_leaf(t, dtype) for t in args]
    T = fn(*a)
    T.backward(up.to(dtype))
    return (T.detach(),) + tuple(t.grad for t in a)


@gpu
@pytest.mark.parametrize("invert", [False, True])
def test_transformation_from_parameters_edges_match_fp64(invert):
    from monodepth2_b200 import layers as L
    aa, tr, up = _pose_batch()
    fn = lambda a, t: O.transformation_from_parameters(a, t, invert)       # noqa: E731
    T32, ga32, gt32 = _pose_ref(fn, (aa, tr), up, torch.float32)
    T64, ga64, gt64 = _pose_ref(fn, (aa, tr), up, torch.float64)
    a, t = aa.to(DEV).requires_grad_(True), tr.to(DEV).requires_grad_(True)
    T = L.transformation_from_parameters(a, t, invert)
    T.backward(up.to(DEV))
    # floors: entries of R are O(1) and the translation column O(|t|): a few ulp of the batch's largest entry;
    # the angle gradient divides by (angle + 1e-7): a few ulp relative to the element, plus 1e-6 of the largest
    p3("pose T", T, T32, T64, abs_=8 * F32_ULP * _amax(T64))
    p3("pose grad_axisangle", a.grad, ga32, ga64, rel=8 * F32_ULP, abs_=1e-6 * _amax(ga64))
    p3("pose grad_translation", t.grad, gt32, gt64, rel=8 * F32_ULP, abs_=1e-6 * _amax(gt64))
    assert bool((a.grad[:2] == 0).all()) and bool((a.grad[280:284] == 0).all())   # zero angle: exactly 0 (torch.norm)


@gpu
def test_get_translation_matrix_and_rot_from_axisangle_backward_match_fp64():
    """Both run the pose kernel with the other leaf at zero; get_translation_matrix always at the zero angle."""
    from monodepth2_b200 import layers as L
    aa, tr, up = _pose_batch()
    _, gt64 = _pose_ref(O.translation_matrix, (tr,), up, torch.float64)
    _, gt32 = _pose_ref(O.translation_matrix, (tr,), up, torch.float32)
    t = tr.to(DEV).requires_grad_(True)
    L.get_translation_matrix(t).backward(up.to(DEV))
    p3("get_translation_matrix grad", t.grad, gt32, gt64)                       # a copy of up[:, :3, 3]: exact
    R32, gv32 = _pose_ref(O.rot_from_axisangle, (aa,), up, torch.float32)
    R64, gv64 = _pose_ref(O.rot_from_axisangle, (aa,), up, torch.float64)
    v = aa.to(DEV).requires_grad_(True)
    R = L.rot_from_axisangle(v)
    R.backward(up.to(DEV))
    p3("rot_from_axisangle", R, R32, R64, abs_=8 * F32_ULP)
    p3("rot_from_axisangle grad", v.grad, gv32, gv64, rel=8 * F32_ULP, abs_=1e-6 * _amax(gv64))


# ------------------------------------------------------------------ disp_to_depth, one output / one gradient NULL
@gpu
def test_disp_to_depth_single_output_branches_match_fp64():
    lib = _lib()
    n, lo, hi = 1003, 0.1, 100.0
    g = torch.Generator().manual_seed(21)
    d, gs, gd = torch.rand(n, generator=g), torch.randn(n, generator=g), torch.randn(n, generator=g)
    dd, gsd, gdd = d.to(DEV), gs.to(DEV), gd.to(DEV)

    def fwd(want_s, want_d):
        s = torch.full_like(dd, float("nan")) if want_s else None
        z = torch.full_like(dd, float("nan")) if want_d else None
        assert lib.md2_disp_to_depth(_p(dd), C.c_float(lo), C.c_float(hi), _p(s), _p(z), C.c_longlong(n), _stream()) == 0
        return s, z

    def bwd(g_s, g_d):
        out = torch.full_like(dd, float("nan"))
        assert lib.md2_disp_to_depth_backward(_p(dd), C.c_float(lo), C.c_float(hi), _p(g_s), _p(g_d), _p(out),
                                              C.c_longlong(n), _stream()) == 0
        return out
    s, z = fwd(True, True)
    s_only, _ = fwd(True, False)
    _, z_only = fwd(False, True)
    gb, gb_s, gb_d = bwd(gsd, gdd), bwd(gsd, None), bwd(None, gdd)
    torch.cuda.synchronize()
    assert torch.equal(s_only, s) and torch.equal(z_only, z)

    def ref(dtype, use_s, use_d):
        x = _leaf(d, dtype)
        rs, rz = O.disp_to_depth(x, lo, hi)
        ((rs * gs.to(dtype)).sum() * use_s + (rz * gd.to(dtype)).sum() * use_d).backward()
        return rs.detach(), rz.detach(), x.grad
    s32, z32, _ = ref(torch.float32, 1, 1)
    s64, z64, _ = ref(torch.float64, 1, 1)
    # floors: one affine map and one reciprocal, each rounded once: 2 ulp relative
    p3("scaled_disp only", s_only, s32, s64, rel=2 * F32_ULP)
    p3("depth only", z_only, z32, z64, rel=2 * F32_ULP)
    for got, us, ud, name in ((gb, 1, 1, "both"), (gb_s, 1, 0, "grad_scaled only"), (gb_d, 0, 1, "grad_depth only")):
        # the two incoming gradients meet in one sum: 4 ulp of the larger term
        p3("disp_to_depth backward " + name, got, ref(torch.float32, us, ud)[2], ref(torch.float64, us, ud)[2],
           rel=4 * F32_ULP, abs_=4 * F32_ULP * _amax(ref(torch.float64, us, ud)[2]))


# ------------------------------------------------------------------ md2_scale_tensors (autograd glue of the fused call)
@gpu
@pytest.mark.parametrize("sizes", [[0, 1, 3, 5, 1023, 4097],
                                   [4, 0, 7, 8, 9, 1, 2, 1024, 1025, 4095, 4096, 4097, 0, 3, 5, 6]],
                         ids=["mixed", "sixteen"])
def test_scale_tensors_is_bitwise_src_times_scale(sizes):
    """Every size not a multiple of 4, zero-size entries and the 16-tensor maximum; nothing is written past numel."""
    lib = _lib()
    g = torch.Generator(device=DEV).manual_seed(len(sizes))
    pad = 8
    srcs = [torch.randn(n + pad, device=DEV, generator=g) for n in sizes]    # zero-size entries still point somewhere
    dsts = [torch.full((n + pad,), float("nan"), device=DEV) for n in sizes]
    scale = torch.tensor([-0.7071067811865476], device=DEV)
    k = len(sizes)
    rc = lib.md2_scale_tensors(k, (C.c_void_p * k)(*[s.data_ptr() for s in srcs]),
                               (C.c_void_p * k)(*[d.data_ptr() for d in dsts]), (C.c_longlong * k)(*sizes),
                               C.c_void_p(scale.data_ptr()), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    for n, s, d in zip(sizes, srcs, dsts):
        want = s[:n] * scale
        assert torch.equal(d[:n].view(torch.int32), want.view(torch.int32)), n
        assert bool(torch.isnan(d[n:]).all()), n


@gpu
def test_scale_tensors_rejects_seventeen():
    lib = _lib()
    bufs = [torch.zeros(4, device=DEV) for _ in range(17)]
    ptrs = (C.c_void_p * 17)(*[b.data_ptr() for b in bufs])
    scale = torch.ones(1, device=DEV)
    assert lib.md2_scale_tensors(17, ptrs, ptrs, (C.c_longlong * 17)(*([4] * 17)), C.c_void_p(scale.data_ptr()),
                                 _stream()) == -1                          # MD2_ERR_INVALID_ARGUMENT


# ------------------------------------------------------------------ depth metrics (md2_monitor.cu)
def split_median_case():
    """Even N, two clusters each in gt and in the prediction: the lower median (rank (N-1)/2) sits in the low
    clusters and the upper one (rank N/2) in the high ones: the median-scaling ratio is ~1 with the one and ~0.6 with
    the other, and every one of the seven metrics moves."""
    g = torch.Generator().manual_seed(41)
    B, H, W = 2, 16, 32
    n = B * H * W
    low = torch.randperm(n, generator=g)[: n // 2]
    gt = 7 + 3 * torch.rand(n, generator=g)
    gt[low] = 4 + 2 * torch.rand(n // 2, generator=g)
    low_p = torch.randperm(n, generator=g)[: n // 2]
    pred = 12 + 3 * torch.rand(n, generator=g)
    pred[low_p] = 5 + torch.rand(n // 2, generator=g)
    return pred.reshape(B, 1, H, W), gt.reshape(B, 1, H, W), (0, H, 0, W)


def metrics_case(name):
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    if name == "split_median":
        return split_median_case()
    if name == "ties":
        depth = torch.tensor([3.0, 6.0, 12.0])[torch.randint(0, 3, (2, 1, 24, 40), generator=g)]
        gt = torch.tensor([0.0, 4.0, 8.0, 16.0, 32.0])[torch.randint(0, 5, (2, 1, 24, 40), generator=g)]
        return depth, gt, (2, 22, 3, 37)
    if name in ("n_one", "n_zero"):
        depth = 1 + 20 * torch.rand(1, 1, 12, 20, generator=g)
        gt = 1 + 40 * torch.rand(1, 1, 12, 20, generator=g)
        gt[:, :, 2:10, 3:17] = 0
        if name == "n_one":
            gt[0, 0, 5, 9] = 7.5
        return depth, gt, (2, 10, 3, 17)
    if name == "downsample":
        return 0.5 + 40 * torch.rand(2, 1, 96, 320, generator=g), 0.5 + 60 * torch.rand(2, 1, 48, 160, generator=g), \
            (5, 40, 10, 150)
    if name == "crop_past_gt":
        gt = 0.5 + 60 * torch.rand(3, 1, 37, 123, generator=g)
        gt[torch.rand(gt.shape, generator=g) < 0.3] = 0
        return 0.5 + 40 * torch.rand(3, 1, 24, 80, generator=g), gt, (20, 375, 50, 1242)
    if name == "clamped":
        depth = 0.5 + 40 * torch.rand(2, 1, 24, 80, generator=g)
        r = torch.rand(depth.shape, generator=g)
        depth[r < 0.25] = 200.0                                   # clamped to 80 before and after median scaling
        depth[r > 0.8] = 1e-4                                     # clamped to 1e-3
        return depth, 0.5 + 60 * torch.rand(2, 1, 48, 160, generator=g), (0, 48, 0, 160)
    raise KeyError(name)


METRIC_CASES = ["split_median", "ties", "n_one", "n_zero", "downsample", "crop_past_gt", "clamped"]


def threshold_margin(depth, gt, crop):
    """Smallest distance, in log units, of a masked pixel's fp64 max(gt/pred, pred/gt) from 1.25, 1.25^2, 1.25^3."""
    Hg, Wg = gt.shape[-2:]
    pred = torch.clamp(F.interpolate(depth.double(), [Hg, Wg], mode="bilinear", align_corners=False), 1e-3, 80)
    mask = torch.zeros_like(gt, dtype=torch.bool)
    mask[:, :, crop[0]:crop[1], crop[2]:crop[3]] = True
    mask &= gt > 0
    g, p = gt.double()[mask], pred[mask]
    if g.numel() == 0:
        return math.inf
    p = torch.clamp(p * (g.median() / p.median()), 1e-3, 80)
    lt = torch.log(torch.max(g / p, p / g)) / math.log(1.25)
    return float((lt.unsqueeze(1) - torch.tensor([1.0, 2.0, 3.0], dtype=torch.float64)).abs().min())


@gpu
@pytest.mark.parametrize("name", METRIC_CASES)
def test_depth_metrics_edges_match_fp64(name):
    from monodepth2_b200 import layers as L
    depth, gt, crop = metrics_case(name)
    r32 = O.depth_metrics(depth, gt, crop)
    r64 = O.depth_metrics(depth.double(), gt.double(), crop)
    got = L.depth_metrics(depth.to(DEV), gt.to(DEV), crop).cpu()
    if name == "n_zero":                              # torch.median of nothing is nan, and so is every metric
        assert bool(torch.isnan(r64).all()) and bool(torch.isnan(got).all()), got
        return
    # floors: the kernel sums in double and rounds each metric to float once; the fp64 oracle rounds its result to
    # float32 too (O.depth_metrics): one ulp each, plus the fp32 ratio and log: 8 ulp relative
    p3("depth metrics " + name, got, r32, r64, rel=8 * F32_ULP, abs_=1e-7)


# ------------------------------------------------------------------ CPU self-checks of the discriminating inputs
def _metrics_with_rank(depth, gt, rank):
    """O.depth_metrics with the median taken at rank(N) of the sorted values (same-size gt and prediction only)."""
    mask = gt > 0
    g, p = gt.double()[mask], depth.double().clamp(1e-3, 80)[mask]
    r = rank(g.numel())
    p = torch.clamp(p * (g.sort().values[r] / p.sort().values[r]), 1e-3, 80)
    return torch.stack([torch.as_tensor(v, dtype=torch.float64) for v in O.compute_depth_errors(g, p)])


def test_split_median_case_separates_lower_and_upper_median():
    depth, gt, crop = split_median_case()
    assert crop == (0, gt.shape[2], 0, gt.shape[3]) and (gt > 0).sum() % 2 == 0
    lower = _metrics_with_rank(depth, gt, lambda n: (n - 1) // 2)
    upper = _metrics_with_rank(depth, gt, lambda n: n // 2)
    oracle = O.depth_metrics(depth.double(), gt.double(), crop).double()
    assert torch.allclose(lower, oracle, rtol=1e-6, atol=0)          # torch.median is the lower median
    tol = 8 * F32_ULP * lower.abs() + 1e-7                           # the GPU test's floor (its 1.5 x term is ~0)
    assert bool(((upper - lower).abs() > 100 * tol).all()), (lower, upper)


@pytest.mark.parametrize("name", METRIC_CASES)
def test_metric_cases_stay_away_from_the_delta_thresholds(name):
    depth, gt, crop = metrics_case(name)
    # 1e-5 in units of log(1.25) is 2e-6 relative: ~20 ulp of the fp32 ratio the kernel compares with 1.25^k
    assert threshold_margin(depth, gt, crop) > 1e-5


@pytest.mark.parametrize("B,Cc,IH,IW,OH,OW,ac", GS_CASES, ids=lambda v: str(v))
def test_grid_lattice_lands_on_both_borders_in_fp32_and_fp64(B, Cc, IH, IW, OH, OW, ac):
    _, grid, _ = _gs_inputs(B, Cc, IH, IW, OH, OW, ac)
    for j, n in ((0, IW), (1, IH)):
        for dtype in (torch.float32, torch.float64):
            u = unnormalize(grid[..., j].to(dtype), n, ac)
            assert bool((u == u.round()).any())
            assert bool((u == 0).any()) and bool((u == n - 1).any()), (j, dtype)
            lat = unnormalize(lattice(n, ac).to(dtype), n, ac)
            assert torch.equal(lat, torch.arange(n, dtype=dtype)) or (ac and n == 1)
        u32 = unnormalize(grid[..., j].float(), n, ac).double()
        assert torch.equal(u32, unnormalize(grid[..., j].double(), n, ac))   # every coordinate exact in fp32


def _own_error(r32, r64):
    e = float((_d(r32) - _d(r64)).abs().max())
    return math.isfinite(e) and e > 0


def test_fp32_references_carry_rounding_error_against_fp64():
    """The 1.5 x term of every P3 bound above is a real fp32 error (finite, non-zero), not a copy of fp64."""
    x, y, up = _ssim_inputs(SSIM_SHAPES[1])
    for a, b in zip(_ssim_ref(x, y, up, torch.float32), _ssim_ref(x, y, up, torch.float64)):
        assert _own_error(a, b)
    x, w, b, up = _head_inputs(*HEAD_CASES[-1][:4], HEAD_CASES[-1][4])
    for a, c in zip(_head_ref(x, w, b, up, torch.float32, (True,) * 3), _head_ref(x, w, b, up, torch.float64, (True,) * 3)):
        assert _own_error(a, c)
    pts, K, T, up = _project_near_plane_inputs(2, 2, 5)
    for a, c in zip(_project_ref(pts, K, T, up, 2, 5, torch.float32), _project_ref(pts, K, T, up, 2, 5, torch.float64)):
        assert _own_error(a, c)
    img, grid, up = _gs_inputs(*GS_CASES[0])
    for a, c in zip(_gs_ref(img, grid, up, False, torch.float32), _gs_ref(img, grid, up, False, torch.float64)):
        assert _own_error(a, c)
    d, img = _smooth_inputs(*SMOOTH_CASES[4])
    for a, c in zip(_smooth_ref(d, img, torch.float32), _smooth_ref(d, img, torch.float64)):
        assert _own_error(a, c)
    aa, tr, up = _pose_batch()
    fn = lambda a, t: O.transformation_from_parameters(a, t, True)       # noqa: E731
    for a, c in zip(_pose_ref(fn, (aa, tr), up, torch.float32), _pose_ref(fn, (aa, tr), up, torch.float64)):
        assert _own_error(a, c)
    depth, gt, crop = metrics_case("ties")
    assert _own_error(O.depth_metrics(depth, gt, crop), O.depth_metrics(depth.double(), gt.double(), crop))
