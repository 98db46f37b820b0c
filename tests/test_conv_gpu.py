"""Implicit-GEMM convolution (fwd / dgrad / wgrad) through the C ABI vs torch fp32 conv2d autograd on the same
bf16-rounded inputs.  Shapes are the ResNet-50 stage shapes of SURVEY.md App. A.1 at small batch."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# (N, H, W, Cin, Cout, R, stride, pad)
CASES = [
    (4, 56, 56, 64, 64, 3, 1, 1),
    (2, 28, 28, 128, 128, 3, 1, 1),
    (3, 14, 14, 256, 256, 3, 1, 1),
    (5, 7, 7, 512, 512, 3, 1, 1),
    (2, 56, 56, 128, 128, 3, 2, 1),
    (2, 28, 28, 256, 256, 3, 2, 1),
    (3, 14, 14, 512, 512, 3, 2, 1),
    (2, 56, 56, 256, 512, 1, 2, 0),
    (2, 56, 56, 64, 256, 1, 1, 0),
    (2, 14, 14, 1024, 256, 1, 1, 0),
    (1, 112, 112, 64, 64, 3, 1, 1),
    # enough 256-wide tiles for the CTA-pair path (gemm.cuh CG = 2): 3x3, 3x3 stride 2 and 1x1, odd number of pixel patches
    (19, 56, 56, 64, 256, 3, 1, 1),
    (25, 28, 28, 256, 256, 3, 1, 1),
    (100, 28, 28, 256, 256, 3, 2, 1),
    (21, 56, 56, 256, 512, 1, 1, 0),
]


def _mk(case, seed=0):
    N, H, W, Cin, Cout, R, stride, pad = case
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(N, H, W, Cin, device="cuda", generator=g).bfloat16()
    w = (torch.randn(Cout, R, R, Cin, device="cuda", generator=g) / (R * R * Cin) ** 0.5).bfloat16()
    return x, w


def _ref(x, w, stride, pad, dy=None):
    xr = x.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    wr = w.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    y = F.conv2d(xr, wr, stride=stride, padding=pad)
    if dy is None:
        return y.permute(0, 2, 3, 1).contiguous()
    y.backward(dy.float().permute(0, 3, 1, 2).contiguous())
    return xr.grad.permute(0, 2, 3, 1).contiguous(), wr.grad.permute(0, 2, 3, 1).contiguous()


def _check(got, ref, tag, rel=2e-2):
    d = (got.float() - ref).abs()
    tol = rel * ref.abs().max().item() + 1e-3
    nbad = int((d > tol).sum())
    info = ""
    if nbad:
        idx = (d > tol).nonzero()
        info = " first bad idx %s .. last %s" % (idx[0].tolist(), idx[-1].tolist())
    assert nbad == 0, "%s: max err %.4g tol %.4g bad %d/%d%s" % (tag, d.max().item(), tol, nbad, d.numel(), info)


@pytest.mark.parametrize("case", CASES)
def test_conv_fwd(case):
    from passl_b200 import kernels as K_
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    x, w = _mk(case)
    stride, pad = case[6], case[7]
    out = K_.conv2d_fwd(x, w, stride=stride, pad=pad)
    torch.cuda.synchronize()
    _check(out, _ref(x, w, stride, pad), "conv fwd %s" % (case,))


@pytest.mark.parametrize("case", CASES)
def test_conv_dgrad(case):
    from passl_b200 import kernels as K_
    torch.backends.cudnn.allow_tf32 = False
    x, w = _mk(case, 1)
    stride, pad = case[6], case[7]
    y = _ref(x, w, stride, pad)
    dy = torch.randn_like(y).bfloat16()
    dx_ref, _ = _ref(x, w, stride, pad, dy)
    dx = K_.conv2d_dgrad(dy, w, tuple(x.shape), stride=stride, pad=pad)
    torch.cuda.synchronize()
    _check(dx, dx_ref, "conv dgrad %s" % (case,))
    # accumulate mode: dx += grad
    base = torch.randn_like(dx)
    acc = base.clone()
    K_.conv2d_dgrad(dy, w, tuple(x.shape), stride=stride, pad=pad, out=acc, accumulate=True)
    torch.cuda.synchronize()
    _check(acc, dx_ref + base.float(), "conv dgrad acc %s" % (case,), rel=3e-2)


@pytest.mark.parametrize("case", CASES)
def test_conv_wgrad(case):
    from passl_b200 import kernels as K_
    torch.backends.cudnn.allow_tf32 = False
    x, w = _mk(case, 2)
    stride, pad = case[6], case[7]
    y = _ref(x, w, stride, pad)
    dy = torch.randn_like(y).bfloat16()
    _, dw_ref = _ref(x, w, stride, pad, dy)
    dw = K_.conv2d_wgrad(x, dy, tuple(w.shape), stride=stride, pad=pad)
    torch.cuda.synchronize()
    _check(dw, dw_ref, "conv wgrad %s" % (case,), rel=1e-2)


def test_conv_fwd_fused_epilogue():
    from passl_b200 import kernels as K_
    case = (2, 28, 28, 128, 256, 3, 1, 1)
    x, w = _mk(case, 3)
    res = torch.randn(2, 28, 28, 256, device="cuda").bfloat16()
    part = K_.stats_buffer(256, "cuda")
    out = K_.conv2d_fwd(x, w, stride=1, pad=1, residual=res, act="relu", col_stats=part)
    torch.cuda.synchronize()
    cs, cq = part[:, 0].sum(0), part[:, 1].sum(0)
    ref = torch.relu(_ref(x, w, 1, 1)) + res.float()
    _check(out, ref, "conv fused")
    o = out.float().reshape(-1, 256)
    assert torch.allclose(cs, o.sum(0), rtol=1e-3, atol=0.5)
    assert torch.allclose(cq, (o * o).sum(0), rtol=1e-3, atol=2.0)


@pytest.mark.parametrize("case", [(8, 56, 56, 64, 256, 1, 1, 0), (4, 14, 14, 256, 1024, 1, 1, 0), (3, 28, 28, 128, 128, 3, 1, 1),
                                  (2, 56, 56, 256, 512, 1, 2, 0), (5, 7, 7, 512, 2048, 1, 1, 0)])
def test_conv_fwd_fused_bn_statistics(case):
    """Statistics emitted by the conv epilogue == statistics of the stored bf16 tensor (what bn_stats would read back), including
    column blocks that move between CTAs (Cout > 256) and ragged last tiles."""
    from passl_b200 import kernels as K_
    x, w = _mk(case, 11)
    N, H, W, Cin, Cout, R, stride, pad = case
    part = K_.stats_buffer(Cout, "cuda")
    y = K_.conv2d_fwd(x, w, stride=stride, pad=pad, col_stats=part)
    y_plain = K_.conv2d_fwd(x, w, stride=stride, pad=pad)
    torch.cuda.synchronize()
    assert torch.equal(y, y_plain)
    o = y.double().reshape(-1, Cout)
    s1, s2 = part[:, 0].double().sum(0), part[:, 1].double().sum(0)
    assert torch.allclose(s1, o.sum(0), rtol=1e-4, atol=1e-2 * o.abs().sum(0).max().item() / o.shape[0] ** 0.5 + 1e-2)
    assert torch.allclose(s2, (o * o).sum(0), rtol=1e-4, atol=1e-3)
    ref_part = K_.bn_stats(y.view(-1, Cout))
    assert torch.allclose(s1.float(), ref_part[:, 0].sum(0), rtol=1e-4, atol=0.5)


@pytest.mark.parametrize("N,HW", [(4, 64), (2, 224), (3, 96)])
def test_stem_repack_conv_matches_conv7x7(N, HW):
    """7x7/2 pad 3 stem through the W-unfolded space-to-depth repack (csrc/stem.cu) == F.conv2d on bf16-rounded operands,
    forward and weight gradient (resnetimagenet.py:190-198)."""
    from passl_b200 import kernels as K_
    g = torch.Generator(device="cuda").manual_seed(5)
    img = torch.randn(N, 3, HW, HW, device="cuda", generator=g)
    w = torch.randn(64, 7, 7, 3, device="cuda", generator=g) / 147 ** 0.5
    W2 = torch.zeros(64, 152, device="cuda")
    W2[:, :147] = w.reshape(64, 147)
    xp = K_.stem_pack_input(img)
    wp = K_.stem_pack_weight(W2)
    part = K_.stats_buffer(64, "cuda")
    y = K_.stem_conv_fwd(xp, wp, col_stats=part)
    xr = img.bfloat16().float().requires_grad_(True)
    wr = w.bfloat16().float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    ref = F.conv2d(xr, wr, stride=2, padding=3)
    _check(y, ref.permute(0, 2, 3, 1), "stem fwd")
    o = y.float().reshape(-1, 64)
    assert torch.allclose(part[:, 0].sum(0), o.sum(0), rtol=1e-3, atol=0.5)
    dy = torch.randn(y.shape, device="cuda", generator=g).bfloat16()
    dw = torch.zeros(64, 152, device="cuda")
    dw[:, :147] = 1.0                                           # accumulate semantics
    K_.stem_conv_wgrad(xp, dy, dw)
    ref.backward(dy.float().permute(0, 3, 1, 2))
    dw_ref = wr.grad.permute(0, 2, 3, 1).reshape(64, 147) + 1.0
    _check(dw[:, :147], dw_ref, "stem wgrad", rel=1e-2)
    assert torch.equal(dw[:, 147:], torch.zeros(64, 5, device="cuda"))


@pytest.mark.parametrize("case", [(2, 56, 56, 64, 64, 3, 1, 1), (3, 13, 20, 64, 128, 3, 1, 1), (9, 14, 14, 256, 256, 3, 1, 1),
                                  (2, 28, 28, 128, 72, 3, 1, 1), (33, 16, 16, 128, 128, 3, 1, 1)])
def test_conv_wgrad_halo_tile_kernel(case):
    """3x3 / stride 1 weight gradient through the halo-tile kernel (wgrad_halo.cu): ragged tiles (W % 16, H % 8 != 0), Cout < 128,
    Cout % 64 != 0, many images (split-K), accumulation into a non-zero buffer."""
    from passl_b200 import kernels as K_, _lib
    _lib.load().passl_b200_wgrad_halo_mode(1)                     # small test shapes would otherwise take the generic kernel
    N, H, W, Cin, Cout, R, stride, pad = case
    g = torch.Generator(device="cuda").manual_seed(17)
    x = torch.randn(N, H, W, Cin, device="cuda", generator=g).bfloat16()
    dy = (torch.randn(N, H, W, Cout, device="cuda", generator=g) / (N * H * W) ** 0.5).bfloat16()
    xr = x.float().permute(0, 3, 1, 2).contiguous()
    wr = torch.zeros(Cout, Cin, 3, 3, device="cuda", requires_grad=True)
    F.conv2d(xr, wr, stride=1, padding=1).backward(dy.float().permute(0, 3, 1, 2).contiguous())
    dw_ref = wr.grad.permute(0, 2, 3, 1).contiguous()
    dw = torch.full((Cout, 3, 3, Cin), 0.5, device="cuda")
    try:
        K_.conv2d_wgrad(x, dy, (Cout, 3, 3, Cin), stride=1, pad=1, out=dw, accumulate=True)
        torch.cuda.synchronize()
    finally:
        _lib.load().passl_b200_wgrad_halo_mode(0)
    _check(dw, dw_ref + 0.5, "halo wgrad %s" % (case,), rel=1e-2)


def test_stem_wgrad_through_halo_kernel():
    """The 4x1 repacked-stem weight gradient through the halo-tile kernel (rows padded (2, 1), no column taps)."""
    from passl_b200 import kernels as K_, _lib
    g = torch.Generator(device="cuda").manual_seed(9)
    img = torch.randn(6, 3, 96, 96, device="cuda", generator=g)
    w = torch.randn(64, 7, 7, 3, device="cuda", generator=g) / 147 ** 0.5
    xp = K_.stem_pack_input(img)
    dy = (torch.randn(6, 48, 48, 64, device="cuda", generator=g) / 100).bfloat16()
    dw_generic = torch.zeros(64, 152, device="cuda")
    _lib.load().passl_b200_wgrad_halo_mode(2)
    try:
        K_.stem_conv_wgrad(xp, dy, dw_generic)
        _lib.load().passl_b200_wgrad_halo_mode(1)
        dw_halo = torch.zeros(64, 152, device="cuda")
        K_.stem_conv_wgrad(xp, dy, dw_halo)
        torch.cuda.synchronize()
    finally:
        _lib.load().passl_b200_wgrad_halo_mode(0)
    xr = img.bfloat16().float()
    wr = w.permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    F.conv2d(xr, wr, stride=2, padding=3).backward(dy.float().permute(0, 3, 1, 2))
    dw_ref = wr.grad.permute(0, 2, 3, 1).reshape(64, 147)
    _check(dw_halo[:, :147], dw_ref, "stem wgrad halo", rel=1e-2)
    _check(dw_generic[:, :147], dw_ref, "stem wgrad generic", rel=1e-2)


@pytest.mark.parametrize("case,halo_mode", [((64, 56, 56, 64, 256, 1, 1, 0), 0), ((64, 28, 28, 128, 128, 3, 1, 1), 1),
                                            ((64, 28, 28, 128, 128, 3, 1, 1), 2), ((32, 28, 28, 128, 256, 3, 2, 1), 0)])
def test_wgrad_split_k_is_bitwise_reproducible(case, halo_mode):
    """Split-K weight gradients sum their slices in a fixed order: two launches on the same operands, accumulating into the same
    starting values, give the same bits.  Cases: the 1x1 GEMM, the 3x3 halo-tile kernel (forced, mode 1), the generic 3x3 kernel
    (halo off, mode 2) and the generic stride-2 kernel."""
    from passl_b200 import _lib
    from passl_b200 import kernels as K
    N, H, W, Cin, Cout, R, stride, pad = case
    torch.manual_seed(0)
    Ho = (H + 2 * pad - R) // stride + 1
    x = torch.randn(N, H, W, Cin, device="cuda").bfloat16()
    dy = torch.randn(N, Ho, Ho, Cout, device="cuda").bfloat16()
    base = torch.randn(Cout, R, R, Cin, device="cuda")
    a, b = base.clone(), base.clone()
    _lib.load().passl_b200_wgrad_halo_mode(halo_mode)
    try:
        K.conv2d_wgrad(x, dy, (Cout, R, R, Cin), stride=stride, pad=pad, out=a, accumulate=True)
        K.conv2d_wgrad(x, dy, (Cout, R, R, Cin), stride=stride, pad=pad, out=b, accumulate=True)
        torch.cuda.synchronize()
    finally:
        _lib.load().passl_b200_wgrad_halo_mode(0)
    assert torch.equal(a, b)
