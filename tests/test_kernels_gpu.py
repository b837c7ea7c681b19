"""Per-kernel parity on the B200: each CUDA kernel, called through the C ABI, against a torch fp32/fp64 restatement."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from breaching_b200 import engine as E  # noqa: E402

DEV = "cuda:0"

# (N, H, W, Ci, Co, R, stride, pad): every distinct ResNet-18/50 conv shape class (SURVEY.md 2.1), scaled spatially
# where the full size adds nothing but time, plus ragged / tiny-channel cases (3-channel stem, odd sizes).
CONV_SHAPES = [
    (1, 224, 224, 3, 64, 7, 2, 3),    # stem (full size; Ci=3 exercises the scalar loaders)
    (1, 56, 56, 64, 64, 3, 1, 1),     # layer1
    (1, 56, 56, 64, 128, 3, 2, 1),    # layer2.0 conv1
    (1, 56, 56, 64, 128, 1, 2, 0),    # layer2.0 downsample
    (1, 28, 28, 128, 128, 3, 1, 1),
    (1, 14, 14, 256, 256, 3, 1, 1),
    (1, 14, 14, 256, 512, 3, 2, 1),
    (1, 7, 7, 512, 512, 3, 1, 1),     # tiny-M, split-K heavy
    (2, 14, 14, 256, 1024, 1, 1, 0),  # bottleneck 1x1 expansions
    (2, 28, 28, 512, 128, 1, 1, 0),
    (2, 32, 32, 3, 64, 3, 1, 1),      # ConvNet stem (small-Ci dgrad kernel, stride 1)
    (2, 12, 13, 1, 8, 3, 2, 1),       # single input channel, stride 2, odd sizes
    (1, 9, 9, 4, 6, 5, 3, 2),         # 5x5 stride 3
    (3, 9, 11, 5, 7, 3, 1, 1),        # ragged everything
    (2, 10, 10, 6, 10, 3, 3, 0),
    (1, 1, 1, 512, 397, 1, 1, 0),     # the linear head as a 1x1 conv
    (4, 1, 1, 2304, 10, 1, 1, 0),
]


def _rand(*shape, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(*shape, generator=g).to(DEV)


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _relerr(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


@pytest.mark.parametrize("shape", CONV_SHAPES)
def test_conv_fprop_dgrad_wgrad_simt(shape):
    N, H, W, Ci, Co, R, st, pd = shape
    x = _rand(N, Ci, H, W, seed=1)
    w = _rand(Co, Ci, R, R, seed=2) * 0.1
    Ho, Wo = (H + 2 * pd - R) // st + 1, (W + 2 * pd - R) // st + 1
    dy = _rand(N, Co, Ho, Wo, seed=3)
    x2, w2, dy2 = _rand(N, Ci, H, W, seed=4), _rand(Co, Ci, R, R, seed=5) * 0.1, _rand(N, Co, Ho, Wo, seed=6)
    xd, wd, dyd = x.double(), w.double(), dy.double()
    w_ohwi = w.permute(0, 2, 3, 1).contiguous()
    w2_ohwi = w2.permute(0, 2, 3, 1).contiguous()
    tol = 2e-5

    out = torch.empty(N, Ho, Wo, Co, device=DEV)
    E.conv_gemm(0, _nhwc(x), w_ohwi, out, N, H, W, Ci, Co, R, R, st, pd)
    ref = F.conv2d(xd, wd, stride=st, padding=pd)
    assert _relerr(out.permute(0, 3, 1, 2), ref) < tol, "fprop"
    E.conv_gemm(0, _nhwc(x), w_ohwi, out, N, H, W, Ci, Co, R, R, st, pd, a2=_nhwc(x2), w2=w2_ohwi)
    ref2 = ref + F.conv2d(x2.double(), w2.double(), stride=st, padding=pd)
    assert _relerr(out.permute(0, 3, 1, 2), ref2) < tol, "fprop dual"

    din = torch.empty(N, H, W, Ci, device=DEV)
    E.conv_gemm(1, _nhwc(dy), w_ohwi, din, N, H, W, Ci, Co, R, R, st, pd)
    refd = torch.nn.grad.conv2d_input((N, Ci, H, W), wd, dyd, stride=st, padding=pd)
    assert _relerr(din.permute(0, 3, 1, 2), refd) < tol, "dgrad"
    E.conv_gemm(1, _nhwc(dy), w_ohwi, din, N, H, W, Ci, Co, R, R, st, pd, a2=_nhwc(dy2), w2=w2_ohwi)
    refd2 = refd + torch.nn.grad.conv2d_input((N, Ci, H, W), w2.double(), dy2.double(), stride=st, padding=pd)
    assert _relerr(din.permute(0, 3, 1, 2), refd2) < tol, "dgrad dual"

    dw = torch.empty(Co, R, R, Ci, device=DEV)
    E.conv_gemm(2, _nhwc(x), _nhwc(dy), dw, N, H, W, Ci, Co, R, R, st, pd)
    refw = torch.nn.grad.conv2d_weight(xd, (Co, Ci, R, R), dyd, stride=st, padding=pd)
    assert _relerr(dw.permute(0, 3, 1, 2), refw) < tol, "wgrad"
    # dual-source wgrad (tangent weight gradients of the FedAvg adjoint): dout^T a + dout2^T a2
    E.conv_gemm(2, _nhwc(x), _nhwc(dy), dw, N, H, W, Ci, Co, R, R, st, pd, a2=_nhwc(x2), w2=_nhwc(dy2))
    refw2 = refw + torch.nn.grad.conv2d_weight(x2.double(), (Co, Ci, R, R), dy2.double(), stride=st, padding=pd)
    assert _relerr(dw.permute(0, 3, 1, 2), refw2) < tol, "wgrad dual"


def test_conv_is_deterministic_across_launches():
    N, H, W, Ci, Co, R, st, pd = 1, 7, 7, 512, 512, 3, 1, 1
    x, w = _nhwc(_rand(N, Ci, H, W, seed=1)), _rand(Co, R, R, Ci, seed=2)
    a = torch.empty(N, H, W, Co, device=DEV)
    b = torch.empty_like(a)
    E.conv_gemm(0, x, w, a, N, H, W, Ci, Co, R, R, st, pd)
    E.conv_gemm(0, x, w, b, N, H, W, Ci, Co, R, R, st, pd)
    assert torch.equal(a, b)  # split-K partials are reduced in a fixed order


@pytest.mark.parametrize("n", [1, 1023, 1024, 4097, 11_380_173])
def test_match_reduce(n):
    G, g = _rand(n, seed=1), _rand(n, seed=2)
    nchunks = (n + 1023) // 1024
    w = torch.rand(nchunks, device=DEV)
    sums = E.match_reduce(G, g, w)
    Gd, gd = G.double(), g.double()
    wl = w.double().repeat_interleave(1024)[:n]
    ref = [(Gd * gd).sum(), (Gd * Gd).sum(), (gd * gd).sum(), ((Gd - gd) ** 2).sum(), (wl * (Gd - gd).abs()).sum()]
    for a, b in zip(sums, ref):
        assert math.isclose(a, b.item(), rel_tol=1e-6, abs_tol=1e-6), (sums, [r.item() for r in ref])
    again = E.match_reduce(G, g, w)
    assert again == sums  # deterministic
    m = E.match_reduce(G, g, None, mask_value=0.5)
    mask = (gd.abs() > 0.5)
    assert math.isclose(m[0], (Gd * gd * mask).sum().item(), rel_tol=1e-6)
    assert math.isclose(m[1], ((Gd * mask) ** 2).sum().item(), rel_tol=1e-6)


@pytest.mark.parametrize("p,q,dbl", [(1, 1, False), (2, 0.5, True), (2, 1.25, False), (1, 1, True)])
@pytest.mark.parametrize("shape", [(1, 3, 224, 224), (2, 3, 32, 32), (3, 3, 17, 45)])
def test_total_variation_value_and_gradient(p, q, dbl, shape):
    from oracle import restate

    x = _rand(*shape, seed=3)
    val, grad = E.total_variation(x, scale=0.2, inner_exp=p, outer_exp=q, double_opponents=dbl)
    xd = x.double().cpu().requires_grad_(True)
    ref = restate.total_variation(xd, scale=0.2, inner_exp=p, outer_exp=q, double_opponents=dbl)
    (gref,) = torch.autograd.grad(ref, xd)
    assert math.isclose(val, ref.item(), rel_tol=2e-5), (val, ref.item())
    assert _relerr(grad.cpu(), gref) < 5e-5
    base = grad.clone()  # accumulate on top of an existing gradient: result must be exactly doubled
    _, acc = E.total_variation(x, scale=0.2, inner_exp=p, outer_exp=q, double_opponents=dbl, grad=base)
    assert _relerr(acc.cpu(), 2 * gref) < 5e-5


def tc_claims(mode, shape):
    """Does the tcgen05 back end take this NHWC convolution (igemm_tc_supported / narrow_tiles_ok)?  Output tiles are 128 x 64, or
    128 x 32 where the tile width (fprop: Co, dgrad: Ci, wgrad: R R Ci) is only a multiple of 32 -- and then dgrad only at stride 1,
    wgrad only with Ci % 32 == 0."""
    N, H, W, Ci, Co, R, st, pd = shape
    width = {0: Co, 1: Ci, 2: R * R * Ci}[mode]
    narrow_ok = (mode != 1 or st == 1) and (mode != 2 or Ci % 32 == 0)
    if R * R > 64 or not (width % 64 == 0 or (width % 32 == 0 and narrow_ok)):
        return False
    return {0: Ci % 32 == 0, 1: Co % 32 == 0, 2: Co % 4 == 0 and Ci % 4 == 0}[mode]


TC_SHAPES = [s for s in CONV_SHAPES if tc_claims(0, s)] + [
    (1, 56, 56, 64, 64, 3, 1, 1), (8, 14, 14, 128, 256, 3, 2, 1),
    (1, 2, 2, 512, 512, 3, 1, 1), (1, 4, 4, 256, 256, 3, 1, 1), (4, 8, 8, 128, 128, 3, 1, 1),   # tiny spatial extents (64x64 inputs)
    (3, 9, 11, 64, 64, 3, 1, 1), (2, 15, 13, 64, 128, 3, 2, 1), (1, 5, 5, 96, 64, 3, 1, 1),    # ragged tiles, odd sizes, Ci = 96
    (8, 56, 56, 64, 256, 1, 1, 0), (8, 28, 28, 128, 128, 3, 1, 1), (2, 28, 28, 256, 64, 1, 2, 0),  # ResNet-50 batch-8 shapes
    # 128 x 32 tiles: Co / Ci in {32, 96}, stride 1 and 2, 1 x 1 and 3 x 3, ragged spatial sizes
    (2, 33, 29, 32, 96, 3, 1, 1), (2, 33, 29, 96, 64, 3, 1, 1), (2, 15, 13, 32, 32, 3, 1, 1), (3, 9, 11, 96, 96, 1, 1, 0),
    (2, 15, 13, 96, 32, 3, 2, 1), (2, 17, 11, 32, 96, 1, 2, 0), (1, 7, 9, 64, 32, 3, 1, 1), (2, 13, 15, 32, 64, 3, 2, 1),
]


@pytest.mark.parametrize("shape", TC_SHAPES)
def test_conv_tcgen05_tf32_backend(shape):
    """tcgen05 TF32 back end (tensor cores, TMEM accumulators): TF32 products (10-bit mantissa), fp32 accumulation,
    tolerance 2e-3 relative l2 -- the precision of the reference's default cuDNN TF32 conv path.  Every mode the dispatcher
    claims must be accepted (a refusal raises), every other mode refused."""
    N, H, W, Ci, Co, R, st, pd = shape
    x = _rand(N, Ci, H, W, seed=1)
    w = _rand(Co, Ci, R, R, seed=2) * 0.1
    Ho, Wo = (H + 2 * pd - R) // st + 1, (W + 2 * pd - R) // st + 1
    dy = _rand(N, Co, Ho, Wo, seed=3)
    x2, w2, dy2 = _rand(N, Ci, H, W, seed=4), _rand(Co, Ci, R, R, seed=5) * 0.1, _rand(N, Co, Ho, Wo, seed=6)
    w_ohwi, w2_ohwi = w.permute(0, 2, 3, 1).contiguous(), w2.permute(0, 2, 3, 1).contiguous()
    tol = 2e-3
    out = torch.empty(N, Ho, Wo, Co, device=DEV)
    E.conv_gemm(0, _nhwc(x), w_ohwi, out, N, H, W, Ci, Co, R, R, st, pd, a2=_nhwc(x2), w2=w2_ohwi, backend=1)
    ref = F.conv2d(x.double(), w.double(), stride=st, padding=pd) + F.conv2d(x2.double(), w2.double(), stride=st, padding=pd)
    assert _relerr(out.permute(0, 3, 1, 2), ref) < tol, "fprop dual"
    again = torch.empty_like(out)
    E.conv_gemm(0, _nhwc(x), w_ohwi, again, N, H, W, Ci, Co, R, R, st, pd, a2=_nhwc(x2), w2=w2_ohwi, backend=1)
    assert torch.equal(out, again)
    assert tc_claims(0, shape)
    for mode in (1, 2):
        if not tc_claims(mode, shape):
            with pytest.raises(E.EngineError):
                E.conv_gemm(mode, _nhwc(dy) if mode == 1 else _nhwc(x), w_ohwi if mode == 1 else _nhwc(dy),
                            torch.empty(N * H * W * Ci if mode == 1 else Co * R * R * Ci, device=DEV), N, H, W, Ci, Co, R, R, st, pd, backend=1)
    if tc_claims(1, shape):
        din = torch.empty(N, H, W, Ci, device=DEV)
        E.conv_gemm(1, _nhwc(dy), w_ohwi, din, N, H, W, Ci, Co, R, R, st, pd, a2=_nhwc(dy2), w2=w2_ohwi, backend=1)
        refd = torch.nn.grad.conv2d_input((N, Ci, H, W), w.double(), dy.double(), stride=st, padding=pd) + \
            torch.nn.grad.conv2d_input((N, Ci, H, W), w2.double(), dy2.double(), stride=st, padding=pd)
        assert _relerr(din.permute(0, 3, 1, 2), refd) < tol, "dgrad dual"
    if tc_claims(2, shape):
        dw = torch.empty(Co, R, R, Ci, device=DEV)
        E.conv_gemm(2, _nhwc(x), _nhwc(dy), dw, N, H, W, Ci, Co, R, R, st, pd, backend=1)
        refw = torch.nn.grad.conv2d_weight(x.double(), (Co, Ci, R, R), dy.double(), stride=st, padding=pd)
        assert _relerr(dw.permute(0, 3, 1, 2), refw) < tol, "wgrad"
        E.conv_gemm(2, _nhwc(x), _nhwc(dy), dw, N, H, W, Ci, Co, R, R, st, pd, a2=_nhwc(x2), w2=_nhwc(dy2), backend=1)
        refw2 = refw + torch.nn.grad.conv2d_weight(x2.double(), (Co, Ci, R, R), dy2.double(), stride=st, padding=pd)
        assert _relerr(dw.permute(0, 3, 1, 2), refw2) < tol, "wgrad dual"


@pytest.mark.gpu
@pytest.mark.parametrize("rows,Ci,Co,dual", [(32, 96, 50304, False), (32, 96, 50304, True), (5, 64, 9000, True), (17, 128, 8192, False)])
def test_tall_linear_dgrad_matches_float64(rows, Ci, Co, dual):
    """dgrad of a linear layer with a very long reduction (the token models' 96 -> 50257 decoder, tag.yaml / BASELINE config 5):
    chunked fp32 register reduction + fixed-order fold (csrc/linear_small.cu) against float64; run twice: bitwise reproducible."""
    from breaching_b200 import engine as E

    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(rows * 1000 + Ci)
    dy = torch.randn(rows, Co, generator=g).to(dev)
    w = (torch.randn(Co, Ci, generator=g) / 8).to(dev)
    dy2 = torch.randn(rows, Co, generator=g).to(dev) if dual else None
    w2 = (torch.randn(Co, Ci, generator=g) / 8).to(dev) if dual else None
    want = dy.double() @ w.double()
    if dual:
        want = want + dy2.double() @ w2.double()
    for backend in (0, 1):
        out = torch.full((rows, Ci), float("nan"), device=dev)
        E.conv_gemm(1, dy, w, out, rows, 1, 1, Ci, Co, 1, 1, 1, 0, a2=dy2, w2=w2, backend=backend)
        again = torch.empty_like(out)
        E.conv_gemm(1, dy, w, again, rows, 1, 1, Ci, Co, 1, 1, 1, 0, a2=dy2, w2=w2, backend=backend)
        torch.cuda.synchronize()
        assert torch.equal(out, again)
        rel = ((out.double() - want).norm() / want.norm()).item()
        assert rel < 2e-6, (backend, rel)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,Ci,Co", [(32, 96, 288), (32, 96, 1536), (20, 96, 96), (32, 1536, 96), (1, 512, 397), (8, 2048, 397)])
def test_small_row_linear_kernels_match_float64(rows, Ci, Co):
    """Linear layers on <= 32 rows (classification heads, token-model projections at batch 1) through the engine's dispatch rule
    (`bre_conv_gemm` backend 2: matrix-vector kernels for short reductions, the GEMM back ends otherwise): fprop / dgrad with one and
    two sources and wgrad against float64."""
    from breaching_b200 import engine as E

    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(rows + Ci + Co)
    x, x2 = (torch.randn(rows, Ci, generator=g).to(dev) for _ in range(2))
    w, w2 = ((torch.randn(Co, Ci, generator=g) / Ci ** 0.5).to(dev) for _ in range(2))
    dy, dy2 = (torch.randn(rows, Co, generator=g).to(dev) for _ in range(2))
    geom = (rows, 1, 1, Ci, Co, 1, 1, 1, 0)

    def rel(a, b):
        return ((a.double() - b).norm() / b.norm()).item()

    for backend, tol in ((0, 2e-6), (2, 2e-3)):   # 2 = engine dispatch: TF32 products where the tcgen05 kernel takes the shape
        out = torch.empty(rows, Co, device=dev)
        E.conv_gemm(0, x, w, out, *geom, backend=backend)
        assert rel(out, x.double() @ w.double().T) < tol, ("fprop", backend)
        E.conv_gemm(0, x, w, out, *geom, a2=x2, w2=w2, backend=backend)
        assert rel(out, x.double() @ w.double().T + x2.double() @ w2.double().T) < tol, ("fprop2", backend)
        din = torch.empty(rows, Ci, device=dev)
        E.conv_gemm(1, dy, w, din, *geom, backend=backend)
        assert rel(din, dy.double() @ w.double()) < tol, ("dgrad", backend)
        E.conv_gemm(1, dy, w, din, *geom, a2=dy2, w2=w2, backend=backend)
        assert rel(din, dy.double() @ w.double() + dy2.double() @ w2.double()) < tol, ("dgrad2", backend)
        dw = torch.empty(Co, Ci, device=dev)
        E.conv_gemm(2, x, dy, dw, *geom, backend=backend)
        assert rel(dw, dy.double().T @ x.double()) < tol, ("wgrad", backend)
