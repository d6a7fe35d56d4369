"""The image branch's streaming kernels (csrc/tm_conv.cu: batch norm + ReLU, 2x2 pooling, OutConv, LeakyReLU) and the
head's column gather / scatter (csrc/tm_fuse.cu), each called through tm_lib and compared with an fp64 reference.

Every kernel has a 128-bit path (C % 4 == 0, 16-byte aligned rows) and a scalar path.  The "vec" layout puts the
tensor inside a wider buffer (pixel stride C + 8, first column 4); the "scalar" layout uses a pixel stride of C + 5 and
a pointer one float past an aligned address, which the ABI must accept.  Where the two paths do the same arithmetic per
element, their results are compared bit for bit."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"
TM_EPI_RELU = 2
MOMENTUM, EPS = 0.1, 1e-5


@pytest.fixture(scope="module")
def lib(pkg):
    import tm_lib
    return tm_lib


def _view(rows, C, layout, fill=float("nan"), dtype=torch.float32):
    """(rows, C) view with a pixel stride and first column set by ``layout``, plus the whole buffer (for the
    untouched-columns checks).  ``fill`` goes everywhere first."""
    ld, c0 = (C + 8, 4) if layout == "vec" else (C + 5, 1)
    buf = torch.full((rows, ld), fill, device=DEV, dtype=dtype)
    return buf[:, c0:c0 + C], buf, ld


def _strided(t, layout):
    v, _, ld = _view(t.shape[0], t.shape[1], layout)
    v.copy_(t)
    return v, ld


def _bits(t):
    return t.contiguous().view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def _bf16_bits(t):
    return t.to(torch.bfloat16).contiguous().view(torch.int16)


def _bn_inputs(npix, C, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    mu = torch.randn(C, device=DEV, generator=g) * 3
    sd = torch.rand(C, device=DEV, generator=g) * 2 + 0.2
    x = torch.randn(npix, C, device=DEV, generator=g) * sd + mu
    if C > 1:
        x[:, 0] = 0.0                                   # an identically-zero channel: y = relu(beta)
    gamma = torch.randn(C, device=DEV, generator=g)
    beta = torch.randn(C, device=DEV, generator=g)
    beta[0] = 0.7
    rm = torch.randn(C, device=DEV, generator=g)
    rv = torch.rand(C, device=DEV, generator=g) + 0.5
    return x, gamma, beta, rm, rv


def _bn_forward(lib, x, ldx, gamma, beta, rm, rv, layout, stats_part=None, nparts=0):
    npix, C = x.shape
    y, ybuf, ldy = _view(npix, C, layout, fill=-7.0)
    smean = torch.empty(C, device=DEV)
    sinv = torch.empty(C, device=DEV)
    yb = torch.empty(npix, C, device=DEV, dtype=torch.bfloat16)
    nb = lib.ws_bytes("tm_bn_ws", npix, C)
    lib.call("tm_bn_relu_forward", npix, C, x, ldx, gamma, beta, rm, rv, MOMENTUM, EPS, y, ldy, smean, sinv, yb,
             stats_part, nparts, lib.workspace(nb, DEV), nb, lib.stream())
    return y, ybuf, ldy, smean, sinv, yb


def _bn_ref(x, gamma, beta, mean=None, var=None):
    x64 = x.double()
    if mean is None:
        mean = x64.mean(0)
        var = ((x64 - mean) ** 2).mean(0)                # two-pass
    invstd = 1.0 / torch.sqrt(var + EPS)
    y = torch.relu((x64 - mean) * invstd * gamma.double() + beta.double())
    return mean, var, invstd, y


@pytest.mark.parametrize("layout", ["vec", "scalar"])
@pytest.mark.parametrize("npix", [2, 7, 591, 593, 4096, 2 ** 18 + 3])
@pytest.mark.parametrize("C", [1, 3, 6, 16, 32, 64, 128, 256])
def test_bn_relu_forward(lib, C, npix, layout):
    """tm_bn_relu_forward (train mode): batch statistics, y, the running statistics (unbiased variance, momentum) and
    the bf16 side output against an fp64 two-pass batch norm; npix around the 592-block partition and beyond."""
    x0, gamma, beta, rm0, rv0 = _bn_inputs(npix, C, seed=npix * 7 + C)
    x, ldx = _strided(x0, layout)
    rm, rv = rm0.clone(), rv0.clone()
    y, ybuf, ldy, smean, sinv, yb = _bn_forward(lib, x, ldx, gamma, beta, rm, rv, layout)
    mean, var, invstd, yref = _bn_ref(x0, gamma, beta)
    assert_close(smean, mean, 1e-6, 1e-6, "save_mean")
    assert_close(sinv, invstd, 1e-5, 0.0, "save_invstd")
    assert_close(y, yref, 1e-5, 1e-5, "y")
    unbiased = var * npix / (npix - 1)
    assert_close(rm, (1 - MOMENTUM) * rm0.double() + MOMENTUM * mean, 1e-6, 1e-6, "running_mean")
    assert_close(rv, (1 - MOMENTUM) * rv0.double() + MOMENTUM * unbiased, 1e-6, 0.0, "running_var")
    assert torch.equal(_bf16_bits(y), yb.view(torch.int16)), "y_bf16 != bf16(y)"
    if C > 1:
        assert bool((y[:, 0] == torch.relu(beta[0])).all()), "zero channel: y != relu(beta)"
    outside = torch.ones_like(ybuf, dtype=torch.bool)
    c0 = 4 if layout == "vec" else 1
    outside[:, c0:c0 + C] = False
    assert bool((ybuf[outside] == -7.0).all()), "y columns outside the tensor were written"


@pytest.mark.parametrize("layout", ["vec", "scalar"])
@pytest.mark.parametrize("npix,C", [(7, 3), (593, 16), (4096, 64), (4096, 256), (65537, 32), (2 ** 18 + 3, 16)])
def test_bn_relu_backward(lib, npix, C, layout):
    """tm_bn_relu_backward: dx, dgamma, dbeta against fp64 autograd of relu(batch_norm(x)); dx with y given equals
    dx with y = NULL (the mask rebuilt from x and the saved statistics) bit for bit; dx_bf16 = bf16(dx) bit for bit.
    The incoming gradient is zero where the fp64 pre-activation is within 1e-4 of 0, so that the ReLU gate's side
    there cannot matter."""
    x0, gamma, beta, rm, rv = _bn_inputs(npix, C, seed=npix + 3 * C)
    gamma[1 % C] = 0.0                                   # a channel whose every gate is decided by beta alone
    x, ldx = _strided(x0, layout)
    y, _, ldy, smean, sinv, _ = _bn_forward(lib, x, ldx, gamma, beta, rm, rv, layout)
    g = torch.Generator(device=DEV).manual_seed(npix + C)
    dy0 = torch.randn(npix, C, device=DEV, generator=g)
    x64 = x0.double().requires_grad_(True)
    g64 = gamma.double().requires_grad_(True)
    b64 = beta.double().requires_grad_(True)
    pre = F.batch_norm(x64, None, None, g64, b64, training=True, momentum=0.0, eps=EPS)
    dy0[pre.detach().abs() < 1e-4] = 0.0
    dx_ref, dg_ref, db_ref = torch.autograd.grad(torch.relu(pre), (x64, g64, b64), dy0.double())
    dy, lddy = _strided(dy0, layout)
    nb = lib.ws_bytes("tm_bn_ws", npix, C)
    outs = []
    for yy in (y, None):
        dx, _, lddx = _view(npix, C, layout)
        dgamma, dbeta = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
        dxb = torch.empty(npix, C, device=DEV, dtype=torch.bfloat16)
        lib.call("tm_bn_relu_backward", npix, C, x, ldx, yy, ldy, dy, lddy, gamma, beta, smean, sinv, dx, lddx,
                 dgamma, dbeta, dxb, lib.workspace(nb, DEV), nb, lib.stream())
        outs.append((dx, dgamma, dbeta, dxb))
    dx, dgamma, dbeta, dxb = outs[0]
    assert_close(dbeta, db_ref, 1e-5, 1e-5, "dbeta")
    assert_close(dgamma, dg_ref, 1e-5, 1e-5, "dgamma")
    assert_close(dx, dx_ref, 1e-4, 1e-5, "dx")
    assert torch.equal(_bf16_bits(dx), dxb.view(torch.int16)), "dx_bf16 != bf16(dx)"
    for a, b, name in zip(outs[0], outs[1], ("dx", "dgamma", "dbeta", "dx_bf16")):
        assert torch.equal(_bits(a), _bits(b)), f"{name} with y = NULL differs from {name} with y"


@pytest.mark.parametrize("npix,C", [(7, 3), (4096, 16), (1000, 256), (65537, 6)])
def test_bn_relu_eval(lib, npix, C):
    """tm_bn_relu_eval: y = relu(gamma (x - running_mean) / sqrt(running_var + eps) + beta) against fp64, the
    statistics it reports, and the vector and scalar paths bit-identical (same statistics, same arithmetic)."""
    x0, gamma, beta, rm, rv = _bn_inputs(npix, C, seed=5 * npix + C)
    _, _, invstd, yref = _bn_ref(x0, gamma, beta, rm.double(), rv.double())
    ys = []
    for layout in ("vec", "scalar"):
        x, ldx = _strided(x0, layout)
        y, _, ldy = _view(npix, C, layout)
        smean, sinv = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
        yb = torch.empty(npix, C, device=DEV, dtype=torch.bfloat16)
        lib.call("tm_bn_relu_eval", npix, C, x, ldx, gamma, beta, rm, rv, EPS, y, ldy, smean, sinv, yb, lib.stream())
        assert torch.equal(smean, rm)
        assert_close(sinv, invstd, 1e-6, 0.0, "eval invstd")
        assert_close(y, yref, 1e-5, 1e-5, "eval y")
        assert torch.equal(_bf16_bits(y), yb.view(torch.int16))
        ys.append(y)
    assert torch.equal(_bits(ys[0]), _bits(ys[1])), "eval: vector and scalar paths differ"


@pytest.mark.parametrize("npix,C,nparts", [(4096, 16, 1000), (593, 3, 7), (1024, 128, 2368)])
def test_bn_relu_forward_stats_part(lib, npix, C, nparts):
    """tm_bn_relu_forward with stats_part: hand-built fp64 partials [nparts][C][2] (sum, sum of squares) describing a
    distribution unlike x's.  y, the saved and the running statistics must follow the partials (the statistics pass
    over x skipped); the vector and scalar apply paths give the same bits."""
    x0, gamma, beta, rm0, rv0 = _bn_inputs(npix, C, seed=npix + nparts)
    g = torch.Generator(device=DEV).manual_seed(nparts)
    m = torch.randn(C, device=DEV, dtype=torch.float64, generator=g) * 2 + 10.0
    v = torch.rand(C, device=DEV, dtype=torch.float64, generator=g) * 4 + 0.25
    w = torch.rand(nparts, C, device=DEV, dtype=torch.float64, generator=g)
    w = w / w.sum(0)                                     # each partial holds a share of the sums
    part = torch.stack([w * (npix * m), w * (npix * (v + m * m))], dim=-1).contiguous()
    _, _, invstd, yref = _bn_ref(x0, gamma, beta, m, v)
    ys = []
    for layout in ("vec", "scalar"):
        x, ldx = _strided(x0, layout)
        rm, rv = rm0.clone(), rv0.clone()
        y, _, _, smean, sinv, yb = _bn_forward(lib, x, ldx, gamma, beta, rm, rv, layout, part, nparts)
        assert_close(smean, m, 1e-6, 0.0, "stats_part mean")
        assert_close(sinv, invstd, 1e-5, 0.0, "stats_part invstd")
        assert_close(y, yref, 1e-5, 1e-5, "stats_part y")
        assert_close(rm, (1 - MOMENTUM) * rm0.double() + MOMENTUM * m, 1e-6, 1e-6, "stats_part running_mean")
        assert_close(rv, (1 - MOMENTUM) * rv0.double() + MOMENTUM * v * npix / (npix - 1), 1e-6, 0.0,
                     "stats_part running_var")
        assert torch.equal(_bf16_bits(y), yb.view(torch.int16))
        ys.append(y)
    assert torch.equal(_bits(ys[0]), _bits(ys[1])), "stats_part: vector and scalar paths differ"


@pytest.mark.parametrize("npix,C", [(64 * 64, 16), (256 * 256, 16), (128 * 128, 64), (4096, 3)])
def test_bn_large_mean_over_std(lib, npix, C):
    """Channels x = 3000 + c + N(0, 1): a mean thousands of standard deviations from zero (a convolution without
    bias over a large constant background).  invstd and y must be no worse than twice the error of PyTorch's
    fp32 CUDA batch norm on the same tensor (or than two fp32 ulps, the resolution of the stored result), and never
    worse than 1e-4 relative.  Unshifted E[x^2] - mean^2 sums lose ~3e-3 of the variance here."""
    g = torch.Generator(device=DEV).manual_seed(npix + C)
    base = 3000.0 + torch.arange(C, device=DEV, dtype=torch.float32)
    x0 = (torch.randn(npix, C, device=DEV, generator=g) + base).contiguous()
    gamma = torch.rand(C, device=DEV, generator=g) + 0.5
    beta = torch.randn(C, device=DEV, generator=g)
    _, _, invstd, yref = _bn_ref(x0, gamma, beta)
    yref_scale = float(yref.abs().max())
    _, t_mean, t_invstd = torch.native_batch_norm(x0, gamma, beta, None, None, True, MOMENTUM, EPS)
    t_y = torch.relu(F.batch_norm(x0, None, None, gamma, beta, training=True, momentum=MOMENTUM, eps=EPS))
    t_err_inv = float(((t_invstd.double() - invstd) / invstd).abs().max())
    t_err_y = float((t_y.double() - yref).abs().max()) / yref_scale
    floor = 2.0 ** -22
    for layout in ("vec", "scalar"):
        x, ldx = _strided(x0, layout)
        rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
        y, _, _, _, sinv, _ = _bn_forward(lib, x, ldx, gamma, beta, rm, rv, layout)
        err_inv = float(((sinv.double() - invstd) / invstd).abs().max())
        err_y = float((y.double() - yref).abs().max()) / yref_scale
        msg = (f"{layout}: invstd rel err {err_inv:.3e} (torch {t_err_inv:.3e}), y err {err_y:.3e} "
               f"(torch {t_err_y:.3e})")
        assert err_inv <= max(2 * t_err_inv, floor) and err_inv <= 1e-4, msg
        assert err_y <= max(2 * t_err_y, floor) and err_y <= 1e-4, msg


# ------------------------------------------------------------------------------------------------- pooling
def _pool_input(B, H, W, C, seed, nan):
    """NHWC values from {-2, -1.5, ..., 2} (many tied windows), signed zeros, and a few NaN."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(-4, 5, (B, H, W, C), generator=g).double() / 2
    zero = x == 0
    neg = torch.rand(B, H, W, C, generator=g) < 0.5
    x[zero & neg] = -0.0
    x[0, :, :, 0] = 1.0                                  # whole windows of one value
    if nan:
        x.view(-1)[torch.randperm(x.numel(), generator=g)[: max(1, x.numel() // 50)]] = float("nan")
    return x


def _same(a, b):
    """equal values, NaN where the other has NaN"""
    a, b = a.double().cpu(), b.double().cpu()
    return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


def _pool_call(lib, x, mode, relu, add, dyo, layout):
    """forward and backward through tm_pool2x2_*; ``layout`` "vec" = contiguous NHWC, "scalar" = every tensor one
    float past an aligned address."""
    B, H, W, C = x.shape
    Ho, Wo = H // 2, W // 2
    sh = 0 if layout == "vec" else 1

    def dev(t):
        buf = torch.empty(t.numel() + 1, device=DEV)
        v = buf[sh:sh + t.numel()].view(t.shape)
        v.copy_(t)
        return v

    xd = dev(x.float())
    y = dev(torch.full((B, Ho, Wo, C), -9.0))
    idx = torch.full((B * Ho * Wo * C,), 255, device=DEV, dtype=torch.uint8)
    flags = TM_EPI_RELU if relu else 0
    lib.call("tm_pool2x2_forward", B, H, W, C, mode, xd, C, y, C, idx, flags, lib.stream())
    dyd = dev(dyo.float())
    ad = dev(add.float()) if add is not None else None
    dx = dev(torch.full((B, H, W, C), -9.0))
    lib.call("tm_pool2x2_backward", B, H, W, C, mode, dyd, C, y, C, idx, dx, C, flags, ad, C, lib.stream())
    return y.cpu(), idx.cpu(), dx.cpu()


@pytest.mark.parametrize("HW", [(8, 8), (7, 9), (6, 5), (9, 4)])
@pytest.mark.parametrize("C", [1, 3, 16, 64])
@pytest.mark.parametrize("add", [False, True])
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("mode", [0, 1])
def test_pool2x2(lib, mode, relu, add, C, HW):
    """tm_pool2x2_forward / _backward, max (mode 0) and avg (mode 1), against fp64 on the CPU: the max winners are
    torch's max_pool2d indices (first maximum in window order, NaN propagates) as the window index 2*dy + dx; the
    backward routes dy to the winner (avg: dy / 4), masked by y > 0 with the ReLU, plus the skip gradient ``add``; the
    trailing odd row and column get 0 + add.  The vector path (C % 4 == 0, even H and W) is also run through the
    scalar path, and both give the same bits.  Only the max pool without the ReLU sees NaN: the ReLU is fmaxf, which
    maps NaN to 0."""
    H, W = HW
    B = 2
    nan = mode == 0 and not relu
    x = _pool_input(B, H, W, C, seed=H * 100 + W * 10 + C + 1000 * mode + 4000 * relu, nan=nan)
    g = torch.Generator().manual_seed(C + H)
    Ho, Wo = H // 2, W // 2
    dyo = torch.randn(B, Ho, Wo, C, generator=g).double()
    addt = torch.randn(B, H, W, C, generator=g).double() if add else None
    # fp64 reference (NCHW on the CPU)
    xn = x.permute(0, 3, 1, 2).contiguous()
    if mode == 0:
        yr, ind = F.max_pool2d(xn, 2, 2, return_indices=True)
        iy, ix = ind // W, ind % W
        oy = torch.arange(Ho).view(1, 1, Ho, 1)
        ox = torch.arange(Wo).view(1, 1, 1, Wo)
        win = (2 * (iy - 2 * oy) + (ix - 2 * ox)).permute(0, 2, 3, 1)
    else:
        yr = F.avg_pool2d(xn, 2, 2)
    if relu:
        yr = torch.relu(yr)
    yr = yr.permute(0, 2, 3, 1)
    gate = yr > 0 if relu else torch.ones_like(yr, dtype=torch.bool)
    g_out = torch.where(gate, dyo, torch.zeros_like(dyo))
    dxr = torch.zeros(B, H, W, C, dtype=torch.float64)
    for q in range(4):
        dy_, dx_ = q >> 1, q & 1
        share = (g_out * (win == q)) if mode == 0 else g_out / 4
        dxr[:, dy_:2 * Ho:2, dx_:2 * Wo:2, :] = share
    if add:
        dxr += addt
    runs = {}
    layouts = ["vec", "scalar"] if (C % 4 == 0 and H % 2 == 0 and W % 2 == 0) else ["scalar"]
    for layout in layouts:
        y, idx, dx = _pool_call(lib, x, mode, relu, addt, dyo, layout)
        assert _same(y, yr), f"{layout}: pooled values differ"
        if mode == 0:
            assert torch.equal(idx.view(B, Ho, Wo, C).long(), win), f"{layout}: max-pool winners differ"
        assert _same(dx, dxr.float()), f"{layout}: dx differs"
        if add:
            if H % 2:
                assert torch.equal(dx[:, H - 1], addt[:, H - 1].float()), "trailing row != 0 + add"
            if W % 2:
                assert torch.equal(dx[:, :, W - 1], addt[:, :, W - 1].float()), "trailing column != 0 + add"
        elif H % 2 or W % 2:
            assert bool((dx[:, 2 * Ho:] == 0).all()) and bool((dx[:, :, 2 * Wo:] == 0).all())
        runs[layout] = (y, idx, dx)
    if len(runs) == 2:
        for a, b in zip(runs["vec"], runs["scalar"]):
            assert torch.equal(a.view(-1).view(torch.uint8), b.view(-1).view(torch.uint8)), "vector / scalar paths differ"


# ------------------------------------------------------------------------------------------------- OutConv
@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("npix", [1, 1000, 2 * 256 * 256])
@pytest.mark.parametrize("C", [16, 3, 5, 64, 256])
def test_conv1x1_c1(lib, C, npix, bias):
    """OutConv (nn.Conv2d(C, 1, 1)): tm_conv1x1_c1_forward, _dgrad and _wgrad against fp64, through the vector and the
    scalar layouts; the data gradient (one fp32 product per element) is exact and bit-identical between the paths;
    two weight-gradient calls are bit-identical."""
    torch.manual_seed(C + npix)
    x0 = torch.randn(npix, C, device=DEV)
    x0[::3] *= 1e-3
    w = torch.randn(C, device=DEV) * 0.2
    b = torch.randn(1, device=DEV) if bias else None
    dy0 = torch.randn(npix, device=DEV)
    yref = x0.double() @ w.double() + (b.double() if bias else 0.0)
    dxref = (dy0.double()[:, None] * w.double()).float()
    dwref = x0.double().t() @ dy0.double()
    dbref = dy0.double().sum()
    dxs = []
    for layout in ("vec", "scalar"):
        x, ldx = _strided(x0, layout)
        ybuf = torch.full((npix, 3), -5.0, device=DEV)
        lib.call("tm_conv1x1_c1_forward", npix, C, x, ldx, w, b, ybuf[:, 1], 3, lib.stream())
        assert_close(ybuf[:, 1], yref, 1e-5, 1e-5, f"{layout} OutConv forward")
        assert bool((ybuf[:, 0] == -5.0).all()) and bool((ybuf[:, 2] == -5.0).all())
        dybuf = torch.full((npix, 2), float("nan"), device=DEV)
        dybuf[:, 0] = dy0
        dx, dxbuf, lddx = _view(npix, C, layout, fill=-5.0)
        lib.call("tm_conv1x1_c1_dgrad", npix, C, dybuf[:, 0], 2, w, dx, lddx, lib.stream())
        assert torch.equal(dx, dxref), f"{layout} OutConv dgrad"
        assert int((dxbuf == -5.0).sum()) == dxbuf.numel() - dx.numel()
        dxs.append(dx)
        nb = lib.ws_bytes("tm_conv1x1_c1_wgrad_ws", C)
        dws = []
        for _ in range(2):
            dw = torch.empty(C, device=DEV)
            db = torch.empty(1, device=DEV) if bias else None
            lib.call("tm_conv1x1_c1_wgrad", npix, C, x, ldx, dybuf[:, 0], 2, dw, db, lib.workspace(nb, DEV), nb,
                     lib.stream())
            dws.append((dw, db))
        assert_close(dws[0][0], dwref, 1e-6, 1e-7, f"{layout} OutConv dw")
        if bias:
            assert_close(dws[0][1], dbref.view(1), 1e-6, 1e-7, f"{layout} OutConv dbias")
            assert torch.equal(dws[0][1], dws[1][1])
        assert torch.equal(dws[0][0], dws[1][0]), "OutConv wgrad is not deterministic"
    assert torch.equal(_bits(dxs[0]), _bits(dxs[1]))


# ------------------------------------------------------------------------------------------------- small helpers
@pytest.mark.parametrize("slope", [0.1, 0.0])
def test_leaky_relu(lib, slope):
    """tm_leaky_relu_forward / _backward: x > 0 ? x : slope x, and the gradient through the OUTPUT y, which must agree
    with PyTorch's gradient through the input at +-0, denormals and tiny negatives; compared bit for bit (signed
    zeros included)."""
    special = torch.tensor([0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.2e-38, -1.2e-38, -1e-30, 1.0, -1.0, -3.4e38,
                            3.4e38, 1e-7, -1e-7])
    x0 = torch.cat([special, torch.randn(100000) * torch.logspace(-30, 3, 100000)]).to(DEV)
    n = x0.numel()
    s64 = float(np.float32(slope))
    x64 = x0.double()
    yref = torch.where(x64 > 0, x64, x64 * s64).float()
    y = torch.empty(n, device=DEV)
    lib.call("tm_leaky_relu_forward", n, x0, slope, y, lib.stream())
    assert torch.equal(_bits(y), _bits(yref)), "leaky_relu forward"
    dy = torch.randn(n, device=DEV)
    dy[: special.numel()] = 1.5
    dxref = torch.where(x64 > 0, dy.double(), dy.double() * s64).float()
    dx = torch.empty(n, device=DEV)
    lib.call("tm_leaky_relu_backward", n, y, dy, slope, dx, lib.stream())
    assert torch.equal(_bits(dx), _bits(dxref)), "leaky_relu backward"


@pytest.mark.parametrize("T,w,gather", [(1, 1, False), (1350, 32, True), (40000, 128, True), (777, 5, False)])
def test_gather_cols(lib, T, w, gather):
    """tm_gather_cols: dst[i, col0:col0+w] = src[rows[i], 0:w] (the head's concat buffer); everything else untouched."""
    torch.manual_seed(T + w)
    lds, ldd, col0 = w + 3, w + 40, 17
    src = torch.randn(T + 9, lds, device=DEV)
    rows = torch.randint(0, T + 9, (T,), device=DEV, dtype=torch.int32) if gather else None
    dst = torch.full((T, ldd), 4.0, device=DEV)
    lib.call("tm_gather_cols", T, w, src, lds, rows, dst, ldd, col0, lib.stream())
    ref = src[rows.long(), :w] if gather else src[:T, :w]
    assert torch.equal(dst[:, col0:col0 + w], ref)
    assert bool((dst[:, :col0] == 4.0).all()) and bool((dst[:, col0 + w:] == 4.0).all())


@pytest.mark.parametrize("T,w,nrows", [(1, 1, 1), (1350, 32, 50), (40000, 128, 3000), (777, 5, 1)])
def test_scatter_add_cols(lib, T, w, nrows):
    """tm_scatter_add_cols: dst[rows[i], 0:w] += src[i, col0:col0+w] with repeated rows (all T onto one row in the
    last case), against fp64 index_add; columns past w untouched."""
    torch.manual_seed(T + w + nrows)
    lds, ldd, col0 = w + 40, w + 2, 23
    src = torch.randn(T, lds, device=DEV)
    rows = torch.randint(0, nrows, (T,), device=DEV, dtype=torch.int32)
    dst = torch.randn(nrows, ldd, device=DEV)
    ref = dst[:, :w].double().index_add(0, rows.long(), src[:, col0:col0 + w].double())
    tail = dst[:, w:].clone()
    lib.call("tm_scatter_add_cols", T, w, src, lds, col0, rows, dst, ldd, lib.stream())
    assert_close(dst[:, :w], ref, 1e-5, 1e-5, "scatter_add_cols")
    assert torch.equal(dst[:, w:], tail)
