"""tf32x3 forms of the TMA-fed tcgen05 convolutions (tm_conv3x3_tf32*, tm_convt2x2_tf32*, csrc/tm_tma.cu) against fp64.

The operands are fp32 with non-zero low mantissa bits, spread over four orders of magnitude, so the lo planes
matter: 3xTF32 (hi*hi + hi*lo + lo*hi) lands near 1e-6 of the output's scale, single-pass TF32 -- or any of the
three products dropped -- near 1e-4.  The bar, 2e-5 of the scale, separates the two."""
import pytest
import torch
import torch.nn.functional as F

from conftest import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"
BAR = 2e-5          # max |err| / max |ref|
WORST = {}          # worst error per kernel, printed with -s


@pytest.fixture(scope="module")
def lib(pkg):
    import tm_lib
    return tm_lib


def _data(*shape, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    mag = 10.0 ** (torch.rand(*shape, generator=g, device=DEV) * 4 - 2)       # 1e-2 .. 1e2
    return torch.randn(*shape, generator=g, device=DEV) * mag


def _check(got, ref, name):
    ref = ref.double()
    scale = float(ref.abs().max())
    err = float((got.double() - ref).abs().max()) / scale
    WORST[name] = max(WORST.get(name, 0.0), err)
    assert err <= BAR, f"{name}: max |err| = {err:.3e} of the scale (bar {BAR:.0e})"


def _nhwc(t):
    return t.detach().permute(0, 2, 3, 1).reshape(-1, t.shape[1])


def _strided(t, C, ld, off):
    """t [npix][C] copied into columns off .. off+C of a [npix][ld] buffer of NaNs: a strided (concat-half) view."""
    buf = torch.full((t.shape[0], ld), float("nan"), device=DEV)
    buf[:, off:off + C] = t
    return buf[:, off:off + C]


# every 3x3 layer of the U-Net at 256 x 256 (B, H, W, Cin, Cout), then small shapes: batch tails, split K
UNET_256 = [(1, 256, 256, 3, 16), (1, 256, 256, 16, 16), (1, 128, 128, 16, 32), (1, 128, 128, 32, 32),
            (1, 64, 64, 32, 64), (1, 64, 64, 64, 64), (1, 32, 32, 64, 128), (1, 32, 32, 128, 128),
            (1, 64, 64, 128, 64), (1, 128, 128, 64, 32), (1, 256, 256, 32, 16)]
SMALL = [(3, 8, 8, 32, 16), (3, 16, 16, 64, 128), (3, 4, 4, 128, 128), (3, 16, 32, 16, 32), (2, 8, 16, 3, 16)]


@pytest.mark.parametrize("B,H,W,Cin,Cout", UNET_256 + SMALL)
def test_conv3x3_tf32_tma(lib, B, H, W, Cin, Cout):
    CinP = max(16, (Cin + 15) // 16 * 16)
    assert lib.ws_bytes("tm_conv3x3_tf32_supported", B, H, W, CinP, Cout) == 1
    seed = B * 7 + H + W + Cin + Cout
    x = _data(B, Cin, H, W, seed=seed).requires_grad_(True)
    w = (_data(Cout, Cin, 3, 3, seed=seed + 1) * 0.01).requires_grad_(True)
    g = _data(B, Cout, H, W, seed=seed + 2)
    bias = _data(Cout, seed=seed + 3)
    ref = F.conv2d(x.double(), w.double(), None, padding=1)
    gx, gw = torch.autograd.grad(ref, (x, w), g.double())
    npix = B * H * W
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    ws = lambda nb: lib.workspace(nb, DEV) if nb else None          # noqa: E731
    # input: 16 zero-padded channels for the 3-channel image; P == 1 layers read a strided (concat-half) view
    P = lib.ws_bytes("tm_conv3x3_tf32_pack", W, CinP, Cout)
    xr = torch.zeros(npix, CinP, device=DEV)
    xr[:, :Cin] = _nhwc(x)
    xv, ldx = (xr, CinP) if P > 1 else (_strided(xr, CinP, 2 * CinP, CinP), 2 * CinP)
    wf = torch.empty(9, P * Cout, P * CinP, device=DEV)
    lib.call("tm_conv3x3_pack_f32", Cout, Cin, w.detach().contiguous(), wf, P, CinP, 0, lib.stream())
    nb = lib.ws_bytes("tm_conv3x3_tf32_ws", B, H, W, CinP, Cout, P)
    # ---- forward with bias + ReLU into the second half of a concat-style buffer
    ybuf = torch.full((npix, 2 * Cout), 7.0, device=DEV)
    lib.call("tm_conv3x3_tf32", B, H, W, CinP, Cout, P, xv, ldx, wf, bias, ybuf[:, Cout:], 2 * Cout, 2, None, ws(nb), nb,
             err, lib.stream())
    refy = _nhwc(ref)
    _check(ybuf[:, Cout:], torch.relu(refy + bias.double()), "fprop")
    assert bool((ybuf[:, :Cout] == 7.0).all())
    y2 = torch.empty_like(ybuf)
    lib.call("tm_conv3x3_tf32", B, H, W, CinP, Cout, P, xv, ldx, wf, bias, y2[:, Cout:], 2 * Cout, 2, None, ws(nb), nb,
             err, lib.stream())
    assert torch.equal(ybuf[:, Cout:], y2[:, Cout:]), "forward is not bit-deterministic"
    # ---- unsplit launches: batch-norm statistics from the epilogue
    if nb == 0 and P * Cout <= 128:
        ns = lib.ws_bytes("tm_conv3x3_bf16_stats_bytes", Cout, P)
        stats = torch.empty(ns // 8, dtype=torch.float64, device=DEV)
        y3 = torch.empty(npix, Cout, device=DEV)
        lib.call("tm_conv3x3_tf32", B, H, W, CinP, Cout, P, xv, ldx, wf, None, y3, Cout, 0, stats, None, 0, err, lib.stream())
        _check(y3, refy, "fprop")
        got = stats.reshape(-1, Cout, 2).sum(0)
        assert_close(got[:, 0], refy.sum(0), 1e-4, 1e-5, "fused BN sum")
        assert_close(got[:, 1], (refy * refy).sum(0), 1e-4, 1e-5, "fused BN sum of squares")
    # ---- data gradient: the forward kernel on dy with the reversed-tap weights, output into a concat half
    gr = _nhwc(g).contiguous()
    if Cin % 16 == 0:
        Pd = lib.ws_bytes("tm_conv3x3_tf32_pack", W, Cout, Cin)
        wd = torch.empty(9, Pd * Cin, Pd * Cout, device=DEV)
        lib.call("tm_conv3x3_pack_f32", Cout, Cin, w.detach().contiguous(), wd, Pd, Cout, 1, lib.stream())
        nbd = lib.ws_bytes("tm_conv3x3_tf32_ws", B, H, W, Cout, Cin, Pd)
        dx = torch.full((npix, 2 * Cin), 7.0, device=DEV)
        lib.call("tm_conv3x3_tf32", B, H, W, Cout, Cin, Pd, gr, Cout, wd, None, dx[:, :Cin], 2 * Cin, 0, None, ws(nbd), nbd,
                 err, lib.stream())
        _check(dx[:, :Cin], _nhwc(gx), "dgrad")
        assert bool((dx[:, Cin:] == 7.0).all())
    # ---- weight gradient
    nbw = lib.ws_bytes("tm_conv3x3_tf32_wgrad_ws", B, H, W, CinP, Cout)
    dw = torch.empty(Cout, Cin, 3, 3, device=DEV)
    lib.call("tm_conv3x3_tf32_wgrad", B, H, W, CinP, Cin, Cout, xr, CinP, gr, Cout, dw, ws(nbw), nbw, err, lib.stream())
    _check(dw, gw, "wgrad")
    dw2 = torch.empty_like(dw)
    lib.call("tm_conv3x3_tf32_wgrad", B, H, W, CinP, Cin, Cout, xr, CinP, gr, Cout, dw2, ws(nbw), nbw, err, lib.stream())
    assert torch.equal(dw, dw2), "weight gradient is not bit-deterministic"
    assert int(err.item()) == 0


# the U-Net's transposed convolutions at 256 x 256 (input maps 32 / 64 / 128), then a batch tail
@pytest.mark.parametrize("B,H,W,Cin,Cout", [(1, 32, 32, 128, 64), (1, 64, 64, 64, 32), (1, 128, 128, 32, 16),
                                            (3, 4, 4, 64, 32), (3, 8, 4, 128, 64)])
def test_convt2x2_tf32_tma(lib, B, H, W, Cin, Cout):
    assert lib.ws_bytes("tm_convt2x2_tf32_supported", B, H, W, Cin, Cout) == 1
    seed = B + H + W + Cin + Cout
    x = _data(B, Cin, H, W, seed=seed).requires_grad_(True)
    w = (_data(Cin, Cout, 2, 2, seed=seed + 1) * 0.01).requires_grad_(True)
    bias = _data(Cout, seed=seed + 2)
    g = _data(B, Cout, 2 * H, 2 * W, seed=seed + 3)
    ref = F.conv_transpose2d(x.double(), w.double(), bias.double(), stride=2)
    gx, gw = torch.autograd.grad(ref, (x, w), g.double())
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    nb = lib.ws_bytes("tm_convt2x2_tf32_ws", B, H, W, Cin, Cout)
    wsb = lib.workspace(nb, DEV) if nb else None
    wf = torch.empty(4 * Cout, Cin, device=DEV)
    wd = torch.empty(4, Cin, Cout, device=DEV)
    lib.call("tm_convt2x2_pack_f32", Cin, Cout, w.detach().contiguous(), wf, wd, lib.stream())
    xr = _nhwc(x).contiguous()
    # forward: scatter epilogue into the second half of a concat buffer
    ybuf = torch.full((B * 4 * H * W, 2 * Cout), 7.0, device=DEV)
    lib.call("tm_convt2x2_tf32", B, H, W, Cin, Cout, xr, Cin, wf, bias, ybuf[:, Cout:], 2 * Cout, wsb, nb, err, lib.stream())
    _check(ybuf[:, Cout:], _nhwc(ref), "convT fwd")
    assert bool((ybuf[:, :Cout] == 7.0).all())
    # data and weight gradient read dy from a concat half (pixel stride 2 * Cout)
    gv = _strided(_nhwc(g), Cout, 2 * Cout, Cout)
    dx = torch.empty(B * H * W, Cin, device=DEV)
    lib.call("tm_convt2x2_tf32_dgrad", B, H, W, Cin, Cout, gv, 2 * Cout, wd, dx, Cin, wsb, nb, err, lib.stream())
    _check(dx, _nhwc(gx), "convT dgrad")
    if lib.ws_bytes("tm_convt2x2_tf32_wgrad_supported", B, H, W, Cin, Cout) == 1:
        dw = torch.empty(Cin, Cout, 2, 2, device=DEV)
        lib.call("tm_convt2x2_tf32_wgrad", B, H, W, Cin, Cout, xr, Cin, gv, 2 * Cout, dw, wsb, nb, err, lib.stream())
        _check(dw, gw, "convT wgrad")
        dw2 = torch.empty_like(dw)
        lib.call("tm_convt2x2_tf32_wgrad", B, H, W, Cin, Cout, xr, Cin, gv, 2 * Cout, dw2, wsb, nb, err, lib.stream())
        assert torch.equal(dw, dw2), "convT weight gradient is not bit-deterministic"
    else:
        assert Cout % 32, "the weight gradient should take every shape with 32-channel multiples"
    assert int(err.item()) == 0


def test_unet_tf32_tma_route_matches_cp_async_route(lib):
    """The whole U-Net in tf32x3 mode on the TMA kernels against the cp.async tf_gemm route: outputs and gradients
    within the fp32-class bar (gradients allow the rows of ReLU gates that sit within rounding of zero)."""
    import Unet as U
    import tm_unet
    torch.manual_seed(11)
    net = U.UNet("max").train().to(DEV)
    x = torch.rand(2, 3, 128, 128, device=DEV)
    g = torch.randn(2, 1, 64, 64, device=DEV)
    old_math, old_tma = tm_unet.MATH, tm_unet.USE_TMA
    res = {}
    try:
        tm_unet.MATH = "tf32x3"
        for tma in (True, False):
            tm_unet.USE_TMA = tma
            out, st = tm_unet.unet_forward(net, x, need_bwd=True, update_stats=False)
            assert all(bool(st[k].get("tf")) == tma for k in ("enc0", "enc1", "enc2", "enc3", "dec0", "dec1", "dec2"))
            assert (st["up0"].get("wdf") is not None) == tma
            res[tma] = (out.clone(), {k: v.clone() for k, v in tm_unet.unet_backward(net, st, g).items()})
    finally:
        tm_unet.MATH, tm_unet.USE_TMA = old_math, old_tma
    assert_close(res[True][0], res[False][0], 1e-3, 1e-4, "unet out, TMA vs cp.async route")
    for k, r in res[False][1].items():
        assert_close(res[True][1][k], r, 1e-3, 2e-4, f"grad {k}, TMA vs cp.async route", flip_frac=2e-3)
    lib.check_err_flags()


def test_report_worst_errors():
    """Runs last in this module: prints the worst error of every kernel (pytest -s)."""
    for k, v in sorted(WORST.items()):
        print(f"tf32x3 TMA {k}: worst max|err| / max|ref| = {v:.2e}")
