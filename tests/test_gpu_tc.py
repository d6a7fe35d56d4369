"""tcgen05 / TMEM kernels (tm_tc_*) against fp64 PyTorch references.

precision 3 (3xTF32, the default) and 2 (bf16 x6) must meet the fp32 bar (rtol 1e-3; checked much tighter here);
precision 1 (split bf16 x3) rtol 1e-3; precision 0 (plain bf16) and 4 (single TF32) the bf16 bar (rtol 2e-2)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {3: (1e-4, 2e-5), 2: (1e-4, 1e-5), 1: (1e-3, 1e-4), 0: (2e-2, 1e-2), 4: (2e-2, 1e-2)}


@pytest.fixture(scope="module")
def lib(pkg):
    import tm_lib
    return tm_lib


def _err():
    return torch.zeros(1, dtype=torch.int32, device=DEV)


@pytest.mark.parametrize("precision", [3, 4, 2, 1, 0])
@pytest.mark.parametrize("M,N,K,b_is_nk", [(128, 32, 64, 1), (300, 256, 36, 1), (1000, 128, 256, 1), (257, 100, 130, 0),
                                           (1350, 576, 288, 1), (77, 1, 576, 1), (500, 256, 2, 1)])
def test_tc_gemm_nn(lib, M, N, K, b_is_nk, precision):
    torch.manual_seed(M + N + K)
    A = torch.randn(M + 3, K, device=DEV)
    B = torch.randn(N, K, device=DEV) if b_is_nk else torch.randn(K, N, device=DEV)
    bias = torch.randn(N, device=DEV)
    rows = torch.randperm(M + 3, device=DEV)[:M].to(torch.int32)
    C = torch.full((M + 3, N), 7.0, device=DEV)
    err = _err()
    lib.call("tm_tc_gemm_nn", M, N, K, A, K, rows, B, B.shape[1], b_is_nk, C, N, rows, bias, None, 0, 1 | 2,
             precision, err, lib.stream())
    Bm = B.double().t() if b_is_nk else B.double()
    ref = torch.relu(A[rows.long()].double() @ Bm + bias.double())
    assert int(err.item()) == 0
    assert_close(C[rows.long()], ref, *TOL[precision], "tc_gemm_nn")
    untouched = torch.ones(M + 3, dtype=torch.bool, device=DEV)
    untouched[rows.long()] = False
    assert bool((C[untouched] == 7.0).all())


@pytest.mark.parametrize("precision", [3, 4, 2, 1, 0])
@pytest.mark.parametrize("M,N,R", [(128, 256, 5000), (256, 36, 3001), (1, 576, 1350), (27, 16, 4096), (256, 128, 20000)])
def test_tc_gemm_tn(lib, M, N, R, precision):
    torch.manual_seed(M + N + R)
    A = torch.randn(R + 3, M, device=DEV)
    B = torch.randn(R + 3, N, device=DEV)
    rows = torch.randperm(R + 3, device=DEV)[:R].to(torch.int32)
    C = torch.empty(M, N, device=DEV)
    nb = lib.ws_bytes("tm_tc_gemm_tn_ws", M, N, R)
    ws = lib.workspace(nb, DEV)
    err = _err()
    lib.call("tm_tc_gemm_tn", M, N, R, A, M, rows, B, N, rows, C, N, 0, precision, ws, nb, err, lib.stream())
    ref = A[rows.long()].double().t() @ B[rows.long()].double()
    assert int(err.item()) == 0
    assert_close(C, ref, *TOL[precision], "tc_gemm_tn")


@pytest.mark.parametrize("precision", [3, 4, 2, 1, 0])
@pytest.mark.parametrize("B,H,W,Cin,Cout,k", [(1, 16, 16, 3, 16, 3), (2, 8, 24, 16, 32, 3), (1, 16, 8, 128, 64, 3),
                                              (1, 12, 12, 2, 32, 9), (1, 16, 16, 16, 1, 1), (1, 32, 32, 64, 128, 3)])
def test_tc_conv(lib, B, H, W, Cin, Cout, k, precision):
    torch.manual_seed(B * H + Cin + Cout + k)
    x = torch.randn(B, Cin, H, W, device=DEV, requires_grad=True)
    w = (torch.randn(Cout, Cin, k, k, device=DEV) * 0.1).requires_grad_(True)
    bias = torch.randn(Cout, device=DEV)
    ref = F.conv2d(x.double(), w.double(), bias.double(), padding=k // 2)
    g = torch.randn(B, Cout, H, W, device=DEV)
    gx, gw = torch.autograd.grad(ref, (x, w), g.double())
    nhwc = lambda t: t.detach().permute(0, 2, 3, 1).contiguous()            # noqa: E731
    xs, gs = nhwc(x), nhwc(g)
    wf = torch.empty(k * k * Cin, Cout, device=DEV)
    wb = torch.empty(k * k * Cout, Cin, device=DEV)
    lib.call("tm_conv_pack_weight", Cout, Cin, k, w.detach().contiguous(), wf, wb, lib.stream())
    err = _err()
    y = torch.empty(B, H, W, Cout, device=DEV)
    lib.call("tm_tc_conv2d_nhwc", B, H, W, Cin, Cout, k, xs, Cin, wf, bias, y, Cout, 0, precision, err, lib.stream())
    assert_close(y.permute(0, 3, 1, 2), ref, *TOL[precision], "tc fprop")
    dx = torch.empty(B, H, W, Cin, device=DEV)
    lib.call("tm_tc_conv2d_nhwc", B, H, W, Cout, Cin, k, gs, Cout, wb, None, dx, Cin, 0, precision, err, lib.stream())
    assert_close(dx.permute(0, 3, 1, 2), gx, *TOL[precision], "tc dgrad")
    nb = lib.ws_bytes("tm_tc_conv2d_wgrad_ws", B, H, W, Cin, Cout, k)
    dwf = torch.empty(k * k * Cin, Cout, device=DEV)
    lib.call("tm_tc_conv2d_wgrad_nhwc", B, H, W, Cin, Cout, k, xs, Cin, gs, Cout, dwf, precision,
             lib.workspace(nb, DEV), nb, err, lib.stream())
    dw = torch.empty(Cout, Cin, k, k, device=DEV)
    lib.call("tm_conv_unpack_wgrad", Cout, Cin, k, dwf, dw, lib.stream())
    assert_close(dw, gw, *TOL[precision], "tc wgrad")
    assert int(err.item()) == 0


@pytest.mark.parametrize("precision", [3, 4])
@pytest.mark.parametrize("B,H,W,Cin,Cout,k,relu", [(1, 32, 32, 128, 128, 3, False), (1, 64, 64, 64, 64, 3, True),
                                                   (1, 32, 32, 256, 64, 3, False), (2, 16, 16, 64, 128, 3, False),
                                                   (1, 256, 256, 16, 16, 3, False)])
def test_tc_conv_splitk(lib, B, H, W, Cin, Cout, k, relu, precision):
    """tm_tc_conv2d_nhwc_splitk: the K = 9 Cin range split over CTAs on the small deep maps of one 256 x 256 design
    (forward and the data gradient through the same entry), bias / ReLU applied by the folding pass, into a strided
    output (a concat buffer); the last shape is large enough that no split is chosen (workspace size 0)."""
    torch.manual_seed(H + Cin + Cout)
    x = torch.randn(B, Cin, H, W, device=DEV)
    w = torch.randn(Cout, Cin, k, k, device=DEV) * 0.05
    bias = torch.randn(Cout, device=DEV)
    ref = F.conv2d(x.double(), w.double(), bias.double(), padding=k // 2)
    if relu:
        ref = ref.relu()
    xs = x.permute(0, 2, 3, 1).contiguous()
    wf = torch.empty(k * k * Cin, Cout, device=DEV)
    wb = torch.empty(k * k * Cout, Cin, device=DEV)
    lib.call("tm_conv_pack_weight", Cout, Cin, k, w.contiguous(), wf, wb, lib.stream())
    err = _err()
    ldy = Cout + 8
    y = torch.full((B, H, W, ldy), 7.0, device=DEV)
    nb = lib.ws_bytes("tm_tc_conv2d_splitk_ws", B, H, W, Cin, Cout, k, precision)
    assert (nb == 0) == (H * W * B >= 148 * 128 // 2)
    lib.call("tm_tc_conv2d_nhwc_splitk", B, H, W, Cin, Cout, k, xs, Cin, wf, bias, y, ldy, 2 if relu else 0, precision,
             lib.workspace(nb, DEV) if nb else None, nb, err, lib.stream())
    assert_close(y[..., :Cout].permute(0, 3, 1, 2), ref, *TOL[precision], "split-K fprop")
    assert bool((y[..., Cout:] == 7.0).all()), "columns past Cout were touched"
    assert int(err.item()) == 0


@pytest.mark.parametrize("R,C,gather", [(5000, 128, False), (70001, 256, True), (3, 128, False), (4097, 36, False), (300, 130, True)])
def test_colsum(lib, R, C, gather):
    """tm_colsum: vectorised path (C % 4 == 0, 256-row chunks) and the scalar fall-back, with and without a row list,
    accumulate on and off, bit-deterministic."""
    torch.manual_seed(R + C)
    X = torch.randn(R + 50, C, device=DEV)
    rows = torch.randint(0, R + 50, (R,), device=DEV, dtype=torch.int32) if gather else None
    ref = (X[rows.long()] if gather else X[:R]).double().sum(0)
    nb = lib.ws_bytes("tm_colsum_ws", R, C)
    out = torch.full((C,), 3.0, device=DEV)
    lib.call("tm_colsum", R, C, X, C, rows, out, 0, lib.workspace(nb, DEV), nb, lib.stream())
    assert_close(out, ref, 1e-5, 1e-4, "colsum")
    out2 = torch.full((C,), 3.0, device=DEV)
    lib.call("tm_colsum", R, C, X, C, rows, out2, 1, lib.workspace(nb, DEV), nb, lib.stream())
    assert_close(out2, ref + 3.0, 1e-5, 1e-4, "colsum accumulate")
    out3 = torch.empty(C, device=DEV)
    lib.call("tm_colsum", R, C, X, C, rows, out3, 0, lib.workspace(nb, DEV), nb, lib.stream())
    assert torch.equal(out, out3)


@pytest.mark.parametrize("M,kx,gather,xscale", [(1000, 2, False, 1.0), (40000, 2, True, 1.0), (129, 1, True, 30.0),
                                                 (5000, 2, False, 1e-4), (70000, 2, True, 1e3)])
def test_selfmlp_gen_forward(lib, M, kx, gather, xscale):
    """tm_selfmlp_gen_forward (Linear(kx,256) -> ReLU -> Linear(256,128), hidden layer generated into fp16 two-term
    split tcgen05 operands): against the fp64 definition at the fp32-class bar, inputs of very different magnitudes
    (the per-row scale), gathered / scattered rows, untouched rows stay untouched."""
    torch.manual_seed(M + kx)
    n_src, n_dst = M + 77, M + 33
    X = torch.randn(n_src, kx, device=DEV) * xscale
    W1 = torch.randn(256, kx, device=DEV) * 0.5
    b1 = torch.randn(256, device=DEV) * 0.3
    W2 = torch.randn(128, 256, device=DEV) * 0.1
    b2 = torch.randn(128, device=DEV) * 0.1
    xr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    orow = torch.randperm(n_dst, device=DEV)[:M].int().contiguous() if gather else None
    xs = X[xr.long()] if gather else X[:M]
    ref = (xs.double() @ W1.double().t() + b1.double()).relu() @ W2.double().t() + b2.double()
    out = torch.full((n_dst, 128), -5.0, device=DEV)
    nb = lib.ws_bytes("tm_selfmlp_ws_bytes")
    lib.call("tm_selfmlp_gen_forward", M, X, kx, xr, kx, W1, b1, W2, b2, out, 128, orow, lib.workspace(nb, DEV), nb, lib.stream())
    got = out[orow.long()] if gather else out[:M]
    assert_close(got, ref, 1e-4, 2e-5, "fused self MLP")
    touched = torch.zeros(n_dst, dtype=torch.bool, device=DEV)
    touched[orow.long() if gather else torch.arange(M, device=DEV)] = True
    assert bool((out[~touched] == -5.0).all())
    out2 = torch.full((n_dst, 128), -5.0, device=DEV)
    lib.call("tm_selfmlp_gen_forward", M, X, kx, xr, kx, W1, b1, W2, b2, out2, 128, orow, lib.workspace(nb, DEV), nb, lib.stream())
    assert torch.equal(out, out2)


@pytest.mark.parametrize("M,kx,gather,gscale", [(1000, 2, False, 1.0), (40000, 2, True, 1e-4), (63, 1, True, 1.0),
                                                 (70001, 2, True, 1e-8), (20000, 2, False, 1e3)])
def test_selfmlp_gen_wgrad2(lib, M, kx, gather, gscale):
    """tm_selfmlp_gen_wgrad2 (dW2 = G^T relu(W1 x + b1), hidden layer generated, contraction over the rows on
    tcgen05 with global power-of-two operand scales) and tm_colsum_absmax (bias gradient + max |G| in one pass):
    against the fp64 definition at the fp32-class bar, gradients of very different magnitudes, rows of G that differ
    by six orders of magnitude, gathered rows, bit-deterministic."""
    torch.manual_seed(M + kx)
    n_src = M + 55
    X = torch.randn(n_src, kx, device=DEV)
    W1 = torch.randn(256, kx, device=DEV) * 0.5
    b1 = torch.randn(256, device=DEV) * 0.3
    G = torch.randn(n_src, 128, device=DEV) * gscale
    G[::7] *= 1e-6                                   # rows far below the global scale
    xr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    gr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    xs = X[xr.long()] if gather else X[:M]
    gs = G[gr.long()] if gather else G[:M]
    h = (xs.double() @ W1.double().t() + b1.double()).relu()
    ref = gs.double().t() @ h
    db = torch.empty(128, device=DEV)
    gmax = torch.empty(1, device=DEV)
    nbc = lib.ws_bytes("tm_colsum_ws", M, 128)
    lib.call("tm_colsum_absmax", M, 128, G, 128, gr, db, gmax, lib.workspace(nbc, DEV), nbc, lib.stream())
    assert float(gmax.item()) == float(gs.abs().max().item())
    assert_close(db, gs.double().sum(0), 1e-4, 1e-4, "bias gradient")
    nb = lib.ws_bytes("tm_selfmlp_wgrad2_ws_bytes")
    dw = torch.empty(128, 256, device=DEV)
    lib.call("tm_selfmlp_gen_wgrad2", M, G, 128, gr, X, kx, xr, kx, W1, b1, gmax, dw, lib.workspace(nb, DEV), nb, lib.stream())
    assert_close(dw, ref, 1e-4, 2e-5, "fused dW2")
    dw2 = torch.empty(128, 256, device=DEV)
    lib.call("tm_selfmlp_gen_wgrad2", M, G, 128, gr, X, kx, xr, kx, W1, b1, gmax, dw2, lib.workspace(nb, DEV), nb, lib.stream())
    assert torch.equal(dw, dw2)


@pytest.mark.parametrize("M,kx,gather,gscale", [(1000, 2, False, 1.0), (40000, 2, True, 1e-4), (129, 1, True, 1.0),
                                                 (70001, 2, True, 1e-8)])
def test_selfmlp_gen_bwd1(lib, M, kx, gather, gscale):
    """tm_selfmlp_gen_bwd1: db1 / dW1 of Linear(kx,256) -> ReLU -> Linear(256,128) from dh = (G W2) * (pre > 0), dh
    never stored; against the fp64 definition (mask taken from the fp32 pre-activation, as the forward takes it)."""
    torch.manual_seed(M + 3 * kx)
    n_src = M + 41
    X = torch.randn(n_src, kx, device=DEV)
    W1 = torch.randn(256, kx, device=DEV) * 0.5
    b1 = torch.randn(256, device=DEV) * 0.3
    W2 = torch.randn(128, 256, device=DEV) * 0.1
    G = torch.randn(n_src, 128, device=DEV) * gscale
    G[::5] *= 1e-5
    xr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    gr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    xs = X[xr.long()] if gather else X[:M]
    gs = G[gr.long()] if gather else G[:M]
    pre = xs.double() @ W1.double().t() + b1.double()
    dh = (gs.double() @ W2.double()) * (pre > 0)
    ref_db = dh.sum(0)
    ref_dw = dh.t() @ xs.double()
    nb = lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")
    dW1 = torch.empty(256, kx, device=DEV)
    db1 = torch.empty(256, device=DEV)
    lib.call("tm_selfmlp_gen_bwd1", M, G, 128, gr, X, kx, xr, kx, W1, b1, W2, dW1, db1, lib.workspace(nb, DEV), nb, lib.stream())
    assert_close(db1, ref_db, 1e-3, 2e-4, "db1", max_bad=4)          # (a gate at |pre| ~ 1 ulp may go either way)
    assert_close(dW1, ref_dw, 1e-3, 2e-4, "dW1", max_bad=8)
    dW1b, db1b = torch.empty_like(dW1), torch.empty_like(db1)
    lib.call("tm_selfmlp_gen_bwd1", M, G, 128, gr, X, kx, xr, kx, W1, b1, W2, dW1b, db1b, lib.workspace(nb, DEV), nb, lib.stream())
    assert torch.equal(dW1, dW1b) and torch.equal(db1, db1b)


@pytest.mark.parametrize("M,gather,gscale", [(1000, False, 1.0), (40000, True, 1e-5), (129, True, 1.0)])
def test_selfmlp_rows_dh(lib, M, gather, gscale):
    """tm_selfmlp_rows_dh: DH[r] = (G[g_rows] W2) * (H[r] > 0) with r through a row list (the cone's rows of a larger
    hidden matrix); rows outside the list stay untouched."""
    torch.manual_seed(M)
    n_src, n_h = M + 41, M + 29
    W2 = torch.randn(128, 256, device=DEV) * 0.1
    G = torch.randn(n_src, 128, device=DEV) * gscale
    G[::3] *= 1e-4
    H = torch.randn(n_h, 256, device=DEV).relu_()
    gr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    hr = torch.randperm(n_h, device=DEV)[:M].int().contiguous() if gather else None
    gs = G[gr.long()] if gather else G[:M]
    hs = H[hr.long()] if gather else H[:M]
    ref = (gs.double() @ W2.double()) * (hs > 0)
    DH = torch.full((n_h, 256), 9.0, device=DEV)
    nb = lib.ws_bytes("tm_selfmlp_rows_dh_ws_bytes")
    lib.call("tm_selfmlp_rows_dh", M, G, 128, gr, W2, H, 256, hr, DH, 256, lib.workspace(nb, DEV), nb, lib.stream())
    got = DH[hr.long()] if gather else DH[:M]
    assert_close(got, ref, 1e-4, 2e-5, "dh")
    touched = torch.zeros(n_h, dtype=torch.bool, device=DEV)
    touched[hr.long() if gather else torch.arange(M, device=DEV)] = True
    assert bool((DH[~touched] == 9.0).all())


@pytest.mark.parametrize("M,kin,gather,xscale", [(1000, 36, False, 1.0), (40000, 36, True, 1e-3), (129, 48, True, 50.0), (777, 4, False, 1.0)])
def test_selfmlp_lin1_relu(lib, M, kin, gather, xscale):
    """tm_selfmlp_lin1_relu: HID = relu(X[x_rows] W1^T + b1) for up to 48 inputs (fc_cell_self: 36), fp32-class."""
    torch.manual_seed(M + kin)
    n_src = M + 19
    X = torch.randn(n_src, kin, device=DEV) * xscale
    X[::4] *= 1e-3
    W1 = torch.randn(256, kin, device=DEV) * 0.3
    b1 = torch.randn(256, device=DEV) * 0.2
    xr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    xs = X[xr.long()] if gather else X[:M]
    ref = (xs.double() @ W1.double().t() + b1.double()).relu()
    H = torch.full((M + 5, 256), -3.0, device=DEV)
    nb = lib.ws_bytes("tm_selfmlp_lin1_ws_bytes")
    rowmax = torch.full((M,), -1.0, device=DEV)
    lib.call("tm_selfmlp_lin1_relu", M, X, kin, xr, kin, W1, b1, H, 256, rowmax, lib.workspace(nb, DEV), nb, lib.stream())
    assert_close(H[:M], ref, 1e-4, 2e-5, "lin1")
    assert bool((H[M:] == -3.0).all())
    assert torch.equal(rowmax, H[:M].max(dim=1).values)
    # second layer from the stored hidden rows, scattered output
    W2 = torch.randn(128, 256, device=DEV) * 0.1
    b2 = torch.randn(128, device=DEV) * 0.1
    orow = torch.randperm(M + 7, device=DEV)[:M].int().contiguous() if gather else None
    out = torch.full((M + 7, 128), 6.0, device=DEV)
    nb2 = lib.ws_bytes("tm_selfmlp_ws_bytes")
    lib.call("tm_selfmlp_rows_forward", M, H, 256, None, rowmax, W2, b2, out, 128, orow, lib.workspace(nb2, DEV), nb2, lib.stream())
    ref2 = H[:M].double() @ W2.double().t() + b2.double()
    assert_close(out[orow.long()] if gather else out[:M], ref2, 1e-4, 2e-5, "rows_forward")
    touched = torch.zeros(M + 7, dtype=torch.bool, device=DEV)
    touched[orow.long() if gather else torch.arange(M, device=DEV)] = True
    assert bool((out[~touched] == 6.0).all())


@pytest.mark.parametrize("M,K,gather,relu", [(1350, 256, False, False), (77, 130, True, True), (5, 3, False, False)])
def test_rowdot(lib, M, K, gather, relu):
    """tm_rowdot: nn.Linear(K, 1) forward, one warp per row (vector and scalar paths, gathered / scattered rows)."""
    torch.manual_seed(M + K)
    X = torch.randn(M + 9, K, device=DEV)
    w = torch.randn(K, device=DEV)
    b = torch.randn(1, device=DEV)
    ar = torch.randperm(M + 9, device=DEV)[:M].int().contiguous() if gather else None
    cr = torch.randperm(M + 4, device=DEV)[:M].int().contiguous() if gather else None
    xs = X[ar.long()] if gather else X[:M]
    ref = xs.double() @ w.double() + b.double()
    if relu:
        ref = ref.relu()
    out = torch.full((M + 4, 2), 4.0, device=DEV)
    lib.call("tm_rowdot", M, K, X, K, ar, w, b, out, 2, cr, 1 if relu else 0, lib.stream())
    got = out[cr.long(), 0] if gather else out[:M, 0]
    assert_close(got, ref, 1e-5, 1e-5, "rowdot")
    assert bool((out[:, 1] == 4.0).all())


def _mlp_inputs(M, kx, hid, nout, seed, n_src):
    """Rows as mlp_alpha and fc_net_self see them: integer level ids in [0, 200] in half of the rows, floats of
    magnitude 1e-3 .. 50 in the others.  Hidden units 0 .. 7 read only the first input with W1 = 0.5 and
    b1 = -0.5 x0 for an integer x0: their pre-activation is exactly 0 on every row whose first input is x0."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    X = torch.randint(0, 201, (n_src, kx), device=DEV, generator=g).float()
    fl = torch.rand(n_src, device=DEV, generator=g) < 0.5
    scale = torch.logspace(-3, float(np.log10(50.0)), n_src, device=DEV)[torch.randperm(n_src, device=DEV, generator=g)]
    X[fl] = (torch.randn(n_src, kx, device=DEV, generator=g) * scale[:, None])[fl]
    X[::5, 0] = 0.0                                      # level 0 ...
    X[1::5, 0] = 17.0                                    # ... and 17 on many rows
    W1 = torch.randn(hid, kx, device=DEV, generator=g) * 0.5
    b1 = torch.randn(hid, device=DEV, generator=g) * 0.3
    W1[:8] = 0.0
    W1[:8, 0] = 0.5
    b1[:8] = -0.5 * torch.tensor([0.0, 17.0, 0.0, 17.0, 3.0, 200.0, 17.0, 0.0], device=DEV)
    W2 = torch.randn(nout, hid, device=DEV, generator=g) * (1.0 / hid ** 0.5)
    b2 = torch.randn(nout, device=DEV, generator=g) * 0.1
    return X, W1, b1, W2, b2


MLP_SHAPES = [(1, 64, 32), (1, 128, 64), (2, 256, 128)]


@pytest.mark.parametrize("precision", [3, 4, 2, 1, 0])
@pytest.mark.parametrize("kx,hid,nout", MLP_SHAPES)
@pytest.mark.parametrize("M,gather", [(1, False), (77, True), (128, False), (129, True), (1350, False), (1350, True),
                                      (40000, True)])
def test_tc_mlp2_smallk_forward(lib, M, gather, kx, hid, nout, precision):
    """tm_tc_mlp2_smallk_forward (Linear(kx, hid) -> ReLU -> Linear(hid, nout), hidden layer generated in the operand
    loader): mlp_alpha's 1 -> 64 -> 32 and fc_net_self's 2 -> 256 -> 128 in every precision, against fp64, written
    at column 256 of a strided buffer as the head writes it (pixel stride 288 for the 32-wide output); rows and
    columns outside the output keep their sentinel."""
    torch.manual_seed(M + hid + precision)
    n_src, n_dst = M + 37, M + 11
    X, W1, b1, W2, b2 = _mlp_inputs(M, kx, hid, nout, M + hid + precision, n_src)
    xr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    orow = torch.randperm(n_dst, device=DEV)[:M].int().contiguous() if gather else None
    xs = X[xr.long()] if gather else X[:M]
    ref = torch.relu(xs.double() @ W1.double().t() + b1.double()) @ W2.double().t() + b2.double()
    col0 = 256
    ldo = 288 if nout == 32 else col0 + nout + 16
    buf = torch.full((n_dst, ldo), -5.0, device=DEV)
    out = buf[:, col0:col0 + nout]
    err = _err()
    lib.call("tm_tc_mlp2_smallk_forward", M, hid, nout, X, kx, xr, kx, W1, b1, W2, b2, out, ldo, orow, precision, err,
             lib.stream())
    assert int(err.item()) == 0
    rows = orow.long() if gather else torch.arange(M, device=DEV)
    assert_close(out[rows], ref, *TOL[precision], "smallk forward")
    touched = torch.zeros_like(buf, dtype=torch.bool)
    touched[rows, col0:col0 + nout] = True
    assert bool((buf[~touched] == -5.0).all()), "smallk forward wrote outside its rows / columns"


@pytest.mark.parametrize("precision", [3, 4, 2, 1, 0])
@pytest.mark.parametrize("kx,hid,nout", MLP_SHAPES)
@pytest.mark.parametrize("R,gather", [(1, False), (77, True), (129, False), (1350, True), (40000, True)])
def test_tc_mlp2_smallk_wgrad2(lib, R, gather, kx, hid, nout, precision):
    """tm_tc_mlp2_smallk_wgrad2: dW2 = G[g_rows]^T relu(X[x_rows] W1^T + b1) with the hidden layer generated as the B
    operand, rows of G scaled from 1e-5 to 1, against fp64; two calls give the same bits."""
    torch.manual_seed(R + hid + precision)
    n_src = R + 29
    X, W1, b1, _, _ = _mlp_inputs(R, kx, hid, nout, R + 3 * hid + precision, n_src)
    G = torch.randn(n_src, nout, device=DEV) * torch.logspace(-5, 0, n_src, device=DEV)[torch.randperm(n_src, device=DEV)][:, None]
    xr = torch.randperm(n_src, device=DEV)[:R].int().contiguous() if gather else None
    gr = torch.randperm(n_src, device=DEV)[:R].int().contiguous() if gather else None
    xs = X[xr.long()] if gather else X[:R]
    gs = G[gr.long()] if gather else G[:R]
    ref = gs.double().t() @ torch.relu(xs.double() @ W1.double().t() + b1.double())
    nb = lib.ws_bytes("tm_tc_gemm_tn_ws", nout, hid, R)
    err = _err()
    outs = []
    for _ in range(2):
        dW2 = torch.full((nout, hid), 3.0, device=DEV)
        lib.call("tm_tc_mlp2_smallk_wgrad2", nout, hid, R, G, nout, gr, X, kx, xr, kx, W1, b1, dW2, precision,
                 lib.workspace(nb, DEV), nb, err, lib.stream())
        outs.append(dW2)
    assert int(err.item()) == 0
    assert_close(outs[0], ref, *TOL[precision], "smallk dW2")
    assert torch.equal(outs[0], outs[1]), "smallk wgrad2 is not deterministic"


@pytest.mark.parametrize("data", ["exact", "float"])
@pytest.mark.parametrize("K", [32, 128])
@pytest.mark.parametrize("N", [64, 256])
@pytest.mark.parametrize("kx", [1, 2])
@pytest.mark.parametrize("M,gather", [(129, True), (1350, False), (40000, True)])
def test_tc_mlp1_bwd_fused(lib, M, gather, kx, N, K, data):
    """tm_tc_mlp1_bwd_fused: db1 = sum dh, dW1 = dh^T X with dh = (G W2) * (pre > 0), the ReLU mask either rebuilt
    from W1, b1 (H = NULL, the generated-hidden backward) or read from a stored H (ldh % 4 == 0), against fp64.
    "exact": integer inputs, W1 and b1 multiples of 1/64, so every pre-activation is exact in fp32 and thousands of
    them are exactly 0 (ReLU off, as torch.relu's gradient): both masks must equal the fp64 one, and the two calls
    give the same bits.  "float": inputs of magnitude 1e-3 .. 50 (a gate within an ulp of 0 may go either way).
    Two calls give the same bits."""
    torch.manual_seed(M + N + K + kx)
    n_src = M + 41
    if data == "exact":
        g = torch.Generator(device=DEV).manual_seed(M + N + K + kx)
        X = torch.randint(-20, 201, (n_src, kx), device=DEV, generator=g).float()
        W1 = torch.randint(-64, 65, (N, kx), device=DEV, generator=g).float() / 64
        b1 = torch.randint(-640, 641, (N,), device=DEV, generator=g).float() / 64
        W1[::3] = 0.5
        b1[::3] = -0.5 * torch.randint(0, 20, (len(range(0, N, 3)),), device=DEV, generator=g).float()
        X[::2, 0] = torch.randint(0, 20, (len(range(0, n_src, 2)),), device=DEV, generator=g).float()
        if kx == 2:
            W1[::3, 1] = 0.0
    else:
        X, W1, b1, _, _ = _mlp_inputs(M, kx, N, K, M + N + K, n_src)
    W2 = torch.randn(K, N, device=DEV) / N ** 0.5
    G = torch.randn(n_src, K, device=DEV)
    G[::7] *= 1e-4
    xr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    gr = torch.randperm(n_src, device=DEV)[:M].int().contiguous() if gather else None
    xs = X[xr.long()] if gather else X[:M]
    gs = G[gr.long()] if gather else G[:M]
    pre = xs.double() @ W1.double().t() + b1.double()
    if data == "exact":
        assert int((pre == 0).sum()) > M // 10, "the exact data lost its zero pre-activations"
    dh = (gs.double() @ W2.double()) * (pre > 0)
    ref_db, ref_dw = dh.sum(0), dh.t() @ xs.double()
    ldh = N + 8
    Hbuf = torch.full((M, ldh), float("nan"), device=DEV)
    Hbuf[:, :N] = torch.relu(pre).float()                # the stored hidden layer: zero wherever pre <= 0
    W2t = W2.t().contiguous()
    nb = lib.ws_bytes("tm_tc_mlp1_bwd_ws", N)
    err = _err()
    res = {}
    for mode in ("gen", "gen2", "stored"):
        H = Hbuf if mode == "stored" else None
        dW1 = torch.full((N, kx), 9.0, device=DEV)
        db1 = torch.full((N,), 9.0, device=DEV)
        lib.call("tm_tc_mlp1_bwd_fused", M, N, K, G, K, gr, W2t, H, ldh, X, kx, xr, kx, W1 if H is None else None,
                 b1 if H is None else None, dW1, db1, lib.workspace(nb, DEV), nb, err, lib.stream())
        res[mode] = (dW1, db1)
    assert int(err.item()) == 0
    bad = 0 if data == "exact" else 4                    # "float": a gate at |pre| ~ 1 ulp may go either way
    for mode in ("gen", "stored"):
        dW1, db1 = res[mode]
        assert_close(db1, ref_db, 1e-4, 2e-5, f"{mode} db1", max_bad=bad)
        assert_close(dW1, ref_dw, 1e-4, 2e-5, f"{mode} dW1", max_bad=2 * bad)
    assert torch.equal(res["gen"][0], res["gen2"][0]) and torch.equal(res["gen"][1], res["gen2"][1]), \
        "mlp1_bwd_fused is not deterministic"
    if data == "exact":
        assert torch.equal(res["gen"][0], res["stored"][0]) and torch.equal(res["gen"][1], res["stored"][1]), \
            "the regenerated ReLU mask differs from the stored hidden layer's"
