"""Several designs in one fused design step (``DesignBatch.concat`` + ``DesignStep``):
  * the segmented batch norm (tm_bn_relu_forward_seg / tm_bn_relu_backward_seg) against single-image calls, bit for bit;
  * the batched mask fusion (tm_fuse_forward_runs_multi / tm_fuse_backward_multi) and the per-design MSE (tm_mse_multi)
    against the one-design kernels;
  * a one-design concat against the one-design step, bit for bit;
  * three designs against the mean of three single-design steps (the data-parallel definition, tests/dp_equivalence.py);
  * capture, prepare_many, tm_loader.prepare_many, pruning, forward and the shape checks."""
import numpy as np
import pytest
import torch

import tm_synth
from conftest import assert_close, assert_grad_close_given_flips, relu_gate_flips

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def mods(pkg):
    import tm_engine, tm_lib, tm_loader, tm_ops, tm_unet  # noqa: E401
    yield dict(engine=tm_engine, lib=tm_lib, loader=tm_loader, ops=tm_ops, unet=tm_unet)
    tm_lib.check_err_flags()


def _eq(a, b, what):
    assert torch.equal(a, b), f"{what}: {int((a != b).sum())}/{a.numel()} elements differ"


# ------------------------------------------------------------------------------------------------------------------
# segmented batch norm
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("C", [6, 16, 32, 64, 128])
def test_bn_segmented_matches_single_image_calls(mods, C, K):
    """Per-image y, statistics and dx bit-identical to single-image calls on a strided input inside a concat buffer,
    with the bf16 side outputs; running statistics equal K sequential single calls; dgamma / dbeta the per-image sum."""
    lib = mods["lib"]
    torch.manual_seed(C + K)
    H = W = 24
    npix = H * W
    cat = torch.randn(K * npix, 2 * C, device=DEV) * 2 + 0.3        # x = first half of each row (ld = 2C)
    x, ldx = cat, 2 * C
    dy = torch.randn(K * npix, C, device=DEV)
    gamma, beta = torch.rand(C, device=DEV) + 0.5, torch.randn(C, device=DEV) * 0.1
    rm0, rv0 = torch.randn(C, device=DEV), torch.rand(C, device=DEV) + 0.5
    mom, eps = 0.1, 1e-5

    # segmented
    rm, rv = rm0.clone(), rv0.clone()
    y = torch.empty(K * npix, C, device=DEV)
    yb = torch.empty(K * npix, C, dtype=torch.bfloat16, device=DEV)
    mean, inv = torch.empty(K * C, device=DEV), torch.empty(K * C, device=DEV)
    nb = lib.ws_bytes("tm_bn_seg_ws", K, npix, C)
    ws = lib.workspace(nb, DEV)
    lib.call("tm_bn_relu_forward_seg", K, npix, C, x, ldx, gamma, beta, rm, rv, mom, eps, y, C, mean, inv, yb, ws, nb,
             lib.stream())
    dx = torch.empty(K * npix, C, device=DEV)
    dxb = torch.empty(K * npix, C, dtype=torch.bfloat16, device=DEV)
    dg, db = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    lib.call("tm_bn_relu_backward_seg", K, npix, C, x, ldx, None, 0, dy, C, gamma, beta, mean, inv, dx, C, dg, db, dxb,
             ws, nb, lib.stream())

    # K single-image calls on the same strided rows
    rm1, rv1 = rm0.clone(), rv0.clone()
    nb1 = lib.ws_bytes("tm_bn_ws", npix, C)
    ws1 = lib.workspace(nb1, DEV)
    dgs, dbs = [], []
    for k in range(K):
        xs = cat[k * npix:(k + 1) * npix]
        y1 = torch.empty(npix, C, device=DEV)
        yb1 = torch.empty(npix, C, dtype=torch.bfloat16, device=DEV)
        m1, i1 = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
        lib.call("tm_bn_relu_forward", npix, C, xs, ldx, gamma, beta, rm1, rv1, mom, eps, y1, C, m1, i1, yb1, None, 0,
                 ws1, nb1, lib.stream())
        dx1 = torch.empty(npix, C, device=DEV)
        dxb1 = torch.empty(npix, C, dtype=torch.bfloat16, device=DEV)
        dg1, db1 = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
        lib.call("tm_bn_relu_backward", npix, C, xs, ldx, None, 0, dy[k * npix:(k + 1) * npix], C, gamma, beta, m1, i1,
                 dx1, C, dg1, db1, dxb1, ws1, nb1, lib.stream())
        torch.cuda.synchronize()
        sl = slice(k * npix, (k + 1) * npix)
        _eq(y[sl], y1, f"y[{k}]")
        _eq(yb[sl], yb1, f"y_bf16[{k}]")
        _eq(mean[k * C:(k + 1) * C], m1, f"mean[{k}]")
        _eq(inv[k * C:(k + 1) * C], i1, f"invstd[{k}]")
        _eq(dx[sl], dx1, f"dx[{k}]")
        _eq(dxb[sl], dxb1, f"dx_bf16[{k}]")
        dgs.append(dg1)
        dbs.append(db1)
    _eq(rm, rm1, "running_mean")
    _eq(rv, rv1, "running_var")
    if K == 1:
        _eq(dg, dgs[0], "dgamma")
        _eq(db, dbs[0], "dbeta")
    else:
        for got, parts, what in ((dg, dgs, "dgamma"), (db, dbs, "dbeta")):
            ref = torch.stack(parts).double().sum(0)
            assert float(((got.double() - ref).abs() / ref.abs().clamp_min(1e-30)).max()) <= 1e-6, what


# ------------------------------------------------------------------------------------------------------------------
# batched fusion and per-design MSE
# ------------------------------------------------------------------------------------------------------------------
def _mask_designs(mods, K):
    """K tiny designs with the same map and different endpoint counts; rows: a random selection with repeats."""
    eng = mods["engine"]
    out = []
    for k in range(K):
        d = tm_synth.make_design(seed=20 + k, n_cells=300 + 50 * k, n_lv=6, map_size=8, n_endpoints=40 - 7 * k)
        b = eng.DesignBatch.from_synth(d, DEV)
        rng = np.random.default_rng(k)
        rows = torch.from_numpy(rng.integers(0, b.mask_csr.num_rows, size=30 - 4 * k).astype(np.int32)).to(DEV)
        out.append(eng.DesignBatch(b.graph, b.mask_csr, b.endpoints[rows.long()].contiguous(),
                                   b.endpoint_level[rows.long()].contiguous(), b.arrival_time[rows.long()].contiguous(),
                                   b.image, rows=rows))
    return out


@pytest.mark.parametrize("K", [1, 3])
def test_batched_fusion_and_mse(mods, K):
    eng, ops, lib = mods["engine"], mods["ops"], mods["lib"]
    parts = _mask_designs(mods, K)
    b = eng.DesignBatch.concat(parts)
    J, T = b.width, int(b.endpoints.numel())
    torch.manual_seed(K)
    feat = torch.rand(K * J, device=DEV)
    w, bias = torch.randn(128, J, device=DEV) * 0.05, torch.randn(128, device=DEV)
    ld = 160
    out = torch.zeros(T, ld, device=DEV)
    tab = b.fuse_table()
    # the multi-design kernels are called directly (the step takes tm_fuse_forward_runs itself at K = 1)
    wt = ops.transpose(w)
    nb = lib.ws_bytes("tm_fuse_runs_multi_ws", K, J)
    lib.call("tm_fuse_forward_runs_multi", K, T, J, 128, tab, b.ep_off, feat, wt, bias, out[:, 8:], ld,
             lib.workspace(nb, DEV), nb, lib.stream())
    g = torch.randn(T, ld, device=DEV)
    dwt = torch.empty(J, 128, device=DEV)
    dF = torch.empty(K * J, device=DEV)
    lib.call("tm_fuse_backward_multi", K, J, 128, tab, b.ep_off, g[:, 8:], ld, feat, wt, dwt, dF, lib.stream())
    pred, y = torch.randn(T, device=DEV), torch.randn(T, device=DEV)
    loss_k, loss = torch.empty(K, device=DEV), torch.empty(1, device=DEV)
    gpred = torch.empty(T, device=DEV)
    lib.call("tm_mse_multi", K, b.ep_off, pred, y, loss_k, loss, gpred, 1.0, lib.stream())
    torch.cuda.synchronize()

    old = ops.FUSE_RUNS
    ops.FUSE_RUNS = True
    try:
        dwt_ref = torch.zeros(J, 128, dtype=torch.float64, device=DEV)
        for k, p in enumerate(parts):
            s, e = int(b.ep_off_h[k]), int(b.ep_off_h[k + 1])
            o1 = torch.zeros(e - s, 128, device=DEV)
            Fk = feat[k * J:(k + 1) * J].contiguous()
            ops.fusion_forward(p.mask_rows, Fk, w, bias, o1, 128)
            gk = g[s:e, 8:136].contiguous()
            dF1, dw1, _ = ops.fusion_backward(p.mask_rows, Fk, wt, gk, 128)
            l1, gp1 = torch.empty(1, device=DEV), torch.empty(e - s, device=DEV)
            lib.call("tm_mse", e - s, pred[s:e].contiguous(), y[s:e].contiguous(), l1, gp1, 1.0 / K, lib.stream())
            torch.cuda.synchronize()
            _eq(out[s:e, 8:136], o1, f"fused rows of design {k}")
            _eq(dF[k * J:(k + 1) * J], dF1, f"dF of design {k}")
            dwt_ref += dw1.t().double()
            if K == 1:
                _eq(dwt, dw1.t().contiguous(), "dWt")
                _eq(loss_k, l1, "loss_k")
                _eq(loss, l1, "loss")
                _eq(gpred, gp1, "dpred")
            else:
                d64 = pred[s:e].double() - y[s:e].double()
                assert_close(loss_k[k], (d64 * d64).mean(), 1e-6, 0, f"loss_{k}")
                assert_close(gpred[s:e], 2 * d64 / ((e - s) * K), 1e-6, 1e-9, f"dpred of design {k}")
        if K > 1:
            assert_close(dwt, dwt_ref, 1e-5, 1e-6, "dWt vs fp64 sum")
            assert_close(loss.reshape(()), loss_k.double().mean(), 1e-6, 0, "mean loss")
    finally:
        ops.FUSE_RUNS = old


# ------------------------------------------------------------------------------------------------------------------
# the step
# ------------------------------------------------------------------------------------------------------------------
NETS = [("unet", None), ("unet", "bf16"), ("layoutnet", "bf16")]


def _design(cnn, seed, n_cells, T):
    kw = dict(img_channels=2, img_scale=4) if cnn == "layoutnet" else {}
    return tm_synth.make_design(seed=seed, n_cells=n_cells, n_lv=20, map_size=32, n_endpoints=T, **kw)


def _models(mods, cnn, math, seed=0, map_size=32):
    model, net = mods["engine"].build_models(map_size, seed=seed, device=DEV, cnn=cnn)
    if math:
        net.math = math
    return model, net


def _params(model, net):
    return list(model.named_parameters()) + [("cnn." + k, p) for k, p in net.named_parameters()]


def _grads(model, net):
    return {k: p.grad.detach().clone() for k, p in _params(model, net) if p.grad is not None}


def _buffers(net):
    return {k: v.detach().clone() for k, v in net.named_buffers()}


@pytest.mark.parametrize("cnn,math", NETS)
def test_one_design_concat_is_the_one_design_step(mods, cnn, math):
    """concat([b]) gives the loss, predictions, every gradient and the BN running statistics of the old step, bit for
    bit."""
    eng = mods["engine"]
    d = _design(cnn, 5, 3000, 700)
    res = []
    for join in (False, True):
        model, net = _models(mods, cnn, math)
        b = eng.DesignBatch.from_synth(d, DEV)
        if join:
            b = eng.DesignBatch.concat([b])
        loss, pred = eng.DesignStep(model, net).run(b)
        torch.cuda.synchronize()
        res.append((loss.clone(), pred.clone(), _grads(model, net), _buffers(net)))
    _eq(res[1][0], res[0][0], "loss")
    _eq(res[1][1], res[0][1], "pred")
    assert set(res[1][2]) == set(res[0][2])
    for k in res[0][2]:
        _eq(res[1][2][k], res[0][2][k], k)
    for k in res[0][3]:
        _eq(res[1][3][k], res[0][3][k], k)


def _close_dp(a, b, what):
    """tests/dp_equivalence.py's bar: 1e-5 relative + 1e-6 of the largest magnitude."""
    a, b = a.double(), b.double()
    tol = 1e-5 * b.abs() + 1e-6 * b.abs().max()
    bad = int(((a - b).abs() > tol).sum())
    assert bad == 0, f"{what}: {bad}/{a.numel()} elements differ (max {float((a - b).abs().max()):.3e})"


@pytest.mark.parametrize("cnn,math", NETS + [("layoutnet", None)])
def test_three_designs_equal_the_mean_of_single_steps(mods, monkeypatch, cnn, math):
    """Three c1-shaped designs (different seeds, sizes and endpoint counts) in one step: per-design predictions and
    losses, the mean loss, every gradient (mean of the single-design gradients) and the running statistics.

    Gradients: the netlist branch and the head at tests/dp_equivalence.py's bar.  The image network's (and fcn's,
    which reads its feature map) at rtol 1e-3 + 2e-3 of the largest image-network gradient (2e-2 + 2e-2 in bf16
    mode): a batch-K weight gradient of a convolution reduces over the pixels of all K images in one order, not image
    by image (and in bf16 mode dy carries the 1/K scale before its bf16 rounding).  Several of these gradients are
    sums that cancel to ~0 (a bias ahead of a batch norm, LayoutNet's first layer), so the reordering shows far above
    their own tiny scale; profiles/r3_bench_multi_design.json records how many elements miss the dp bar at full size."""
    eng = mods["engine"]
    if math == "bf16":
        # the multi-design step takes per-image statistics from the batch-norm pass (the convolution epilogue's cover
        # the whole batch); the single-design reference takes them from the same pass
        monkeypatch.setattr(mods["unet"], "FUSE_BN_STATS", False)
    ds = [_design(cnn, 11, 5000, 1350), _design(cnn, 12, 3500, 900), _design(cnn, 13, 4200, 1100)]
    model_s, net_s = _models(mods, cnn, math)
    step_s = eng.DesignStep(model_s, net_s)
    singles = []
    for d in ds:
        b = eng.DesignBatch.from_synth(d, DEV)
        loss, pred = step_s.run(b)
        torch.cuda.synchronize()
        with torch.no_grad():
            H = model_s.gnn.propagate(b.graph)
        singles.append((loss.clone(), pred.clone(), _grads(model_s, net_s), H.detach().clone()))
    model, net = _models(mods, cnn, math)
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(d, DEV) for d in ds])
    loss, pred = eng.DesignStep(model, net).run(b)
    torch.cuda.synchronize()
    with torch.no_grad():
        H = model.gnn.propagate(b.graph)
    flips = set()
    for k, s in enumerate(singles):
        e0, e1 = int(b.ep_off_h[k]), int(b.ep_off_h[k + 1])
        p0, p1 = int(b.pin_off_h[k]), int(b.pin_off_h[k + 1])
        flips |= relu_gate_flips(H[p0:p1], s[3])
        assert_close(pred[e0:e1], s[1], 1e-5, 1e-6, f"pred of design {k}")
        assert_close(b.design_losses[k], s[0].reshape(()), 1e-5, 0, f"loss of design {k}")
    assert_close(loss.reshape(()), torch.stack([s[0] for s in singles]).double().mean(), 1e-5, 0, "mean loss")
    got = _grads(model, net)
    assert set(got) == set(singles[0][2])
    refs = {k: torch.stack([s[2][k] for s in singles]).double().mean(0) for k in got}
    rtol, atol = (2e-2, 2e-2) if math == "bf16" else (1e-3, 2e-3)
    img_scale = max(float(r.abs().max()) for k, r in refs.items() if k.startswith("cnn."))
    for k, g in got.items():
        ref = refs[k]
        if k.startswith("cnn.") or k in ("fcn.weight", "fcn.bias"):
            scale = img_scale if k.startswith("cnn.") else float(ref.abs().max())
            err = (g.double() - ref).abs()
            bad = int((err > rtol * ref.abs() + atol * scale).sum())
            assert bad == 0, f"{k}: {bad}/{g.numel()} elements off (max err {float(err.max()):.3e}, scale {scale:.3e})"
        elif flips and k.startswith("gnn."):
            assert_grad_close_given_flips(g, ref, k, flips, rtol=1e-5, atol_scale=1e-6)
        else:
            _close_dp(g, ref, k)
    for k, v in _buffers(net).items():
        if k.endswith("num_batches_tracked"):
            _eq(v, _buffers(net_s)[k], k)
        else:
            assert_close(v, _buffers(net_s)[k], 1e-5, 1e-7, k)


def _tiny(seed, T, **kw):
    return tm_synth.make_design(seed=seed, n_cells=300 + 40 * seed, n_lv=6, map_size=8, n_endpoints=T, **kw)


def _assert_same(a, b):
    _eq(a[0], b[0], "loss")
    _eq(a[1], b[1], "pred")
    assert set(a[2]) == set(b[2])
    for k in a[2]:
        _eq(a[2][k], b[2][k], k)


@pytest.mark.parametrize("cnn,math", [("unet", None), ("layoutnet", "bf16")])
def test_capture_and_prepare_many(mods, cnn, math):
    """A captured three-design step replays the eager step bit for bit, twice in a row; prepare_many fed new values
    from host memory equals the eager step on those values."""
    eng = mods["engine"]
    kw = dict(img_channels=2, img_scale=4) if cnn == "layoutnet" else {}
    ds = [_tiny(s, T, **kw) for s, T in ((1, 40), (2, 31), (3, 25))]
    model, net = _models(mods, cnn, math, map_size=8)
    step = eng.DesignStep(model, net)
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(d, DEV) for d in ds])
    loss, pred = step.run(b)
    torch.cuda.synchronize()
    eager = (loss.clone(), pred.clone(), _grads(model, net))
    eager_k = b.design_losses.clone()
    replay = step.capture(b)
    for _ in range(2):
        loss_r, pred_r = replay()
        torch.cuda.synchronize()
        _assert_same((loss_r.clone(), pred_r.clone(), _grads(model, net)), eager)
        _eq(b.design_losses, eager_k, "per-design losses")
    hosts = [eng.HostDesign(d, pin=True) for d in ds]
    prep = step.prepare_many(hosts, DEV)
    ds2 = [_tiny(s, T, **kw) for s, T in ((1, 40), (2, 31), (3, 25))]
    for d in ds2:
        d.cell_feat = (d.cell_feat * 0.5).astype(np.float32)
        d.image = np.ascontiguousarray(d.image[:, ::-1, :]).astype(np.float32)
        d.arrival_time = (d.arrival_time * 1.1).astype(np.float32)
    hosts2 = [eng.HostDesign(d, pin=True) for d in ds2]
    loss_p, pred_p = prep.step(hosts2)
    torch.cuda.synchronize()
    got = (loss_p.clone(), pred_p.clone(), _grads(model, net))
    got_k = prep.batch.design_losses.clone()
    b2 = eng.DesignBatch.concat([eng.DesignBatch.from_host(h, DEV) for h in hosts2])
    loss_e, pred_e = step.run(b2)
    torch.cuda.synchronize()
    _assert_same(got, (loss_e.clone(), pred_e.clone(), _grads(model, net)))
    _eq(got_k, b2.design_losses, "per-design losses")
    assert not torch.equal(loss_p, loss)
    step.close()


def test_loader_prepare_many_shuffled_batches(mods):
    """tm_loader.prepare_many (one capture, every design's endpoint batch refreshed in place) against eager
    multi-design steps on the same path ids, over several shuffled batches with Adam steps in between."""
    eng, ldr = mods["engine"], mods["loader"]
    lds = [ldr.load_design(ldr.design_tuple_from_synth(_tiny(s, 40)), DEV) for s in (4, 5, 6)]
    model, net = _models(mods, "unet", None, seed=4, map_size=8)
    step = eng.DesignStep(model, net)
    bs = 16
    run = ldr.prepare_many(lds, step, batch_size=bs)
    gen = torch.Generator().manual_seed(0)
    for _ in range(3):
        ids = [[ld.paths[i] for i in torch.randperm(len(ld.paths), generator=gen)[:bs].tolist()] for ld in lds]
        loss_r, pred_r = run(ids)
        torch.cuda.synchronize()
        got = (loss_r.clone(), pred_r.clone(), _grads(model, net))
        loss_e, pred_e = step.run(eng.DesignBatch.concat([ld.batch(i) for ld, i in zip(lds, ids)]))
        torch.cuda.synchronize()
        assert_close(got[0], loss_e, 1e-6, 1e-7, "loss")
        assert_close(got[1], pred_e, 1e-6, 1e-6, "pred")
        for k, g in _grads(model, net).items():
            assert_close(got[2][k], g, 1e-6, 1e-6, k)
        step.adam_step({}, lr=1e-3)
    step.close()


def test_prune_on_joined_netlist(mods):
    """prune=True on three joined designs: the cone of the union, with test_design_step_on_cone_subnetlist's
    tolerances."""
    eng = mods["engine"]
    ds = [_design("unet", s, 3000, 600) for s in (7, 8, 9)]
    model, net = _models(mods, "unet", None, seed=7)
    out = {}
    for prune in (False, True):
        parts = []
        for k, d in enumerate(ds):
            b = eng.DesignBatch.from_synth(d, DEV)
            sel = np.sort(np.random.default_rng(k).choice(len(d.endpoints), size=20 + 5 * k, replace=False))
            idx = torch.from_numpy(sel).to(DEV)
            parts.append(eng.DesignBatch(b.graph, b.mask_csr, b.endpoints[idx].contiguous(),
                                         b.endpoint_level[idx].contiguous(), b.arrival_time[idx].contiguous(), b.image,
                                         cell_feat=b.cell_feat, net_feat=b.net_feat, rows=idx.int().contiguous()))
        b = eng.DesignBatch.concat(parts)
        for p in list(model.parameters()) + list(net.parameters()):
            p.grad = None
        loss, pred = eng.DesignStep(model, net, prune=prune).run(b)
        torch.cuda.synchronize()
        assert (b._cone is not None) == prune
        out[prune] = (loss.clone(), pred.clone(), _grads(model, net))
    assert b.cone().fraction < 1.0
    assert_close(out[True][1], out[False][1], 1e-6, 1e-6, "pred")
    assert_close(out[True][0], out[False][0], 1e-6, 1e-7, "loss")
    assert set(out[True][2]) == set(out[False][2])
    for k, gfull in out[False][2].items():
        scale = max(float(gfull.abs().max()), 1e-30)
        assert float((out[True][2][k] - gfull).abs().max()) <= 2e-5 * scale, k


@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_forward_equals_per_design_forward(mods, cnn):
    eng = mods["engine"]
    kw = dict(img_channels=2, img_scale=4) if cnn == "layoutnet" else {}
    ds = [_tiny(s, T, **kw) for s, T in ((1, 40), (2, 31), (3, 25))]
    model, net = _models(mods, cnn, None, map_size=8)
    step = eng.DesignStep(model, net)
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(d, DEV) for d in ds])
    pred = step.forward(b)
    for k, d in enumerate(ds):
        p1 = step.forward(eng.DesignBatch.from_synth(d, DEV))
        assert_close(pred[int(b.ep_off_h[k]):int(b.ep_off_h[k + 1])], p1, 1e-5, 1e-6, f"design {k}")


def test_concat_rejects_mismatched_designs(mods):
    eng = mods["engine"]
    a = eng.DesignBatch.from_synth(_tiny(1, 40), DEV)
    img = eng.DesignBatch.from_synth(_tiny(2, 30, img_scale=4), DEV)
    with pytest.raises(ValueError, match=r"design 1 has image \(3, 32, 32\) but design 0 has \(3, 16, 16\)"):
        eng.DesignBatch.concat([a, img])
    wide = eng.DesignBatch.from_synth(tm_synth.make_design(seed=3, n_cells=300, n_lv=6, map_size=16, n_endpoints=30,
                                                           img_scale=1), DEV)
    with pytest.raises(ValueError, match=r"design 1 has mask width \(256,\) but design 0 has \(64,\)"):
        eng.DesignBatch.concat([a, wide])
    c = eng.DesignBatch.from_synth(_tiny(4, 30), DEV)
    c.cell_feat = c.cell_feat[:, :10]
    with pytest.raises(ValueError, match=r"design 1 has cell_feat width \(10,\) but design 0 has \(36,\)"):
        eng.DesignBatch.concat([a, c])
