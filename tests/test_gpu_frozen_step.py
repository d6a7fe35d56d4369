"""Input-gradient steps against a frozen predictor: ``DesignStep.run(b, input_grads=True, param_grads=False)``.

1. ``tm_selfmlp_rows_dx`` (the fused data gradient of ``fc_cell_self``) against fp64, and its unserved arguments.
2. The NULL forms of the weight-gradient halves (``tm_selfmlp_gen_bwd1_dx`` without dW1 / db1, ``tm_fuse_backward`` /
   ``tm_fuse_backward_multi`` without dWt, ``tm_gnn_backward`` without GHID / GZC on both back ends): the data output is
   the same bits as the full call's.
3. The frozen step against ``run(input_grads=True)``: loss, predictions, image and net-pin gradients bit for bit, the
   cell-pin gradient against the fp64 oracle, and the model left exactly as it was.
4. ``pred_grad``, ``prune``, joined designs, graph replays, config 2, and the modules with frozen parameters.
"""
import numpy as np
import pytest
import torch

import tm_synth
from conftest import assert_close, design_to_oracle, relu_gate_flips
from test_gpu_multi_design import _design, _models
from test_gpu_step_input_grads import KEYS, _forced_and_gate, _oracle, _setup

DEV = "cuda"


@pytest.fixture(scope="module")
def mods(pkg):
    import tm_engine, tm_lib, tm_ops, tm_unet  # noqa: E401
    yield dict(engine=tm_engine, lib=tm_lib, ops=tm_ops, unet=tm_unet)
    if torch.cuda.is_available():
        tm_lib.check_err_flags()                 # no tensor-core barrier ever timed out


# ------------------------------------------------------------------------------------------------------------------
# 1. tm_selfmlp_rows_dx
# ------------------------------------------------------------------------------------------------------------------
def _rows_dx_inputs(M, kin, gather, seed):
    """Rows of G span 7 orders of magnitude; H has exact zeros and negatives (the gate is H > 0)."""
    g = torch.Generator().manual_seed(seed)
    n_src = M + 29
    W1 = torch.randn(256, kin, generator=g) * 0.2
    W2 = torch.randn(128, 256, generator=g) * 0.1
    H = torch.randn(n_src, 256, generator=g)
    H[torch.rand(n_src, 256, generator=g) < 0.1] = 0.0
    expo = torch.randint(-3, 4, (n_src,), generator=g)
    G = torch.randn(n_src, 128, generator=g) * torch.pow(10.0, expo.double()).float()[:, None]
    perm = (lambda: torch.randperm(n_src, generator=g)[:M].int()) if gather else (lambda: None)
    return n_src, W1, W2, H, G, expo, perm(), perm(), perm()


@pytest.mark.gpu
@pytest.mark.parametrize("kin", [4, 36, 48])
@pytest.mark.parametrize("gather", [False, True])
@pytest.mark.parametrize("M", [1, 127, 128, 129, 3001])
def test_selfmlp_rows_dx_vs_fp64(mods, M, kin, gather):
    """dX[x_rows[m]] = ((G[g_rows[m]] W2) * (H[h_rows[m]] > 0)) W1 against fp64 at the test_selfmlp_* bar (rtol 1e-4,
    atol 2e-5 of the scale, per order of magnitude of G's rows: the kernel scales each row on its own); rows no m maps
    to stay untouched; bit-identical on a second call."""
    lib = mods["lib"]
    n_src, W1, W2, H, G, expo, gr, hr, xr = _rows_dx_inputs(M, kin, gather, 7 * M + kin)
    sel = (lambda t, r: t[r.long()]) if gather else (lambda t, r: t[:M])
    ref = ((sel(G, gr).double() @ W2.double()) * (sel(H, hr) > 0)) @ W1.double()
    gexp = sel(expo, gr)
    W1d, W2d, Hd, Gd = (t.to(DEV) for t in (W1, W2, H, G))
    gr_d, hr_d, xr_d = (None if t is None else t.to(DEV) for t in (gr, hr, xr))
    nb = lib.ws_bytes("tm_selfmlp_rows_dh_ws_bytes")

    def run():
        dX = torch.full((n_src, 48), -7.0, device=DEV)          # row stride 48: kin < 48 leaves columns untouched
        lib.call("tm_selfmlp_rows_dx", M, Gd, 128, gr_d, W2d, Hd, 256, hr_d, W1d, kin, dX, 48, xr_d,
                 lib.workspace(nb, DEV), nb, lib.stream())
        return dX
    dX = run()
    rows = xr.long() if gather else torch.arange(M)
    got = dX.cpu()[rows, :kin]
    for e in torch.unique(gexp).tolist():
        s = gexp == e
        assert_close(got[s], ref[s], 1e-4, 2e-5, f"dX (rows of |G| ~ 1e{e})")
    untouched = torch.ones(n_src, dtype=torch.bool)
    untouched[rows] = False
    assert bool((dX.cpu()[untouched] == -7.0).all()) and bool((dX.cpu()[:, kin:] == -7.0).all())
    assert torch.equal(dX, run()), "not bit-deterministic"


@pytest.mark.parametrize("kin,G,ws_bytes,dX,lddx,what", [
    (6, 256, 1 << 30, 256, 8, "multiple of 4"),
    (52, 256, 1 << 30, 256, 52, "multiple of 4, <= 48"),
    (36, 260, 1 << 30, 256, 36, "16-byte aligned"),
    (36, 256, 1 << 30, 256, 34, "16-byte aligned"),
    (36, 256, 1024, 256, 36, "workspace too small"),
    (36, 256, 1 << 30, None, 36, "required"),
])
def test_selfmlp_rows_dx_rejects_unserved_arguments(mods, kin, G, ws_bytes, dX, lddx, what):
    """Unserved arguments fail with an error naming them before any launch (no device needed)."""
    lib = mods["lib"]
    before = lib.launch_count()
    with pytest.raises(RuntimeError, match=f"tm_selfmlp_rows_dx.*{what}"):
        lib.call("tm_selfmlp_rows_dx", 1000, G, 128, None, 256, 256, 256, None, 256, kin, dX, lddx, None,
                 256, ws_bytes, None)
    assert lib.launch_count() == before


@pytest.mark.parametrize("fn,dW1,db1,dX,what", [
    ("tm_selfmlp_gen_bwd1", None, None, None, "served with dX only"),
    ("tm_selfmlp_gen_bwd1_dx", None, 256, 256, "dW1 and db1 must be both set or both NULL"),
    ("tm_selfmlp_gen_bwd1_dx", 256, None, 256, "dW1 and db1 must be both set or both NULL"),
])
def test_null_weight_gradients_rejected_where_unserved(mods, fn, dW1, db1, dX, what):
    """NULL weight-gradient outputs are served only where the data gradient is produced (no device needed)."""
    lib = mods["lib"]
    before = lib.launch_count()
    with pytest.raises(RuntimeError, match=f"{fn}.*{what}"):
        if fn == "tm_selfmlp_gen_bwd1":
            lib.call(fn, 1000, 256, 128, None, 256, 2, None, 2, 256, 256, 256, dW1, db1, 256, 1 << 30, None)
        else:
            lib.call(fn, 1000, 256, 128, None, 256, 2, None, 2, 256, 256, 256, dW1, db1, dX, 2, 256, 1 << 30, None)
    with pytest.raises(RuntimeError, match="tm_fuse_backward.*dF missing"):
        lib.call("tm_fuse_backward", 10, 100, 128, 256, 256, 256, 128, 256, 256, None, None, None)
    with pytest.raises(RuntimeError, match="tm_fuse_backward_multi.*dF missing"):
        lib.call("tm_fuse_backward_multi", 2, 100, 128, 256, 256, 256, 128, 256, 256, None, None, None)
    assert lib.launch_count() == before


# ------------------------------------------------------------------------------------------------------------------
# 2. NULL forms: the data output is the full call's
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("M,kx,gather", [(129, 2, True), (100003, 1, False)])
def test_gen_bwd1_dx_without_weight_gradients_is_bitwise(mods, M, kx, gather):
    lib = mods["lib"]
    g = torch.Generator().manual_seed(M)
    n_src = M + 37
    X = torch.randn(n_src, kx, generator=g).to(DEV)
    W1, b1 = torch.randn(256, kx, generator=g).to(DEV), torch.randn(256, generator=g).to(DEV)
    W2, G = (torch.randn(128, 256, generator=g) * 0.1).to(DEV), torch.randn(n_src, 128, generator=g).to(DEV)
    xr = torch.randperm(n_src, generator=g)[:M].int().to(DEV) if gather else None
    gr = torch.randperm(n_src, generator=g)[:M].int().to(DEV) if gather else None
    nb = lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")
    out = []
    for wg in (True, False):
        dW1, db1 = (torch.empty(256, kx, device=DEV), torch.empty(256, device=DEV)) if wg else (None, None)
        dX = torch.full((n_src, kx), -7.0, device=DEV)
        lib.call("tm_selfmlp_gen_bwd1_dx", M, G, 128, gr, X, kx, xr, kx, W1, b1, W2, dW1, db1, dX, kx,
                 lib.workspace(nb, DEV), nb, lib.stream())
        out.append(dX)
    assert torch.equal(out[0], out[1])


def _fuse_case(mods, K):
    eng = mods["engine"]
    ds = [_design("unet", 21 + k, 3000, 700 + 50 * k) for k in range(K)]
    bs = [eng.DesignBatch.from_synth(d, DEV) for d in ds]
    b = bs[0] if K == 1 else eng.DesignBatch.concat(bs)
    J = b.width
    g = torch.Generator().manual_seed(K)
    feat = torch.randn(K * J, generator=g).to(DEV)
    wt = torch.randn(J, 128, generator=g).to(DEV)
    T = int(b.endpoints.numel())
    gy = torch.randn(T, 128, generator=g).to(DEV)
    return b, feat, wt, gy


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3])
def test_fuse_backward_without_weight_gradient_is_bitwise(mods, K):
    """tm_fuse_backward (K = 1) and tm_fuse_backward_multi (K = 3) with dWt = NULL: dF is the full call's."""
    ops = mods["ops"]
    b, feat, wt, gy = _fuse_case(mods, K)
    tab = b.fuse_table() if K > 1 else None
    full = ops.fusion_backward_multi(b.mask_rows_list, tab, b.ep_off, feat, wt, gy, 128)
    only = ops.fusion_backward_multi(b.mask_rows_list, tab, b.ep_off, feat, wt, gy, 128, need_wgrad=False)
    torch.cuda.synchronize()
    assert only[1] is None and only[2] is None
    assert torch.equal(full[0], only[0])


@pytest.mark.gpu
@pytest.mark.parametrize("impl", [0, 16, 3])
def test_gnn_backward_without_weight_gradient_operands_is_bitwise(mods, impl):
    """tm_gnn_backward with GHID = GZC = NULL on the per-level back end (3xTF32 and fp16-split cell kernels, impl 0 /
    16) and the persistent one (impl 3): G and the net-pin feature gradient are the full call's bits, the cell-pin one
    (fused tm_selfmlp_rows_dx) is within rtol 1e-4 + 2e-5 of the scale of it."""
    eng, ops, lib = mods["engine"], mods["ops"], mods["lib"]
    d = tm_synth.make_design(seed=4, **tm_synth.CONFIGS["c1"])
    model, _ = eng.build_models(d.map_size, seed=4, device=DEV)
    b = eng.DesignBatch.from_synth(d, DEV)
    sched = b.graph.schedule()
    gp = [p.detach() for p in eng.DesignStep(model, _).gnn_params]
    old = lib.lib().tm_gnn_set_impl(impl)
    try:
        H, saved = ops.gnn_forward(sched, b.cell_feat, b.net_feat, gp, save=True)
        G0 = torch.zeros(sched.n, 128, device=DEV)
        G0[b.endpoints.long()] = torch.randn(int(b.endpoints.numel()), 128, generator=torch.Generator().manual_seed(1)).to(DEV)
        G1, G2 = G0.clone(), G0.clone()
        _, dcf1, dnf1 = ops.gnn_backward(sched, saved, gp, G1, need_dx=True)
        none, dcf2, dnf2 = ops.gnn_backward(sched, saved, gp, G2, need_dx=True, need_wgrad=False)
        torch.cuda.synchronize()
    finally:
        lib.lib().tm_gnn_set_impl(old)
    assert none is None
    assert torch.equal(G1, G2), "G differs"
    assert torch.equal(dnf1, dnf2), "dnet_feat differs"
    assert_close(dcf2, dcf1, 1e-4, 2e-5, "dcell_feat")
    assert bool((dcf2[sched.net_class.long()] == 0).all())


# ------------------------------------------------------------------------------------------------------------------
# 3. the frozen step
# ------------------------------------------------------------------------------------------------------------------
def _model_state(model, net):
    """Every parameter's bits, every .grad (the object and its bits), every buffer (BN statistics, num_batches_tracked)."""
    named = [("m." + k, p) for k, p in model.named_parameters()] + [("c." + k, p) for k, p in net.named_parameters()]
    bufs = [("m." + k, v) for k, v in model.named_buffers()] + [("c." + k, v) for k, v in net.named_buffers()]
    return dict(params={k: p.detach().clone() for k, p in named},
                grads={k: (p.grad, None if p.grad is None else p.grad.clone()) for k, p in named},
                bufs={k: v.clone() for k, v in bufs})


def _assert_state_unchanged(model, net, before):
    after = _model_state(model, net)
    for k, v in before["params"].items():
        assert torch.equal(after["params"][k], v), f"parameter {k} changed"
    for k, (obj, bits) in before["grads"].items():
        now = after["grads"][k][0]
        assert now is obj, f"{k}.grad was re-pointed"
        assert (bits is None and now is None) or torch.equal(now, bits), f"{k}.grad changed"
    assert set(after["bufs"]) == set(before["bufs"])
    for k, v in before["bufs"].items():
        assert torch.equal(after["bufs"][k], v), f"buffer {k} changed"


def _outs(b, loss, pred):
    return loss.clone(), pred.clone(), {k: v.clone() for k, v in b.input_grads.items()}


def _assert_frozen_matches(got, ref, cell_rtol=1e-3, cell_atol=2e-4):
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), "loss / predictions differ"
    for k in ("image", "net_feat"):
        assert torch.equal(got[2][k], ref[2][k]), k
    assert_close(got[2]["cell_feat"], ref[2]["cell_feat"], cell_rtol, cell_atol, "cell_feat")


def _check_frozen(mods, cnn, pooling, math=None, cfg="tiny", seed=0):
    """Training step with input gradients, then the frozen step on a fresh batch of the same design: bitwise loss /
    predictions / image and net-pin gradients, the cell-pin gradient against the teacher-forced fp64 oracle at the bar
    of test_gpu_step_input_grads, and the model (after the training step) untouched by the frozen one."""
    eng = mods["engine"]
    d, model, net, sd_m, sd_c = _setup(mods, cnn, cfg, pooling, math, seed)
    step = eng.DesignStep(model, net)
    b1 = eng.DesignBatch.from_synth(d, DEV)
    ref = _outs(b1, *step.run(b1, input_grads=True))
    torch.cuda.synchronize()
    before = _model_state(model, net)
    b2 = eng.DesignBatch.from_synth(d, DEV)
    got = _outs(b2, *step.run(b2, input_grads=True, param_grads=False))
    torch.cuda.synchronize()
    _assert_state_unchanged(model, net, before)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), "loss / predictions differ"
    for k in ("image", "net_feat"):
        assert torch.equal(got[2][k], ref[2][k]), k
    sched = b2.graph.schedule()
    other = torch.ones(d.n, dtype=torch.bool, device=DEV)
    other[sched.cell_class.long()] = False
    assert bool((got[2]["cell_feat"][other] == 0).all())
    forced, H = _forced_and_gate(mods, cnn, model, net, b2)
    od = design_to_oracle(d)
    rounding = "bf16" if math == "bf16" else None
    # the oracle's parameters are the ones the step ran with (sd_* were taken before the training step; it changed no
    # parameter, only .grad and the BN statistics, which the batch-statistics forward does not read)
    _, Hfree, _, _ = _oracle(sd_m, sd_c, od, cnn, pooling, rounding=rounding, forced=forced)
    relu_gate_flips(H, Hfree)
    _, _, rin, _ = _oracle(sd_m, sd_c, od, cnn, pooling, rounding=rounding, forced=forced, gate=(H.detach().cpu() > 0))
    assert_close(got[2]["cell_feat"], rin["cell_feat"], 1e-3, 2e-4, "dcell_feat")
    return step, model, net, d


@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
@pytest.mark.parametrize("math", [None, "bf16"])
@pytest.mark.parametrize("pooling", ["max", "avg"])
def test_frozen_step_vs_training_step(mods, cnn, math, pooling):
    """U-Net and LayoutNet, tf32x3 (default) and bf16 image modes, max and avg pooling."""
    _check_frozen(mods, cnn, pooling, math)


@pytest.mark.gpu
def test_config2_frozen_step(mods):
    """The full-size config-2 frozen step in the default arithmetic."""
    assert mods["ops"].MATH == "tf32x3"
    _check_frozen(mods, "unet", "max", cfg="c2")


@pytest.mark.gpu
def test_frozen_step_posts_no_collective_and_keeps_none_grads(mods):
    """A step built for several ranks posts nothing when frozen (no bucket is created); a model that never trained
    keeps every .grad None and its BN statistics."""
    eng = mods["engine"]
    d, model, net, _, _ = _setup(mods, "unet")
    step = eng.DesignStep(model, net, world_size=2)
    before = _model_state(model, net)
    assert all(g is None for g, _ in before["grads"].values())
    b = eng.DesignBatch.from_synth(d, DEV)
    step.run(b, input_grads=True, param_grads=False)
    torch.cuda.synchronize()
    assert step._buckets == {}
    _assert_state_unchanged(model, net, before)


def test_frozen_step_needs_input_grads(mods):
    """param_grads=False without input_grads is refused before any work (no device needed)."""
    eng = mods["engine"]
    model, net = eng.build_models(32, device="cpu")
    step = eng.DesignStep(model, net)
    with pytest.raises(ValueError, match="input_grads"):
        step.run(None, param_grads=False)
    with pytest.raises(ValueError, match="input_grads"):
        step.capture(None, param_grads=False)


# ------------------------------------------------------------------------------------------------------------------
# 4. pred_grad, prune, joined designs, replays, modules
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_frozen_step_with_pred_grad(mods):
    eng = mods["engine"]
    d, model, net, _, _ = _setup(mods, "layoutnet", math="bf16")
    step = eng.DesignStep(model, net)
    b = eng.DesignBatch.from_synth(d, DEV)
    seed = torch.randn(int(b.endpoints.numel()), generator=torch.Generator().manual_seed(3)).to(DEV)
    ref = _outs(b, *step.run(b, input_grads=True, pred_grad=seed))
    before = _model_state(model, net)
    got = _outs(b, *step.run(b, input_grads=True, pred_grad=seed, param_grads=False))
    torch.cuda.synchronize()
    _assert_state_unchanged(model, net, before)
    _assert_frozen_matches(got, ref)


@pytest.mark.gpu
def test_pruned_frozen_step(mods):
    eng = mods["engine"]
    d = tm_synth.make_design(seed=5, **tm_synth.CONFIGS["c1"])
    model, net = eng.build_models(d.map_size, seed=5, device=DEV)
    rng = np.random.default_rng(5)
    T = len(d.endpoints)
    sel = torch.from_numpy(np.sort(rng.choice(T, size=max(2, T // 20), replace=False))).to(DEV)
    host = eng.HostDesign(d, pin=False)

    def batch():
        b = eng.DesignBatch.from_host(host, DEV)
        return eng.DesignBatch(b.graph, b.mask_csr, b.endpoints[sel].contiguous(), b.endpoint_level[sel].contiguous(),
                               b.arrival_time[sel].contiguous(), b.image, cell_feat=b.cell_feat, net_feat=b.net_feat,
                               rows=sel.int().contiguous())
    step = eng.DesignStep(model, net, prune=True)
    b = batch()
    ref = _outs(b, *step.run(b, input_grads=True))
    before = _model_state(model, net)
    b = batch()
    got = _outs(b, *step.run(b, input_grads=True, param_grads=False))
    torch.cuda.synchronize()
    assert b.cone().fraction < 1.0
    _assert_state_unchanged(model, net, before)
    _assert_frozen_matches(got, ref)
    assert bool((got[2]["cell_feat"][~b.cone().active] == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_three_designs_frozen_step(mods, cnn):
    eng = mods["engine"]
    ds = [_design(cnn, 11, 5000, 1350), _design(cnn, 12, 3500, 900), _design(cnn, 13, 4200, 1100)]
    model, net = _models(mods, cnn, None)
    step = eng.DesignStep(model, net)
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(d, DEV) for d in ds])
    ref = _outs(b, *step.run(b, input_grads=True))
    ref_losses = b.design_losses.clone()
    before = _model_state(model, net)
    b2 = eng.DesignBatch.concat([eng.DesignBatch.from_synth(d, DEV) for d in ds])
    got = _outs(b2, *step.run(b2, input_grads=True, param_grads=False))
    torch.cuda.synchronize()
    _assert_state_unchanged(model, net, before)
    _assert_frozen_matches(got, ref)
    assert torch.equal(b2.design_losses, ref_losses)


@pytest.mark.gpu
def test_frozen_capture_prepare_and_prepare_many(mods):
    """Replays of a captured / prepared frozen step after the inputs were refreshed in place equal an eager frozen run
    on the new values bit for bit, and leave every .grad (object and bits), parameter and BN buffer alone."""
    eng = mods["engine"]
    d, model, net, _, _ = _setup(mods, "unet")
    step = eng.DesignStep(model, net)
    b0 = eng.DesignBatch.from_synth(d, DEV)
    step.run(b0)                                          # the model has .grad tensors and moved BN statistics
    torch.cuda.synchronize()
    before = _model_state(model, net)
    b = eng.DesignBatch.from_synth(d, DEV)
    T = int(b.endpoints.numel())
    seed = torch.randn(T, device=DEV)
    replay = step.capture(b, input_grads=True, pred_grad=seed, param_grads=False)
    b.cell_feat.mul_(0.5)
    b.net_feat.add_(0.25)
    b.image.copy_(b.image.flip(-1))
    seed.copy_(torch.randn(T, device=DEV))
    got = _outs(b, *replay())
    b2 = eng.DesignBatch.from_synth(d, DEV)
    for k in ("cell_feat", "net_feat", "image"):
        getattr(b2, k).copy_(getattr(b, k))
    ref = _outs(b2, *step.run(b2, input_grads=True, pred_grad=seed.clone(), param_grads=False))
    torch.cuda.synchronize()
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    for k in KEYS:
        assert torch.equal(got[2][k], ref[2][k]), k
    _assert_state_unchanged(model, net, before)
    # prepare
    d2 = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["tiny"])
    d2.cell_feat = (d.cell_feat * 0.5).astype(np.float32)
    d2.image = np.ascontiguousarray(d.image[:, ::-1, :]).astype(np.float32)
    host2 = eng.HostDesign(d2, pin=True)
    prep = step.prepare(eng.HostDesign(d, pin=True), DEV, input_grads=True, param_grads=False)
    got = _outs(prep.batch, *prep.step(host2))
    b3 = eng.DesignBatch.from_host(host2, DEV)
    ref = _outs(b3, *step.run(b3, input_grads=True, param_grads=False))
    torch.cuda.synchronize()
    assert torch.equal(got[0], ref[0])
    for k in KEYS:
        assert torch.equal(got[2][k], ref[2][k]), k
    _assert_state_unchanged(model, net, before)
    step.close()
    # prepare_many: three designs (map size 32), new values for all of them
    model, net = _models(mods, "unet", None)
    step = eng.DesignStep(model, net)
    ds = [_design("unet", 31 + k, 2500, 600) for k in range(3)]
    hosts = [eng.HostDesign(x, pin=True) for x in ds]
    before = _model_state(model, net)
    many = step.prepare_many(hosts, DEV, input_grads=True, param_grads=False)
    for x in ds:
        x.image = np.ascontiguousarray(x.image[:, :, ::-1]).astype(np.float32)
        x.net_feat = (x.net_feat + 0.5).astype(np.float32)
    hosts2 = [eng.HostDesign(x, pin=True) for x in ds]
    got = _outs(many.batch, *many.step(hosts2))
    b4 = eng.DesignBatch.concat([eng.DesignBatch.from_host(h, DEV) for h in hosts2])
    ref = _outs(b4, *step.run(b4, input_grads=True, param_grads=False))
    torch.cuda.synchronize()
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    for k in KEYS:
        assert torch.equal(got[2][k], ref[2][k]), k
    _assert_state_unchanged(model, net, before)
    step.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_module_image_grad_with_frozen_parameters(mods, cnn):
    """UNet / LayoutNet modules whose parameters have requires_grad=False: the image .grad is the bits it has with
    trainable parameters, no weight-gradient kernel runs (fewer launches) and every parameter .grad stays None."""
    lib = mods["lib"]
    d = _design(cnn, 3, 2000, 300)
    _, net = _models(mods, cnn, None)
    x0 = torch.from_numpy(d.image).to(DEV)

    def grad(frozen):
        for p in net.parameters():
            p.requires_grad_(not frozen)
            p.grad = None
        x = x0.clone().requires_grad_(True)
        out = net(x)
        g = torch.randn(out.shape, generator=torch.Generator().manual_seed(9)).to(DEV)
        before = lib.launch_count()
        out.backward(g)
        torch.cuda.synchronize()
        return x.grad.clone(), lib.launch_count() - before
    ref, n_full = grad(False)
    got, n_frozen = grad(True)
    assert torch.equal(got, ref)
    assert n_frozen < n_full
    assert all(p.grad is None for p in net.parameters())
