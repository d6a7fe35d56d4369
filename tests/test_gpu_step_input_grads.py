"""Input gradients of the fused design step (``DesignStep.run(input_grads=True, pred_grad=...)``): the gradients with
respect to ``cell_feat``, ``net_feat`` and the layout image.

1. ``tm_selfmlp_gen_bwd1_dx`` (the net pins' feature gradient, fused into the first-layer backward of the generated
   MLP) against its fp64 definition, and its unserved arguments (no device needed).
2. The step against an oracle built from ``oracle/restate.py``'s pieces in the order ``restate.design_step`` runs
   them, with the features and the image as leaves that require grad.  The oracle's image network is teacher-forced
   with the product's convolution outputs and its propagation with the product's output gates (``restate._force``,
   ``gnn_gate``), so both differentiate the same piecewise-linear function.
3. ``pred_grad``: the backward seeded by the caller is ``autograd.grad(pred, ..., seed)``.
4. Invariants: parameter gradients untouched, determinism, CUDA-graph replay, ``prune``, several designs.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import tm_synth
from conftest import assert_close, design_to_oracle, relu_gate_flips
from oracle import restate
from test_gpu_input_grads import _unet_forced
from test_gpu_layoutnet import _forced as _layoutnet_forced, _layout_design, _layoutnet_oracle
from test_gpu_multi_design import _design, _models

DEV = "cuda"
KEYS = ("cell_feat", "net_feat", "image")


@pytest.fixture(scope="module")
def mods(pkg):
    import tm_engine, tm_lib, tm_ops, tm_unet  # noqa: E401
    yield dict(engine=tm_engine, lib=tm_lib, ops=tm_ops, unet=tm_unet)
    if torch.cuda.is_available():
        tm_lib.check_err_flags()                 # no tensor-core barrier ever timed out


@pytest.fixture(params=["tf32x3", "tc6", "fp32"])
def math_mode(request, mods):
    old = mods["ops"].MATH
    mods["ops"].MATH = request.param
    yield request.param
    mods["ops"].MATH = old


# ------------------------------------------------------------------------------------------------------------------
# 1. tm_selfmlp_gen_bwd1_dx
# ------------------------------------------------------------------------------------------------------------------
def _bwd1_inputs(M, kx, gather, seed):
    """Exactly representable X, W1, b1 (quarters, eighths, sixteenths): the fp32 pre-activation the kernel masks with is
    exact, so the fp64 mask is the kernel's, and many pre-activations are exactly 0.  Rows of G span 13 orders of
    magnitude."""
    g = torch.Generator().manual_seed(seed)
    n_src = M + 37
    X = torch.randint(-8, 9, (n_src, kx), generator=g).float() / 4
    W1 = torch.randint(-16, 17, (256, kx), generator=g).float() / 8
    b1 = torch.randint(-32, 33, (256,), generator=g).float() / 16
    W2 = torch.randn(128, 256, generator=g) * 0.1
    expo = torch.randint(-6, 7, (n_src,), generator=g)
    G = torch.randn(n_src, 128, generator=g) * torch.pow(10.0, expo.double()).float()[:, None]
    xr = torch.randperm(n_src, generator=g)[:M].int() if gather else None
    gr = torch.randperm(n_src, generator=g)[:M].int() if gather else None
    return n_src, X, W1, b1, W2, G, xr, gr, expo


@pytest.mark.gpu
@pytest.mark.parametrize("M,kx,gather", [(1, 2, True), (127, 1, True), (128, 2, False), (129, 2, True), (129, 1, False),
                                         (100003, 2, True), (100003, 1, False)])
def test_selfmlp_gen_bwd1_dx_vs_fp64(mods, M, kx, gather):
    """dX[x_rows[m]] = ((G[g_rows[m]] W2) * (W1 x + b1 > 0)) W1 against fp64, every element at the test_selfmlp_* bar
    (rtol 1e-4, atol 2e-5 of the scale) with the scale taken per order of magnitude of G's rows (the kernel scales
    each row on its own); rows no m maps to stay untouched; dW1 / db1 are bitwise tm_selfmlp_gen_bwd1's; bit-identical
    on a second call."""
    lib = mods["lib"]
    n_src, X, W1, b1, W2, G, xr, gr, expo = _bwd1_inputs(M, kx, gather, M + kx)
    xs = X[xr.long()] if gather else X[:M]
    gs = G[gr.long()] if gather else G[:M]
    pre = xs.double() @ W1.double().t() + b1.double()
    assert int((pre == 0).sum()) > 0 or M < 100
    ref = ((gs.double() @ W2.double()) * (pre > 0)) @ W1.double()
    gexp = expo[gr.long()] if gather else expo[:M]
    X, W1, b1, W2, G = (t.to(DEV) for t in (X, W1, b1, W2, G))
    xr_d, gr_d = (None if t is None else t.to(DEV) for t in (xr, gr))
    nb = lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")

    def run(dx_variant):
        dW1, db1 = torch.empty(256, kx, device=DEV), torch.empty(256, device=DEV)
        dX = torch.full((n_src, kx), -7.0, device=DEV)
        if dx_variant:
            lib.call("tm_selfmlp_gen_bwd1_dx", M, G, 128, gr_d, X, kx, xr_d, kx, W1, b1, W2, dW1, db1, dX, kx,
                     lib.workspace(nb, DEV), nb, lib.stream())
        else:
            lib.call("tm_selfmlp_gen_bwd1", M, G, 128, gr_d, X, kx, xr_d, kx, W1, b1, W2, dW1, db1,
                     lib.workspace(nb, DEV), nb, lib.stream())
        return dW1, db1, dX
    dW1, db1, dX = run(True)
    rows = xr.long() if gather else torch.arange(M)
    got = dX.cpu()[rows]
    for e in torch.unique(gexp).tolist():
        sel = gexp == e
        assert_close(got[sel], ref[sel], 1e-4, 2e-5, f"dX (rows of |G| ~ 1e{e})")
    untouched = torch.ones(n_src, dtype=torch.bool)
    untouched[rows] = False
    assert bool((dX.cpu()[untouched] == -7.0).all())
    dW1p, db1p, _ = run(False)
    assert torch.equal(dW1, dW1p) and torch.equal(db1, db1p), "dW1 / db1 differ from tm_selfmlp_gen_bwd1"
    dW1b, db1b, dXb = run(True)
    assert torch.equal(dX, dXb) and torch.equal(dW1, dW1b) and torch.equal(db1, db1b), "not bit-deterministic"


@pytest.mark.parametrize("kx,G,ws_bytes,dX,lddx,what", [
    (3, 256, 1 << 30, 256, 3, "1 or 2 inputs"),
    (2, 260, 1 << 30, 256, 2, "16-byte aligned"),
    (2, 256, 1024, 256, 2, "workspace too small"),
    (2, 256, 1 << 30, None, 2, "dX missing"),
    (2, 256, 1 << 30, 256, 1, "lddx"),
])
def test_selfmlp_gen_bwd1_dx_rejects_unserved_arguments(mods, kx, G, ws_bytes, dX, lddx, what):
    """Unserved arguments fail with an error before any launch (no device needed: the pointers are never read)."""
    lib = mods["lib"]
    before = lib.launch_count()
    with pytest.raises(RuntimeError, match=f"tm_selfmlp_gen_bwd1_dx.*{what}"):
        lib.call("tm_selfmlp_gen_bwd1_dx", 1000, G, 128, None, 256, kx, None, kx, 256, 256, 256, 256, 256, dX, lddx,
                 256, ws_bytes, None)
    assert lib.launch_count() == before


# ------------------------------------------------------------------------------------------------------------------
# oracle
# ------------------------------------------------------------------------------------------------------------------
def _oracle(sd_m, sd_c, od, cnn, pooling="max", rounding=None, forced=None, gate=None, seed=None):
    """``restate.design_step``'s computation with cell_feat, net_feat and the image as leaves.  Returns (pred, H,
    {input: gradient}, {parameter: gradient}) of the MSE, or of <pred, seed> when ``seed`` is given."""
    P = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd_m.items()}
    C = {k: (v.detach().clone().requires_grad_(v.is_floating_point() and "running" not in k)) for k, v in sd_c.items()}
    x = {k: od[k].detach().clone().float().requires_grad_(True) for k in KEYS}
    if cnn == "unet":
        fmap, _ = restate.unet_forward(C, x["image"], pooling, rounding=rounding, forced=forced)
    else:
        fmap = _layoutnet_oracle(C, x["image"], pooling, rounding=rounding, forced=forced)
    feat = fmap.reshape(1, -1)
    H = restate.gnn_propagate(P, "gnn", od["n"], od["levels"], od["net_csr"], od["cell_csr"], x["cell_feat"],
                              x["net_feat"], gate=gate)
    preds = []
    ep, el = od["endpoints"], od["endpoint_level"]
    for lid in torch.unique(el).tolist():
        sel = torch.nonzero(el == lid).squeeze(1)
        dm = restate.dense_mask_rows(od["mask_indptr"], od["mask_cols"], sel.tolist(), feat.shape[1])
        preds.append(restate.head_level(P, H[ep[sel]], dm * feat, lid))
    pred = torch.cat(preds)
    obj = F.mse_loss(pred, od["arrival_time"]) if seed is None else (pred * seed).sum()
    pn = [k for k, v in P.items() if v.requires_grad] + ["cnn." + k for k, v in C.items() if v.requires_grad]
    pt = [v for v in P.values() if v.requires_grad] + [v for v in C.values() if v.requires_grad]
    gr = torch.autograd.grad(obj, [x[k] for k in KEYS] + pt, allow_unused=True)
    return pred.detach(), H.detach(), dict(zip(KEYS, gr[:3])), dict(zip(pn, gr[3:]))


def _setup(mods, cnn, cfg="tiny", pooling="max", math=None, seed=0):
    eng = mods["engine"]
    d = _layout_design(cfg, seed=seed) if cnn == "layoutnet" else tm_synth.make_design(seed=seed, **tm_synth.CONFIGS[cfg])
    model, net = eng.build_models(d.map_size, pooling=pooling, seed=seed, device=DEV, cnn=cnn)
    if math:
        net.math = math
    sd_m = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    sd_c = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    return d, model, net, sd_m, sd_c


def _forced_and_gate(mods, cnn, model, net, b):
    """The product's convolution outputs (same deterministic forward as the step's) and its propagation output H."""
    with torch.no_grad():
        H = model.gnn.propagate(b.graph)
        if cnn == "unet":
            _, ust = mods["unet"].unet_forward(net, b.image, need_bwd=False, update_stats=False)
            Hh, Ww = b.image.shape[-2:]
            forced = _unet_forced(ust, 1, Hh, Ww)
        else:
            _, st = mods["unet"].layoutnet_forward(net, b.image, need_bwd=False)
            forced = _layoutnet_forced(st)
    return {k: v.float() for k, v in forced.items()}, H


def _check_step(mods, cnn, pooling, math=None, cfg="tiny", seed=0, with_seed=False):
    eng = mods["engine"]
    d, model, net, sd_m, sd_c = _setup(mods, cnn, cfg, pooling, math, seed)
    b = eng.DesignBatch.from_synth(d, DEV)
    T = int(b.endpoints.numel())
    pg = torch.randn(T, generator=torch.Generator().manual_seed(seed + 1)) if with_seed else None
    loss, pred = eng.DesignStep(model, net).run(b, input_grads=True,
                                                pred_grad=None if pg is None else pg.to(DEV))
    torch.cuda.synchronize()
    ig = b.input_grads
    assert set(ig) == set(KEYS)
    for k in KEYS:
        assert ig[k].shape == getattr(b, k).shape and ig[k].dtype == torch.float32, k
    # rows the propagation never reads are exactly zero
    sched = b.graph.schedule()
    for k, own in (("cell_feat", sched.cell_class), ("net_feat", sched.net_class)):
        other = torch.ones(d.n, dtype=torch.bool, device=DEV)
        other[own.long()] = False
        assert bool((ig[k][other] == 0).all()), f"{k}: a row the propagation never reads is not zero"
    forced, H = _forced_and_gate(mods, cnn, model, net, b)
    od = design_to_oracle(d)
    rounding = "bf16" if math == "bf16" else None
    _, Hfree, _, _ = _oracle(sd_m, sd_c, od, cnn, pooling, rounding=rounding, forced=forced)
    relu_gate_flips(H, Hfree)                     # any disagreeing output gate is a proven tie ...
    ref_pred, _, rin, rpar = _oracle(sd_m, sd_c, od, cnn, pooling, rounding=rounding, forced=forced,
                                     gate=(H.detach().cpu() > 0), seed=pg)   # ... and takes the product's side here
    assert_close(pred, ref_pred, 2e-2 if rounding else 1e-3, 2e-2 if rounding else 1e-4, "pred")
    for k in ("cell_feat", "net_feat"):
        assert_close(ig[k], rin[k], 1e-3, 2e-4, f"d{k}")
    rtol = 2e-2 if rounding else 1e-3
    assert_close(ig["image"], rin["image"], rtol, 2e-2 if rounding else 2e-4, "dimage")
    return model, net, rpar


# ------------------------------------------------------------------------------------------------------------------
# 2. the step against the oracle
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
@pytest.mark.parametrize("pooling", ["max", "avg"])
def test_step_input_grads_vs_oracle(mods, math_mode, cnn, pooling):
    """Tiny design, fp32-class modes: cell_feat / net_feat / image gradients at rtol 1e-3, atol 2e-4 x max|ref|."""
    _check_step(mods, cnn, pooling)


@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_step_input_grads_bf16_image_mode(mods, cnn):
    """bf16 image mode: against the oracle whose image network rounds its operands to bf16 and is teacher-forced; the
    image gradient at rtol 2e-2, the feature gradients at the fp32 bar."""
    _check_step(mods, cnn, "max", math="bf16")


@pytest.mark.gpu
def test_config2_step_input_grads(mods):
    """The config-2 step in the default arithmetic (tf32x3, U-Net on the TMA-fed kernels) against the fp32 oracle."""
    assert mods["ops"].MATH == "tf32x3"
    _check_step(mods, "unet", "max", cfg="c2")


# ------------------------------------------------------------------------------------------------------------------
# 3. pred_grad
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_pred_grad_is_the_vjp_of_the_predictions(mods, cnn):
    """Seeded by the caller: input and parameter gradients are autograd.grad(pred, inputs + params, seed) of the
    oracle."""
    model, net, rpar = _check_step(mods, cnn, "max", with_seed=True)
    for k, p in model.named_parameters():
        if rpar.get(k) is not None:
            assert_close(p.grad, rpar[k], 1e-3, 2e-4, k)
    for k, p in net.named_parameters():
        if k.endswith(".up.bias"):                 # cancelling sum ahead of a batch norm: scaled to the weight's gradient
            r, wscale = rpar["cnn." + k].double(), float(rpar["cnn." + k[:-4] + "weight"].abs().max())
            assert bool(((p.grad.double().cpu() - r).abs() <= 1e-3 * r.abs() + 2e-4 * wscale).all()), k
            continue
        assert_close(p.grad, rpar["cnn." + k], 1e-3, 2e-4, "cnn." + k)


def _snapshot(model, net, b, loss, pred):
    grads = {k: p.grad.clone() for k, p in list(model.named_parameters()) + [("cnn." + k, p) for k, p in
                                                                             net.named_parameters()] if p.grad is not None}
    ig = {k: v.clone() for k, v in b.input_grads.items()} if b.input_grads is not None else None
    return loss.clone(), pred.clone(), grads, ig


@pytest.mark.gpu
def test_pred_grad_with_the_mse_gradient_is_the_default_step(mods):
    """Seeding with the default step's own dLoss/dpred reproduces its parameter and input gradients (1e-6); the loss
    is still computed."""
    eng = mods["engine"]
    d, model, net, _, _ = _setup(mods, "unet")
    step = eng.DesignStep(model, net)
    b = eng.DesignBatch.from_synth(d, DEV)
    ref = _snapshot(model, net, b, *step.run(b, input_grads=True))
    T = int(b.endpoints.numel())
    seed = (2.0 / T) * (ref[1] - b.arrival_time)
    got = _snapshot(model, net, b, *step.run(b, input_grads=True, pred_grad=seed.contiguous()))
    torch.cuda.synchronize()
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    for what, a, r in [(k, got[2][k], ref[2][k]) for k in ref[2]] + [(k, got[3][k], ref[3][k]) for k in KEYS]:
        # (a bias ahead of conv3x3 + batch norm is a cancelling sum: scaled to its layer's weight gradient, as in
        #  test_config2_full_step_vs_oracle)
        r_scale = ref[2][what[:-4] + "weight"] if what.endswith(".up.bias") else r
        scale = max(float(r_scale.abs().max()), 1e-30)
        assert float((a - r).abs().max()) <= 1e-6 * scale, what
    with pytest.raises(ValueError, match="pred_grad"):
        step.run(b, pred_grad=seed[:-1].contiguous())
    with pytest.raises(ValueError, match="grad_scale"):
        step.run(b, grad_scale=0.5, pred_grad=seed.contiguous())


# ------------------------------------------------------------------------------------------------------------------
# 4. invariants
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cnn,math", [("unet", None), ("layoutnet", "bf16")])
def test_input_grads_leave_the_step_unchanged(mods, cnn, math):
    """Loss, predictions and every parameter gradient are the same bits with input_grads on and off; two runs give
    the same input gradients bit for bit."""
    eng = mods["engine"]
    d, model, net, _, _ = _setup(mods, cnn, math=math)
    step = eng.DesignStep(model, net)
    b = eng.DesignBatch.from_synth(d, DEV)
    off = _snapshot(model, net, b, *step.run(b))
    assert off[3] is None
    on = [_snapshot(model, net, b, *step.run(b, input_grads=True)) for _ in range(2)]
    torch.cuda.synchronize()
    for r in on:
        assert torch.equal(r[0], off[0]) and torch.equal(r[1], off[1])
        assert set(r[2]) == set(off[2])
        for k in off[2]:
            assert torch.equal(r[2][k], off[2][k]), k
    for k in KEYS:
        assert torch.equal(on[0][3][k], on[1][3][k]), k


@pytest.mark.gpu
def test_input_grads_capture_and_prepare(mods):
    """A captured step (input_grads + pred_grad) replayed after the features, the image and the seed were refreshed in
    place equals an eager run on the new values, bit for bit; prepare(..., input_grads=True) likewise."""
    eng = mods["engine"]
    d, model, net, _, _ = _setup(mods, "unet")
    step = eng.DesignStep(model, net)
    b = eng.DesignBatch.from_synth(d, DEV)
    T = int(b.endpoints.numel())
    seed = torch.randn(T, device=DEV)
    replay = step.capture(b, input_grads=True, pred_grad=seed)
    b.cell_feat.mul_(0.5)
    b.net_feat.add_(0.25)
    b.image.copy_(b.image.flip(-1))
    seed.copy_(torch.randn(T, device=DEV))
    got = _snapshot(model, net, b, *replay())
    b2 = eng.DesignBatch.from_synth(d, DEV)
    b2.cell_feat.copy_(b.cell_feat)
    b2.net_feat.copy_(b.net_feat)
    b2.image.copy_(b.image)
    ref = _snapshot(model, net, b2, *step.run(b2, input_grads=True, pred_grad=seed.clone()))
    torch.cuda.synchronize()
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    for k in ref[2]:
        assert torch.equal(got[2][k], ref[2][k]), k
    for k in KEYS:
        assert torch.equal(got[3][k], ref[3][k]), k
    # prepare: new host values, replay, against an eager run on them
    d2 = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["tiny"])
    d2.cell_feat = (d.cell_feat * 0.5).astype(np.float32)
    d2.image = np.ascontiguousarray(d.image[:, ::-1, :]).astype(np.float32)
    host2 = eng.HostDesign(d2, pin=True)
    prep = step.prepare(eng.HostDesign(d, pin=True), DEV, input_grads=True)
    got = _snapshot(model, net, prep.batch, *prep.step(host2))
    b3 = eng.DesignBatch.from_host(host2, DEV)
    ref = _snapshot(model, net, b3, *step.run(b3, input_grads=True))
    torch.cuda.synchronize()
    assert torch.equal(got[0], ref[0])
    for k in KEYS:
        assert torch.equal(got[3][k], ref[3][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,seed,keep", [("tiny", 3, 0.15), ("c1", 5, 0.05)])
def test_pruned_step_input_grads(mods, cfg, seed, keep):
    """prune=True: the input gradients of the whole-netlist step, at the bar of test_design_step_on_cone_subnetlist
    (2e-5 of the scale); pins outside the cone have exactly zero feature gradients."""
    eng = mods["engine"]
    d = tm_synth.make_design(seed=seed, **tm_synth.CONFIGS[cfg])
    rng = np.random.default_rng(seed)
    T = len(d.endpoints)
    sel = np.sort(rng.choice(T, size=max(2, int(T * keep)), replace=False))
    model, net = eng.build_models(d.map_size, seed=seed, device=DEV)
    host = eng.HostDesign(d, pin=False)
    out = {}
    for prune in (False, True):
        b = eng.DesignBatch.from_host(host, DEV)
        idx = torch.from_numpy(sel).to(DEV)
        b = eng.DesignBatch(b.graph, b.mask_csr, b.endpoints[idx].contiguous(), b.endpoint_level[idx].contiguous(),
                            b.arrival_time[idx].contiguous(), b.image, cell_feat=b.cell_feat, net_feat=b.net_feat,
                            rows=idx.int().contiguous())
        eng.DesignStep(model, net, prune=prune).run(b, input_grads=True)
        torch.cuda.synchronize()
        out[prune] = ({k: v.clone() for k, v in b.input_grads.items()}, b.cone())
    cone = out[True][1]
    assert cone.fraction < 1.0
    for k in KEYS:
        g, r = out[True][0][k], out[False][0][k]
        scale = max(float(r.abs().max()), 1e-30)
        assert float((g - r).abs().max()) <= 2e-5 * scale, k
    for k in ("cell_feat", "net_feat"):
        assert bool((out[True][0][k][~cone.active] == 0).all()), k


@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_three_designs_input_grads(mods, cnn):
    """K = 3 joined designs: design k's rows (pin_off_h) and image are 1/3 of its single-design input gradients --
    features at tests/dp_equivalence.py's bar (rtol 1e-5 + 1e-6 of the scale), the image at
    test_three_designs_equal_the_mean_of_single_steps's bar for the image network (rtol 1e-3 + 2e-3 of the scale):
    its convolutions run as one batch of K images instead of K batches of one."""
    eng = mods["engine"]
    ds = [_design(cnn, 11, 5000, 1350), _design(cnn, 12, 3500, 900), _design(cnn, 13, 4200, 1100)]
    model_s, net_s = _models(mods, cnn, None)
    step_s = eng.DesignStep(model_s, net_s)
    singles = []
    for d in ds:
        b = eng.DesignBatch.from_synth(d, DEV)
        step_s.run(b, input_grads=True)
        torch.cuda.synchronize()
        singles.append({k: v.clone() for k, v in b.input_grads.items()})
    model, net = _models(mods, cnn, None)
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(d, DEV) for d in ds])
    eng.DesignStep(model, net).run(b, input_grads=True)
    torch.cuda.synchronize()
    ig = b.input_grads
    for k in KEYS:
        assert ig[k].shape == getattr(b, k).shape, k
    # A LayoutNet layer's output at batch K may differ in the last bits from batch 1; where that flips a ReLU gate (a
    # proven tie: conftest.relu_gate_flips), the gradient of the gate's receptive field takes another route, so that
    # design's image gradient is not compared per element.
    tied = set()
    if cnn == "layoutnet":
        with torch.no_grad():
            _, stK = mods["unet"].layoutnet_forward(net, b.image, need_bwd=False)
            for i in range(len(ds)):
                _, st1 = mods["unet"].layoutnet_forward(net, b.image[i], need_bwd=False)
                for rK, r1 in zip(stK["layers"], st1["layers"]):
                    if relu_gate_flips(rK["y"].reshape(len(ds), -1, rK["cout"])[i], r1["y"].reshape(-1, r1["cout"])):
                        tied.add(i)
    assert len(tied) < len(ds)
    for i, s in enumerate(singles):
        p0, p1 = int(b.pin_off_h[i]), int(b.pin_off_h[i + 1])
        for k in ("cell_feat", "net_feat"):
            # the joined step differs from a single one in the last bits (its seed carries the 1/K, an output gate of
            # the propagation may sit at a tie), and an element is a 256-term sum that may cancel far below its terms:
            # up to 4 elements per design may miss the relative bar, by at most 50x
            assert_close(ig[k][p0:p1], s[k] / 3, 1e-5, 1e-6, f"{k} of design {i}", max_bad=4, flip_factor=50.0)
        if i in tied:
            continue
        r = s["image"].double() / 3
        err = (ig["image"][i].double() - r).abs()
        bad = int((err > 1e-3 * r.abs() + 2e-3 * float(r.abs().max())).sum())
        assert bad == 0, f"image of design {i}: {bad}/{r.numel()} elements off (max err {float(err.max()):.3e})"
