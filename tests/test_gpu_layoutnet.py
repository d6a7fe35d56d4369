"""LayoutNet (model.py:216-247, the reference's default image network) on the fast paths:
  * the TMA-fed tcgen05 k x k convolutions of its bf16 mode (tm_convkxk_bf16*, csrc/tm_tma.cu) against fp64 PyTorch
    on the same bf16-rounded operands, at the bar of the 3x3 kernels (rtol 1e-4, atol 1e-5 x max|ref|);
  * the whole network in bf16 mode against the bf16-rounded oracle (``_layoutnet_oracle(rounding="bf16")`` below);
  * the fused design step (tm_engine.DesignStep) with a LayoutNet, fp32-class and bf16, against
    restate.design_step(cnn="layoutnet"), and its CUDA-graph capture, prepared designs, shuffled-batch replay and
    cone pruning against the eager step.

``_layoutnet_oracle`` is restate.layoutnet_forward (model.py:216-247) with the two oracle modes restate.unet_forward
has: bf16 operand rounding at the product's rounding points, and teacher forcing.  With neither it computes exactly
what restate.layoutnet_forward computes; design_step is pointed at it through ``monkeypatch``."""
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import tm_synth
from conftest import assert_close, assert_grad_close_given_flips, design_to_oracle, relu_gate_flips
from oracle import restate

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def mods(pkg):
    import tm_engine, tm_lib, tm_loader, tm_ops, tm_unet  # noqa: E401
    yield dict(engine=tm_engine, lib=tm_lib, loader=tm_loader, ops=tm_ops, unet=tm_unet)
    tm_lib.check_err_flags()                     # no tensor-core barrier ever timed out


@pytest.fixture(params=["tf32x3", "tc6", "fp32"])
def math_mode(request, mods):
    old = mods["ops"].MATH
    mods["ops"].MATH = request.param
    yield request.param
    mods["ops"].MATH = old


def _bf(t):
    return t.bfloat16().float()


def _nhwc_bf16(lib, t):
    B, C, H, W = t.shape
    src = t.detach().permute(0, 2, 3, 1).contiguous()
    out = torch.empty(B * H * W, C, dtype=torch.bfloat16, device=DEV)
    lib.call("tm_to_bf16_rows", B * H * W, C, src, C, out, C, lib.stream())
    return out


def _rows(t):
    """(B,C,H,W) -> NHWC rows (B*H*W, C)."""
    return t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])


# ------------------------------------------------------------------------------------------------------------------
# oracle: LayoutNet with bf16 operand rounding and teacher forcing
# ------------------------------------------------------------------------------------------------------------------
class _ConvBf16(torch.autograd.Function):
    """k x k convolution (stride 1, zero padding k//2) whose three contractions see bf16-rounded operands: x and w are
    rounded when they become tensor-core operands, the incoming gradient is rounded ONCE and that copy feeds the data
    and the weight gradient, the bias gradient sums the unrounded gradient -- the rounding points of the product's
    bf16 mode on either convolution route (restate._ContractBf16 for the U-Net's 3x3 layers)."""

    @staticmethod
    def forward(ctx, x, w, b):
        xb, wb = restate._bf16_rn(x.detach()), restate._bf16_rn(w.detach())
        ctx.save_for_backward(xb, wb)
        return F.conv2d(xb, wb, b, padding=wb.shape[-1] // 2)

    @staticmethod
    def backward(ctx, g):
        xb, wb = ctx.saved_tensors
        with torch.enable_grad():
            x_, w_ = xb.detach().requires_grad_(True), wb.detach().requires_grad_(True)
            dx, dw = torch.autograd.grad(F.conv2d(x_, w_, None, padding=w_.shape[-1] // 2), (x_, w_), restate._bf16_rn(g))
        return dx, dw, g.sum((0, 2, 3))


def _layoutnet_oracle(sd, x, pooling="max", rounding=None, forced=None):
    """``rounding="bf16"``: every convolution through ``_ConvBf16``.  ``forced``: {"encode.<0|3|6|8>": (B,C,H,W)} --
    the convolution's output including its bias takes that VALUE while gradients flow through it (restate._force)."""
    batched = x.dim() == 3 and (rounding is not None or forced is not None)    # (C,H,W) -> (1,C,H,W) like `forced`

    def conv(y, i):
        w, b = sd[f"encode.{i}.weight"], sd[f"encode.{i}.bias"]
        z = F.conv2d(y, w, b, padding=w.shape[-1] // 2) if rounding is None else _ConvBf16.apply(y, w, b)
        return restate._force(z, forced, f"encode.{i}")
    y = x.unsqueeze(0) if batched else x
    y = restate._pool(F.relu(conv(y, 0)), pooling)
    y = restate._pool(F.relu(conv(y, 3)), pooling)
    y = F.relu(conv(y, 6))
    y = F.leaky_relu(conv(y, 8), 0.1)
    return y[0] if batched else y


def _design_step(monkeypatch, *args, rounding=None, forced=None, **kw):
    """restate.design_step(cnn="layoutnet") with its LayoutNet in the oracle modes of ``_layoutnet_oracle``."""
    with monkeypatch.context() as m:
        m.setattr(restate, "layoutnet_forward", functools.partial(_layoutnet_oracle, rounding=rounding, forced=forced))
        return restate.design_step(*args, cnn="layoutnet", **kw)


def test_layoutnet_oracle_modes_off_is_restate():
    """Without rounding and forcing the test's oracle is restate.layoutnet_forward, bit for bit; forcing every
    convolution with its own output changes nothing either."""
    import model as M
    torch.manual_seed(2)
    sd = {k: v.detach().clone() for k, v in M.LayoutNet("max").state_dict().items()}
    x = torch.rand(2, 32, 32)
    ref = restate.layoutnet_forward(sd, x, "max")
    assert torch.equal(_layoutnet_oracle(sd, x, "max"), ref)
    xb = x.unsqueeze(0)
    z0 = F.conv2d(xb, sd["encode.0.weight"], sd["encode.0.bias"], padding=4)
    forced = {"encode.0": z0}
    assert torch.allclose(_layoutnet_oracle(sd, x, "max", forced=forced), ref, rtol=1e-6, atol=1e-7)


# ------------------------------------------------------------------------------------------------------------------
# 1. kernels against fp64
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,Cin,Cout,B,H,W", [(7, 32, 64, 1, 256, 256), (9, 64, 32, 1, 128, 128), (7, 32, 64, 2, 16, 32),
                                              (9, 64, 32, 1, 8, 8)])
def test_convkxk_bf16_tma(mods, k, Cin, Cout, B, H, W):
    """Forward without and with bias + ReLU, data gradient (tap-reversed operand) and weight gradient (taps in groups,
    partials folded in a fixed order): against fp64 on the same bf16 operands, and bit-identical on a second run."""
    lib = mods["lib"]
    torch.manual_seed(k + Cin + B + H + W)
    assert lib.ws_bytes("tm_convkxk_bf16_supported", B, H, W, Cin, Cout, k) == 1
    x = _bf(torch.randn(B, Cin, H, W, device=DEV)).requires_grad_(True)
    w = _bf(torch.randn(Cout, Cin, k, k, device=DEV) * 0.05).requires_grad_(True)
    g = _bf(torch.randn(B, Cout, H, W, device=DEV))
    bias = torch.randn(Cout, device=DEV)
    ref = F.conv2d(x.double(), w.double(), None, padding=k // 2)
    gx, gw = torch.autograd.grad(ref, (x, w), g.double())
    xb, gb = _nhwc_bf16(lib, x), _nhwc_bf16(lib, g)
    wq = torch.empty(k * k, Cout, Cin, dtype=torch.bfloat16, device=DEV)
    wd = torch.empty(k * k, Cin, Cout, dtype=torch.bfloat16, device=DEV)
    lib.call("tm_convkxk_pack_bf16", Cout, Cin, k, w.detach().contiguous(), wq, Cin, 0, lib.stream())
    lib.call("tm_convkxk_pack_bf16", Cout, Cin, k, w.detach().contiguous(), wd, Cout, 1, lib.stream())
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    npix = B * H * W

    def fwd(b, flags):
        y = torch.empty(npix, Cout, device=DEV)
        lib.call("tm_convkxk_bf16", B, H, W, Cin, Cout, k, xb, wq, b, y, Cout, flags, err, lib.stream())
        return y
    y0 = fwd(None, 0)
    assert_close(y0, _rows(ref), 1e-4, 1e-5, "kxk fprop")
    y1 = fwd(bias, 2)
    assert_close(y1, _rows(torch.relu(ref + bias.double().view(1, -1, 1, 1))), 1e-4, 1e-5, "kxk fprop + bias + ReLU")
    assert torch.equal(y1, fwd(bias, 2)), "forward is not bit-deterministic"

    def dgrad():
        dx = torch.empty(npix, Cin, device=DEV)
        lib.call("tm_convkxk_bf16", B, H, W, Cout, Cin, k, gb, wd, None, dx, Cin, 0, err, lib.stream())
        return dx
    dx = dgrad()
    assert_close(dx, _rows(gx), 1e-4, 1e-5, "kxk dgrad")
    assert torch.equal(dx, dgrad()), "data gradient is not bit-deterministic"
    nb = lib.ws_bytes("tm_convkxk_bf16_wgrad_ws", B, H, W, Cin, Cout, k)

    def wgrad():
        dw = torch.empty(Cout, Cin, k, k, device=DEV)
        lib.call("tm_convkxk_bf16_wgrad", B, H, W, Cin, Cout, k, xb, gb, dw, lib.workspace(nb, DEV), nb, err, lib.stream())
        return dw
    dw = wgrad()
    assert_close(dw, gw, 1e-4, 1e-5, "kxk wgrad")
    assert torch.equal(dw, wgrad()), "weight gradient is not bit-deterministic"
    assert int(err.item()) == 0


@pytest.mark.parametrize("k,Cin,Cout,H,W", [(7, 2, 32, 64, 64), (7, 32, 1, 64, 64), (8, 32, 64, 64, 64),
                                            (11, 32, 64, 64, 64), (7, 32, 64, 48, 64), (9, 128, 32, 64, 64)])
def test_convkxk_bf16_unsupported_shape_does_not_launch(mods, k, Cin, Cout, H, W):
    lib = mods["lib"]
    assert lib.ws_bytes("tm_convkxk_bf16_supported", 1, H, W, Cin, Cout, k) == 0
    x = torch.zeros(H * W, max(Cin, 16), dtype=torch.bfloat16, device=DEV)
    wq = torch.zeros(max(k, 1) ** 2 * max(Cout, 16) * max(Cin, 16), dtype=torch.bfloat16, device=DEV)
    y = torch.empty(H * W, max(Cout, 16), device=DEV)
    before = lib.launch_count()
    with pytest.raises(RuntimeError):
        lib.call("tm_convkxk_bf16_wgrad", 1, H, W, Cin, Cout, k, x, x, y, y, y.numel() * 4, None, lib.stream())
    if Cin % 16 or Cout % 16 or k not in (3, 5, 7, 9) or H & (H - 1):
        with pytest.raises(RuntimeError):
            lib.call("tm_convkxk_bf16", 1, H, W, Cin, Cout, k, x, wq, None, y, max(Cout, 16), 0, None, lib.stream())
    torch.cuda.synchronize()
    assert lib.launch_count() == before


# ------------------------------------------------------------------------------------------------------------------
# 2. LayoutNet in bf16 mode against the bf16-rounded oracle
# ------------------------------------------------------------------------------------------------------------------
def _forced(st):
    """The product's convolution outputs (after the fused bias / ReLU epilogue; the last one before its LeakyReLU) as
    the oracle's NCHW tensors, keyed like restate._force.  Forcing relu(z) onto z leaves relu(z) and its gate as the
    product's."""
    B = st["B"]
    return {r["name"]: r["y"].detach().float().reshape(B, r["H"], r["W"], r["cout"]).permute(0, 3, 1, 2).contiguous().cpu()
            for r in st["layers"]}


@pytest.mark.parametrize("B,H,pooling", [(1, 512, "max"), (2, 64, "max"), (2, 64, "avg")])
def test_layoutnet_bf16_vs_rounded_oracle(mods, B, H, pooling):
    """encode.3 (7x7) and encode.6 (9x9) run on the TMA route, encode.0 / encode.8 on the cp.async one.  Output
    against the free-running bf16-rounded oracle; EVERY parameter gradient, per element, against that oracle
    teacher-forced with the product's convolution outputs (same ReLU gates and max-pool winners), rtol 2e-2.  No
    tensor needs a special case: LayoutNet has no BatchNorm, so no bias gradient is a cancelling sum."""
    import model as M
    unet = mods["unet"]
    torch.manual_seed(5)
    net = M.LayoutNet(pooling).train()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    names = [k for k, _ in net.named_parameters()]
    x = torch.rand(B, 2, H, H)
    net = net.to(DEV)
    net.math = "bf16"
    out, st = unet.layoutnet_forward(net, x.to(DEV), need_bwd=True)
    routes = {r["name"]: r["tma"] for r in st["layers"]}
    assert routes == {"encode.0": False, "encode.3": True, "encode.6": True, "encode.8": False}, routes
    out2, _ = unet.layoutnet_forward(net, x.to(DEV), need_bwd=False)
    assert torch.equal(out, out2), "forward is not bit-deterministic"

    def oracle(forced):
        P = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        return _layoutnet_oracle(P, x, pooling, rounding="bf16", forced=forced), P
    free, _ = oracle(None)
    assert_close(out, free, 2e-2, 2e-2, "layoutnet out vs free-running bf16 oracle")
    g = torch.randn(B, 1, H // 4, H // 4, generator=torch.Generator().manual_seed(9))
    grads = unet.layoutnet_backward(net, st, g.to(DEV))
    ref, P = oracle(_forced(st))
    gref = torch.autograd.grad(ref, [P[k] for k in names], g)
    for k, r in zip(names, gref):
        assert_close(grads[k].reshape(r.shape), r, 2e-2, 2e-2, f"grad {k} (bf16, teacher-forced oracle)")


# ------------------------------------------------------------------------------------------------------------------
# 3. / 5. the fused step against restate.design_step(cnn="layoutnet")
# ------------------------------------------------------------------------------------------------------------------
def _layout_design(cfg, seed=0, **kw):
    return tm_synth.make_design(seed=seed, img_channels=2, img_scale=4, **tm_synth.CONFIGS[cfg], **kw)


def _step(mods, d, pooling="max", seed=0, math=None):
    eng = mods["engine"]
    model, cnn = eng.build_models(d.map_size, pooling=pooling, seed=seed, device=DEV, cnn="layoutnet")
    if math:
        cnn.math = math
    sd_m = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    sd_c = {k: v.detach().cpu().clone() for k, v in cnn.state_dict().items()}
    batch = eng.DesignBatch.from_synth(d, DEV)
    loss, pred = eng.DesignStep(model, cnn).run(batch)
    torch.cuda.synchronize()
    with torch.no_grad():
        H = model.gnn.propagate(batch.graph)                  # the same kernels: bit-identical to the step's H
        fmap, st = mods["unet"].layoutnet_forward(cnn, batch.image, need_bwd=False)
    return model, cnn, sd_m, sd_c, loss, pred, H, fmap, st


def _check_fp32_step(mods, monkeypatch, d, pooling):
    model, cnn, sd_m, sd_c, loss, pred, H, fmap, st = _step(mods, d, pooling)
    od = design_to_oracle(d)
    free = restate.design_step(sd_m, sd_c, od, pooling, cnn="layoutnet", with_grad=False)
    assert_close(fmap.reshape(-1), free["feat_map"].reshape(-1), 1e-3, 1e-4, "feature map")
    assert_close(pred, free["pred"], 1e-3, 1e-4, "pred")
    assert_close(loss.reshape(()), free["loss"], 1e-3, 1e-4, "loss")
    # gradients: the oracle's LayoutNet teacher-forced with the product's convolution outputs (ReLU / max-pool ties of
    # the image branch), the propagation's output gates as in the U-Net step tests
    flips = relu_gate_flips(H, free["H"])
    ref = _design_step(monkeypatch, sd_m, sd_c, od, pooling, forced=_forced(st),
                       gnn_gate=(H.detach().cpu() > 0) if flips else None)
    for k, p in model.named_parameters():
        g = ref["grads"][k]
        if g is None:
            assert p.grad is None, k
        elif k.startswith("gnn."):
            assert_grad_close_given_flips(p.grad, g, k, set(), atol_scale=2e-4)
        else:
            assert_close(p.grad, g, 1e-3, 2e-4, k)
    for k, p in cnn.named_parameters():
        assert_close(p.grad, ref["grads"]["cnn." + k], 1e-3, 2e-4, "cnn." + k)


@pytest.mark.parametrize("pooling", ["max", "avg"])
def test_layoutnet_step_vs_oracle(mods, monkeypatch, math_mode, pooling):
    """tiny design, 2x32x32 image: predictions, loss and every parameter gradient of model and LayoutNet."""
    _check_fp32_step(mods, monkeypatch, _layout_design("tiny"), pooling)


def test_layoutnet_config2_full_step_vs_oracle(mods, monkeypatch):
    """config-2 netlist with a 2x512x512 image, default arithmetic (tf32x3)."""
    assert mods["ops"].MATH == "tf32x3"
    _check_fp32_step(mods, monkeypatch, _layout_design("c2"), "max")


@pytest.mark.parametrize("cfg", ["tiny", "c1"])
def test_layoutnet_step_mixed_precision(mods, monkeypatch, cfg):
    """cnn.math = "bf16": predictions and loss against the fp32 oracle at rtol 2e-2; every gradient against the
    bf16-rounded oracle teacher-forced with the product's convolution outputs at rtol 2e-2."""
    d = _layout_design(cfg, seed=1)
    model, cnn, sd_m, sd_c, loss, pred, H, fmap, st = _step(mods, d, seed=1, math="bf16")
    assert [r["tma"] for r in st["layers"]] == [False, True, True, False]
    od = design_to_oracle(d)
    free = restate.design_step(sd_m, sd_c, od, cnn="layoutnet", with_grad=False)
    assert_close(pred, free["pred"], 2e-2, 2e-2, "pred vs fp32 oracle")
    assert_close(loss.reshape(()), free["loss"], 2e-2, 2e-2, "loss vs fp32 oracle")
    ref = _design_step(monkeypatch, sd_m, sd_c, od, rounding="bf16", forced=_forced(st))
    for k, p in model.named_parameters():
        g = ref["grads"][k]
        if g is None:
            assert p.grad is None, k
        else:
            assert_close(p.grad, g, 2e-2, 2e-2, "model." + k)
    for k, p in cnn.named_parameters():
        assert_close(p.grad, ref["grads"]["cnn." + k], 2e-2, 2e-2, "cnn." + k)


# ------------------------------------------------------------------------------------------------------------------
# 4. capture, prepared designs, shuffled batches, pruning
# ------------------------------------------------------------------------------------------------------------------
def _grads(model, cnn):
    return {k: p.grad.clone() for k, p in list(model.named_parameters()) + [("cnn." + k, p) for k, p in cnn.named_parameters()]
            if p.grad is not None}


def _assert_same_step(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert set(a[2]) == set(b[2])
    for k in a[2]:
        assert torch.equal(a[2][k], b[2][k]), k


@pytest.mark.parametrize("math", [None, "bf16"])
def test_layoutnet_step_capture_and_prepare(mods, math):
    """step.capture(b) and prepare(host).step(host2) reproduce the eager step bit for bit."""
    eng = mods["engine"]
    d = _layout_design("tiny", seed=2)
    model, cnn = eng.build_models(d.map_size, seed=2, device=DEV, cnn="layoutnet")
    if math:
        cnn.math = math
    step = eng.DesignStep(model, cnn)
    b = eng.DesignBatch.from_synth(d, DEV)
    loss, pred = step.run(b)
    torch.cuda.synchronize()
    eager = (loss.clone(), pred.clone(), _grads(model, cnn))
    replay = step.capture(b)
    loss_r, pred_r = replay()
    torch.cuda.synchronize()
    _assert_same_step((loss_r.clone(), pred_r.clone(), _grads(model, cnn)), eager)
    # a prepared design fed new values from host memory
    host = eng.HostDesign(d, pin=True)
    prep = step.prepare(host, DEV)
    d2 = _layout_design("tiny", seed=2)
    d2.cell_feat = (d.cell_feat * 0.5).astype(np.float32)
    d2.image = np.ascontiguousarray(d.image[:, ::-1, :]).astype(np.float32)
    host2 = eng.HostDesign(d2, pin=True)
    loss_p, pred_p = prep.step(host2)
    torch.cuda.synchronize()
    got = (loss_p.clone(), pred_p.clone(), _grads(model, cnn))
    loss_e, pred_e = step.run(eng.DesignBatch.from_host(host2, DEV))
    torch.cuda.synchronize()
    _assert_same_step(got, (loss_e.clone(), pred_e.clone(), _grads(model, cnn)))
    assert not torch.equal(loss_p, loss)
    step.close()


def test_layoutnet_loaded_design_shuffled_batches(mods):
    """LoadedDesign.prepare (one capture, endpoint batches refreshed in place) against the eager step on the same
    path ids, over several shuffled batches, with Adam steps between them applied identically to both."""
    eng, ldr = mods["engine"], mods["loader"]
    d = tm_synth.make_design(seed=4, **tm_synth.CONFIGS["tiny"])
    ld = ldr.load_design(ldr.design_tuple_from_synth(d, unet=False), DEV)
    assert tuple(ld.image.shape) == (2, 4 * d.map_size, 4 * d.map_size)
    model, cnn = eng.build_models(d.map_size, seed=4, device=DEV, cnn="layoutnet")
    step = eng.DesignStep(model, cnn)
    bs = 16
    run = ld.prepare(step, batch_size=bs)
    gen = torch.Generator().manual_seed(0)
    for _ in range(3):
        ids = [ld.paths[i] for i in torch.randperm(len(ld.paths), generator=gen)[:bs].tolist()]
        loss_r, pred_r = run(ids)
        torch.cuda.synchronize()
        got = (loss_r.clone(), pred_r.clone(), _grads(model, cnn))
        loss_e, pred_e = step.run(ld.batch(ids))
        torch.cuda.synchronize()
        assert_close(got[0], loss_e, 1e-6, 1e-7, "loss")
        assert_close(got[1], pred_e, 1e-6, 1e-6, "pred")
        for k, g in _grads(model, cnn).items():
            assert_close(got[2][k], g, 1e-6, 1e-6, k)
        step.adam_step({}, lr=1e-3)
    step.close()


def test_layoutnet_step_on_cone_subnetlist(mods):
    """prune=True: same predictions, loss and gradients as the step on the whole netlist (tolerances of
    test_gpu_parity.py::test_design_step_on_cone_subnetlist)."""
    eng = mods["engine"]
    d = _layout_design("c1", seed=4)
    rng = np.random.default_rng(4)
    T = len(d.endpoints)
    sel = np.sort(rng.choice(T, size=max(2, int(T * 0.03)), replace=False))
    model, cnn = eng.build_models(d.map_size, seed=4, device=DEV, cnn="layoutnet")
    host = eng.HostDesign(d, pin=False)
    out = {}
    for prune in (False, True):
        b = eng.DesignBatch.from_host(host, DEV)
        idx = torch.from_numpy(sel).to(DEV)
        b = eng.DesignBatch(b.graph, b.mask_csr, b.endpoints[idx].contiguous(), b.endpoint_level[idx].contiguous(),
                            b.arrival_time[idx].contiguous(), b.image, cell_feat=b.cell_feat, net_feat=b.net_feat,
                            rows=idx.int().contiguous())
        for p in list(model.parameters()) + list(cnn.parameters()):
            p.grad = None
        loss, pred = eng.DesignStep(model, cnn, prune=prune).run(b)
        torch.cuda.synchronize()
        assert (b._cone is not None) == prune
        out[prune] = (loss.clone(), pred.clone(), _grads(model, cnn))
    assert b.cone().fraction < 1.0
    assert_close(out[True][1], out[False][1], 1e-6, 1e-6, "pred")
    assert_close(out[True][0], out[False][0], 1e-6, 1e-7, "loss")
    assert set(out[True][2]) == set(out[False][2])
    for k, gfull in out[False][2].items():
        scale = max(float(gfull.abs().max()), 1e-30)
        assert float((out[True][2][k] - gfull).abs().max()) <= 2e-5 * scale, k


def test_layoutnet_feature_map_must_match_mask_width(mods):
    """An image whose LayoutNet feature map is not map_size**2 pixels is rejected by name, not run into the fusion."""
    eng = mods["engine"]
    d = tm_synth.make_design(seed=0, img_channels=2, img_scale=2, **tm_synth.CONFIGS["tiny"])     # 16x16 -> 4x4 map
    model, cnn = eng.build_models(d.map_size, seed=0, device=DEV, cnn="layoutnet")
    step = eng.DesignStep(model, cnn)
    b = eng.DesignBatch.from_synth(d, DEV)
    with pytest.raises(ValueError, match=r"16 pixels.*64 columns"):
        step.run(b)
    with pytest.raises(ValueError, match=r"16 pixels.*64 columns"):
        step.forward(b)
    torch.cuda.synchronize()
