"""The fused evaluation step: ``DesignStep.evaluate`` / ``capture_evaluate`` / ``prepare(evaluate=True)`` and the loader's
``prepare_evaluate``, with validate()'s and test()'s metrics per design and per level from ``tm_eval_metrics``.

1. ``tm_eval_metrics`` against numpy in fp64: empty, one-element, constant-label and overlapping segments, with and
   without required times / labels; bit-identical launches; the whole-batch row against ``tm_step_metrics``.
2. ``evaluate`` against ``run`` (same bits), ``forward`` (fp32-class) and the reference fixture, and the model left as
   ``forward`` leaves it.
3. Per-design and per-level rows of a joined batch, capture / prepare / prepare_many replays, the loader, the errors.
"""
import types

import numpy as np
import pytest
import torch

import tm_synth
from conftest import assert_close, load_golden_step

DEV = "cuda"
MAPE_EPS = np.float32(1.17e-6)


@pytest.fixture(scope="module")
def mods(pkg):
    import tm_engine, tm_lib, tm_loader, tm_ops  # noqa: E401
    yield dict(engine=tm_engine, lib=tm_lib, loader=tm_loader, ops=tm_ops)
    if torch.cuda.is_available():
        tm_lib.check_err_flags()                 # no tensor-core barrier ever timed out


# ------------------------------------------------------------------------------------------------------------------
# numpy reference
# ------------------------------------------------------------------------------------------------------------------
def _ref_row(pred, y, req, lab, idx):
    """[mse, r2, correct, tp, fn, tn, fp, count, mape] of the endpoints idx, in fp64 (two-pass total sum of squares)."""
    n = len(idx)
    if n == 0:
        return np.array([np.nan, np.nan, 0, 0, 0, 0, 0, 0, np.nan])
    p, t = pred[idx].astype(np.float64), y[idx].astype(np.float64)
    d = p - t
    sst = float(((t - t.mean()) ** 2).sum())
    r2 = 1.0 - float((d * d).sum()) / sst if n >= 2 and sst > 0 else np.nan
    mape = float((np.abs(d) / np.maximum(np.abs(y[idx]), MAPE_EPS).astype(np.float64)).mean())
    counts = [0] * 5
    if req is not None and lab is not None:
        crit = (req[idx] - pred[idx]) < np.float32(0)                 # judge_critical, in fp32 as the kernel does
        l = lab[idx]
        pos = l != 0
        counts = [int(((crit == pos) & ((l == 0) | (l == 1))).sum()), int((crit & pos).sum()), int((~crit & pos).sum()),
                  int((~crit & ~pos).sum()), int((crit & ~pos).sum())]
    return np.array([float((d * d).mean()), r2] + counts + [n, mape])


def _assert_rows(got, ref, rtol=1e-6, what=""):
    """Counts exact; mse / r2 / mape within rtol, NaN exactly where the reference is NaN."""
    got, ref = np.asarray(got, np.float64).reshape(-1, 9), np.asarray(ref, np.float64).reshape(-1, 9)
    assert got.shape == ref.shape, what
    np.testing.assert_array_equal(got[:, 2:8], ref[:, 2:8], err_msg=f"{what}: counts")
    for c, name in ((0, "mse"), (1, "r2"), (8, "mape")):
        np.testing.assert_array_equal(np.isnan(got[:, c]), np.isnan(ref[:, c]), err_msg=f"{what}: NaN pattern of {name}")
        ok = ~np.isnan(ref[:, c])
        np.testing.assert_allclose(got[ok, c], ref[ok, c], rtol=rtol, atol=0, err_msg=f"{what}: {name}")


def _bits(t):
    return t.detach().contiguous().view(torch.int32).clone()        # NaN-safe bitwise comparison


def _host(t):
    return None if t is None else t.detach().cpu().numpy()


def _level_rows(pred, y, req, lab, levels, L):
    return np.stack([_ref_row(pred, y, req, lab, np.nonzero(levels == l)[0]) for l in range(L)])


# ------------------------------------------------------------------------------------------------------------------
# 1. the kernel
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("with_labels", [False, True])
def test_eval_metrics_kernel_vs_fp64(mods, with_labels):
    ops = mods["ops"]
    rng = np.random.default_rng(5 + with_labels)
    T = 7001
    y = (rng.random(T) * 3 + 0.5).astype(np.float32)
    y[:7] = [0.0, 1e-8, -2e-7, 1e-6, -0.3, 2.0, 0.0]               # labels at and around MAPE's clamp
    y[2000:2300] = np.float32(1.625)                                # a constant segment: r2 NaN
    pred = (y + rng.normal(0, 0.4, T)).astype(np.float32)
    req = (y + rng.normal(0, 0.3, T)).astype(np.float32) if with_labels else None
    lab = rng.integers(0, 2, T).astype(np.int64) if with_labels else None
    if with_labels:
        lab[rng.choice(T, 50, replace=False)] = 2                  # neither 0 nor 1: never "correct"
    segs = [np.arange(T), np.array([], np.int64), np.array([17]), np.arange(2000, 2300), np.arange(2100, 2200),
            rng.choice(T, 3000, replace=False), rng.choice(T, 3000, replace=False), np.arange(1, 300),
            np.array([], np.int64), np.arange(0, 7), np.array([5, 5, 5, 9])]
    ptr = np.concatenate([[0], np.cumsum([len(s) for s in segs])]).astype(np.int32)
    idx = np.concatenate(segs).astype(np.int32)
    dv = lambda a: None if a is None else torch.from_numpy(a).to(DEV)          # noqa: E731
    args = (dv(pred), dv(y), dv(ptr), dv(idx), dv(req), dv(lab))
    out = ops.eval_metrics(*args)
    again = ops.eval_metrics(*args)
    torch.cuda.synchronize()
    assert out.shape == (len(segs), 9) and out.dtype == torch.float32
    ref = np.stack([_ref_row(pred, y, req, lab, s) for s in segs])
    _assert_rows(out.cpu().numpy(), ref, 1e-6, "segments")
    assert torch.equal(_bits(out), _bits(again)), "not bit-deterministic"
    assert bool(torch.isnan(out[3, 1])) and int(out[1, 7]) == 0 and bool(torch.isnan(out[2, 1]))
    sm = ops.step_metrics(args[0], args[1], args[4], args[5]).cpu().numpy()
    np.testing.assert_allclose(out[0, :8].cpu().numpy(), sm, rtol=1e-6, atol=0)


# ------------------------------------------------------------------------------------------------------------------
# 2. evaluate against run, forward and the reference fixture; side effects
# ------------------------------------------------------------------------------------------------------------------
def _design(cnn, seed, n_cells, T):
    kw = dict(img_channels=2, img_scale=4) if cnn == "layoutnet" else {}
    return tm_synth.make_design(seed=seed, n_cells=n_cells, n_lv=20, map_size=32, n_endpoints=T, **kw)


def _models(eng, cnn, math, seed=0, map_size=32):
    model, net = eng.build_models(map_size, seed=seed, device=DEV, cnn=cnn)
    if math:
        net.math = math
    return model, net


def _batch(eng, ds, labels=False):
    bs = [eng.DesignBatch.from_synth(d, DEV) for d in ds]
    if labels:
        for k, b in enumerate(bs):
            g = torch.Generator().manual_seed(100 + k)
            T = int(b.endpoints.numel())
            b.required = (b.arrival_time.cpu() + torch.randn(T, generator=g)).to(DEV)
            b.label = torch.randint(0, 2, (T,), generator=g).to(DEV)
    return bs[0] if len(bs) == 1 else eng.DesignBatch.concat(bs)


def _state(model, net):
    named = [("m." + k, p) for k, p in model.named_parameters()] + [("c." + k, p) for k, p in net.named_parameters()]
    bufs = [("m." + k, v) for k, v in model.named_buffers()] + [("c." + k, v) for k, v in net.named_buffers()]
    return dict(params={k: p.detach().clone() for k, p in named},
                grads={k: (p.grad, None if p.grad is None else p.grad.clone()) for k, p in named},
                bufs={k: v.clone() for k, v in bufs})


def _assert_params_and_grads_unchanged(model, net, before):
    after = _state(model, net)
    for k, v in before["params"].items():
        assert torch.equal(after["params"][k], v), f"parameter {k} changed"
    for k, (obj, bits) in before["grads"].items():
        now = after["grads"][k][0]
        assert now is obj, f"{k}.grad was re-pointed"
        assert (bits is None and now is None) or torch.equal(now, bits), f"{k}.grad changed"


def _check_metrics_vs_numpy(b, pred, met):
    """Every row of ``met`` against numpy over the batch's predictions, labels and endpoint levels."""
    p, y = _host(pred), _host(b.arrival_time)
    req, lab = _host(b.required), _host(b.label)
    lv = _host(b.endpoint_level).astype(np.int64)
    L = int(lv.max()) + 1
    h = met.to_host()
    assert h.level.shape == (b.K, L, 9) and h.design.shape == (b.K, 9) and h.batch.shape == (9,)
    _assert_rows(h.batch, _ref_row(p, y, req, lab, np.arange(len(p))), 1e-6, "batch row")
    for k in range(b.K):
        s, e = int(b.ep_off_h[k]), int(b.ep_off_h[k + 1])
        _assert_rows(h.design[k], _ref_row(p, y, req, lab, np.arange(s, e)), 1e-6, f"design {k}")
        sl = lambda a: None if a is None else a[s:e]              # noqa: E731
        _assert_rows(h.level[k], _level_rows(sl(p), sl(y), sl(req), sl(lab), lv[s:e], L), 1e-6, f"levels of design {k}")
    return h


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("cnn,math", [("unet", None), ("layoutnet", "bf16")])
def test_evaluate_vs_run_and_forward(mods, cnn, math, K):
    """U-Net tf32x3 and LayoutNet bf16: evaluate's predictions are run's bits and forward's at the fp32-class bar
    (forward runs the persistent propagation kernel, evaluate the per-level chain run uses); its metric rows are numpy's
    over those predictions."""
    eng = mods["engine"]
    ds = [_design(cnn, 11 + k, 3000 + 600 * k, 500 + 150 * k) for k in range(K)]
    model, net = _models(eng, cnn, math)
    step = eng.DesignStep(model, net)
    b = _batch(eng, ds, labels=True)
    pred, met = step.evaluate(b)
    pred = pred.clone()
    _, pred_run = step.run(b)
    pred_fwd = step.forward(b)
    torch.cuda.synchronize()
    assert pred.shape == (int(b.endpoints.numel()),)
    assert torch.equal(pred, pred_run), "evaluate and run predict different bits"
    assert_close(pred, pred_fwd, 1e-3, 1e-4, "evaluate vs forward")
    _check_metrics_vs_numpy(b, pred, met)


@pytest.mark.gpu
def test_evaluate_vs_golden_and_side_effects(mods):
    """The reference fixture's predictions and BN running statistics after one evaluate; no parameter or .grad touched,
    the BN buffers those forward leaves from the same start, no bucket on a two-rank step."""
    eng = mods["engine"]
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["tiny"])
    z, sd_m, sd_c = load_golden_step("tiny")
    model, net = eng.build_models(d.map_size, device="cpu")
    model.load_state_dict(sd_m)
    net.load_state_dict(sd_c)
    model, net = model.to(DEV).train(), net.to(DEV).train()
    step = eng.DesignStep(model, net, world_size=2)
    before = _state(model, net)
    assert all(g is None for g, _ in before["grads"].values())
    b = eng.DesignBatch.from_synth(d, DEV)
    pred, met = step.evaluate(b)
    torch.cuda.synchronize()
    assert step._buckets == {}
    _assert_params_and_grads_unchanged(model, net, before)
    assert_close(pred, z["pred"], 1e-3, 1e-4, "pred vs reference fixture")
    n_stats = 0
    for k in z.files:
        if k.startswith("after.cnn.") and "running" in k:
            assert_close(net.state_dict()[k[len("after.cnn."):]], z[k], 1e-4, 1e-5, k)
            n_stats += 1
    assert n_stats > 0
    after_eval = {k: v.clone() for k, v in net.named_buffers()}
    for k, v in net.named_buffers():                       # back to the start, then forward
        v.copy_(before["bufs"]["c." + k])
    step.forward(eng.DesignBatch.from_synth(d, DEV))
    torch.cuda.synchronize()
    for k, v in net.named_buffers():
        assert torch.equal(v, after_eval[k]), f"buffer {k}: evaluate and forward leave different statistics"
    # a model with gradients: evaluate leaves every .grad object and its bits alone
    step1 = eng.DesignStep(model, net)
    step1.run(eng.DesignBatch.from_synth(d, DEV))
    torch.cuda.synchronize()
    before = _state(model, net)
    assert any(g is not None for g, _ in before["grads"].values())
    step1.evaluate(eng.DesignBatch.from_synth(d, DEV))
    torch.cuda.synchronize()
    _assert_params_and_grads_unchanged(model, net, before)
    assert step1._buckets == {}


# ------------------------------------------------------------------------------------------------------------------
# 3. per design / per level, capture, prepare, loader, errors
# ------------------------------------------------------------------------------------------------------------------
def _assert_close_rows(got, ref, rtol, what):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    np.testing.assert_array_equal(got[..., 2:8], ref[..., 2:8], err_msg=f"{what}: counts")
    for c in (0, 1, 8):
        np.testing.assert_array_equal(np.isnan(got[..., c]), np.isnan(ref[..., c]), err_msg=what)
        ok = ~np.isnan(ref[..., c])
        np.testing.assert_allclose(got[..., c][ok], ref[..., c][ok], rtol=rtol, atol=0, err_msg=what)


@pytest.mark.gpu
def test_joined_batch_rows_equal_designs_alone(mods):
    """metrics.design[k] / metrics.level[k] of three joined designs equal each design evaluated alone (rtol 1e-5: the
    joined predictions are the single ones' at 1e-5); levels a design lacks are empty rows."""
    eng = mods["engine"]
    ds = [_design("unet", 21, 4000, 900), _design("unet", 22, 2500, 400), _design("unet", 23, 3300, 700)]
    model, net = _models(eng, "unet", None)
    step = eng.DesignStep(model, net)
    b = _batch(eng, ds, labels=True)
    pred, met = step.evaluate(b)
    joined = _check_metrics_vs_numpy(b, pred, met)
    for k, d in enumerate(ds):
        bk = eng.DesignBatch.from_synth(d, DEV)
        bk.required = b.required[int(b.ep_off_h[k]):int(b.ep_off_h[k + 1])].clone()
        bk.label = b.label[int(b.ep_off_h[k]):int(b.ep_off_h[k + 1])].clone()
        _, mk = step.evaluate(bk)
        alone = mk.to_host()
        assert alone.K == 1 and alone.L <= joined.L
        _assert_close_rows(joined.design[k], alone.batch, 1e-5, f"design {k}")
        _assert_close_rows(joined.level[k, :alone.L], alone.level[0], 1e-5, f"levels of design {k}")
        assert bool((joined.level[k, alone.L:, 7] == 0).all())


@pytest.mark.gpu
def test_capture_prepare_and_prepare_many_evaluate(mods):
    """Replays equal eager evaluate bit for bit (predictions and the metric table), twice in a row and after the inputs
    were refreshed in place; prepare / prepare_many(evaluate=True) fed new host values equal eager evaluate on them."""
    eng = mods["engine"]
    ds = [_design("unet", 31 + k, 2500, 600) for k in range(3)]
    model, net = _models(eng, "unet", None)
    step = eng.DesignStep(model, net)
    b = _batch(eng, ds[:1], labels=True)
    replay = step.capture_evaluate(b)
    b_eager = _batch(eng, ds[:1], labels=True)
    for _ in range(2):
        pred, met = replay()
        got = (pred.clone(), _bits(met.table))
        pe, me = step.evaluate(b_eager)
        torch.cuda.synchronize()
        assert torch.equal(got[0], pe) and torch.equal(got[1], _bits(me.table))
    for x in (b, b_eager):
        x.cell_feat.mul_(0.5)
        x.image.copy_(x.image.flip(-1))
        x.arrival_time.add_(0.125)
    pred, met = replay()
    got = (pred.clone(), _bits(met.table))
    pe, me = step.evaluate(b_eager)
    torch.cuda.synchronize()
    assert torch.equal(got[0], pe) and torch.equal(got[1], _bits(me.table))
    # prepare: one design, new values from pinned host memory
    prep = step.prepare(eng.HostDesign(ds[0], pin=True), DEV, evaluate=True)
    d2 = _design("unet", 31, 2500, 600)
    d2.cell_feat = (d2.cell_feat * 0.5).astype(np.float32)
    d2.image = np.ascontiguousarray(d2.image[:, ::-1, :]).astype(np.float32)
    d2.arrival_time = (d2.arrival_time + 0.25).astype(np.float32)
    host2 = eng.HostDesign(d2, pin=True)
    pred, met = prep.step(host2)
    got = (pred.clone(), _bits(met.table))
    pe, me = step.evaluate(eng.DesignBatch.from_host(host2, DEV))
    torch.cuda.synchronize()
    assert torch.equal(got[0], pe) and torch.equal(got[1], _bits(me.table))
    # prepare_many: three designs, new values for all of them
    many = step.prepare_many([eng.HostDesign(x, pin=True) for x in ds], DEV, evaluate=True)
    for x in ds:
        x.image = np.ascontiguousarray(x.image[:, :, ::-1]).astype(np.float32)
        x.net_feat = (x.net_feat + 0.5).astype(np.float32)
    hosts2 = [eng.HostDesign(x, pin=True) for x in ds]
    pred, met = many.step(hosts2)
    got = (pred.clone(), _bits(met.table))
    assert met.design.shape == (3, 9)
    b4 = eng.DesignBatch.concat([eng.DesignBatch.from_host(h, DEV) for h in hosts2])
    pe, me = step.evaluate(b4)
    torch.cuda.synchronize()
    assert torch.equal(got[0], pe) and torch.equal(got[1], _bits(me.table))
    step.close()


def _tiny(seed):
    return tm_synth.make_design(seed=seed, n_cells=300 + 40 * seed, n_lv=6, map_size=8, n_endpoints=60)


def _check_loader_rows(ld, paths, pred, met_level):
    """Per-level rows against numpy from the loader's own tables (path_level, path_endpoint, labels)."""
    ids = paths.long()
    ep = ld.path_endpoint[ids].long()
    lv = ld.path_level[ids].numpy().astype(np.int64)
    cpu = lambda t: t.detach().cpu()[ep].numpy()                # noqa: E731
    ref = _level_rows(_host(pred), cpu(ld.arrival), cpu(ld.required), cpu(ld.label), lv, met_level.shape[0])
    _assert_rows(met_level, ref, 1e-6, "levels")


@pytest.mark.gpu
def test_loader_prepare_evaluate(mods):
    """prepare_evaluate (training usage: every path once, the oversampled duplicates dropped; test usage: the validation
    split) and prepare_evaluate_many against eager evaluate on ld.batch(run.paths), and their per-level rows against
    numpy over path_level."""
    eng, ldr = mods["engine"], mods["loader"]
    model, net = _models(eng, "unet", None, seed=4, map_size=8)
    step = eng.DesignStep(model, net)
    lds = [ldr.load_design(ldr.design_tuple_from_synth(_tiny(s), seed=s), DEV) for s in (4, 5, 6)]
    ld = lds[0]
    run = ld.prepare_evaluate(step)
    assert sorted(run.paths.tolist()) == sorted(set(ld.paths)) and len(ld.paths) > len(run.paths)
    pred, met = run()
    pe, _ = step.evaluate(ld.batch(run.paths))
    torch.cuda.synchronize()
    assert torch.equal(pred, pe)
    h = met.to_host()
    _check_loader_rows(ld, run.paths, pred, h.level[0])
    assert int(h.batch[7]) == len(run.paths) and float(h.batch[2]) > 0      # labels attached: confusion counts
    # usage "test": the validation split
    ldt = ldr.load_design(ldr.design_tuple_from_synth(_tiny(7), seed=7), DEV, usage="test")
    runt = ldt.prepare_evaluate(step)
    assert sorted(runt.paths.tolist()) == sorted(ldt.paths) and len(runt.paths) < int((ldt.path_level >= 0).sum())
    pred, met = runt()
    pe, _ = step.evaluate(ldt.batch(runt.paths))
    torch.cuda.synchronize()
    assert torch.equal(pred, pe)
    _check_loader_rows(ldt, runt.paths, pred, met.to_host().level[0])
    # several designs in one graph, the middle one on an explicit path list
    explicit = list(range(0, 60, 3))
    runm = ldr.prepare_evaluate_many(lds, step, paths=[None, explicit, None])
    assert sorted(runm.paths[1].tolist()) == explicit
    pred, met = runm()
    pe, _ = step.evaluate(eng.DesignBatch.concat([x.batch(p) for x, p in zip(lds, runm.paths)]))
    torch.cuda.synchronize()
    assert torch.equal(pred, pe)
    h = met.to_host()
    for k, x in enumerate(lds):
        s, e = int(runm.batch.ep_off_h[k]), int(runm.batch.ep_off_h[k + 1])
        _check_loader_rows(x, runm.paths[k], pred[s:e], h.level[k])
    step.close()


def test_evaluate_option_errors(mods):
    """Invalid combinations are refused before any device work (no device needed)."""
    eng = mods["engine"]
    model, net = eng.build_models(32, device="cpu")
    step = eng.DesignStep(model, net)
    for kw in (dict(input_grads=True), dict(param_grads=False), dict(input_grads=True, param_grads=False)):
        with pytest.raises(ValueError, match="evaluate"):
            step.prepare(None, "cpu", evaluate=True, **kw)
        with pytest.raises(ValueError, match="evaluate"):
            step.prepare_many([None], "cpu", evaluate=True, **kw)
    with pytest.raises(ValueError, match="dynamic"):
        step.capture_evaluate(types.SimpleNamespace(dynamic=True))
