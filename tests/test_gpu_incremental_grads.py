"""Incremental input gradients: the fan-in cone of seeded endpoints (``tm_fanin_cone``), the recomputed saved
activations (``tm_gnn_save_cone``), the backward sweep over the cone (``tm_gnn_backward_cone``), the self-MLP data
gradients with device row counts and ``IncrementalEvaluation.input_grads`` / ``capture_input_grads``.

1. ``tm_fanin_cone`` against a numpy fan-in search over the backward's edges, laid out as the header documents it:
   tiny / c1 / c2 designs, duplicate endpoints, an all-zero seed, a 1.7M-pin netlist (bitmap in the workspace).
2. Bitwise against the persistent full backward (``tm_gnn_set_impl(3)``, the head's data gradient scattered into G,
   ``gnn_backward(..., need_dx=True, need_wgrad=False)``): G on the cone, the reference's G zero off the cone, the
   recomputed A / LSE / HID rows, the feature gradients.  U-Net and LayoutNet, one design and a joined batch of three,
   seeds on 1, 7 and all endpoints.
3. After updates, captured updates and ``WhatIf.commit``: the bitwise reference on the edited features, and the frozen
   step to fp32 class (other back ends).
4. Captured replays; 5. the state left untouched; 6. the errors.
"""
import ctypes

import numpy as np
import pytest
import torch

import tm_synth

DEV = "cuda"
NUM_CTYPES = 34


@pytest.fixture(scope="module")
def mods(pkg):
    import tm_engine, tm_graph, tm_lib, tm_ops  # noqa: E401
    yield dict(engine=tm_engine, graph=tm_graph, lib=tm_lib, ops=tm_ops)
    if torch.cuda.is_available():
        tm_lib.check_err_flags()


# ------------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------------
def _np(t):
    return t.cpu().numpy().astype(np.int64)


def _host(sched):
    ns = sched.n_sched
    return dict(level=_np(sched.level), order=_np(sched.order), level_ptr=sched.h_level_ptr.astype(np.int64),
                cell_base=sched.h_cell_base.astype(np.int64), crow=_np(sched.crow), L=sched.num_levels, ns=ns,
                ncr=sched.n_cell_rows, f_ptr=_np(sched.f_ptr), f_src=_np(sched.f_src), bn_ptr=_np(sched.bn_ptr),
                bn_dst=_np(sched.bn_dst), bn_w=sched.bn_w.cpu().numpy(), bc_ptr=_np(sched.bc_ptr),
                bc_row=_np(sched.bc_row))


def _ref_fanin(h, endpoints, seed):
    """Fan-in search from the scheduled endpoints with a non-zero seed over the backward's edges (bn_dst, and bc_row's
    pins), then the sub-schedule laid out from the end of the buffers as tm_fanin_cone documents it."""
    lv, order, ns, ncr = h["level"], h["order"], h["ns"], h["ncr"]
    n = lv.size
    row_pin = np.full(max(ncr, 1), -1, np.int64)
    has = h["crow"] >= 0
    row_pin[h["crow"][has]] = np.nonzero(has)[0]
    mark = np.zeros(n, bool)
    ep = np.asarray(endpoints, np.int64)[np.asarray(seed) != 0]
    ep = ep[(ep >= 0) & (ep < n)]
    mark[ep[lv[ep] >= 0]] = True
    pos_n = np.repeat(np.arange(ns), np.diff(h["bn_ptr"][:ns + 1]))
    pos_c = np.repeat(np.arange(ns), np.diff(h["bc_ptr"][:ns + 1]))
    src = np.concatenate([order[pos_n], order[pos_c]])
    dst = np.concatenate([h["bn_dst"][:pos_n.size], row_pin[h["bc_row"][:pos_c.size]]])
    while True:
        new = src[mark[dst] & ~mark[src]]
        if new.size == 0:
            break
        mark[new] = True
    inpos = mark[order]
    C = int(inpos.sum())
    base = ns - C
    cum = np.concatenate([[0], np.cumsum(inpos)])
    lp = base + cum[h["level_ptr"]]
    cpos = np.nonzero(inpos)[0]
    is_cellrow = (lv[order] > 0) & (lv[order] % 2 == 0)
    c_cell = inpos & is_cellrow
    Cc = int(c_cell.sum())
    ccum = np.concatenate([[0], np.cumsum(c_cell)])
    cb = ncr - Cc + ccum[h["level_ptr"]]
    cone_row = np.full(max(ncr, 1), -1, np.int64)
    cone_row[h["crow"][order[c_cell]]] = ncr - Cc + np.arange(Cc)

    def lay(ptr, keep, vals):
        """kept edges of the cone's positions, right-aligned at the parent's edge count; -> (ptr over [base, ns],
        values)"""
        E = ptr[ns]
        pos = np.repeat(np.arange(ns), np.diff(ptr[:ns + 1]))
        sel = inpos[pos] & keep(np.arange(E))
        deg = np.bincount(pos[sel], minlength=ns)[cpos]
        cptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64) + E - int(deg.sum())
        return cptr, vals(np.arange(E))[sel]

    f = lay(h["f_ptr"], lambda e: np.ones(e.size, bool), lambda e: h["f_src"][e])
    bn = lay(h["bn_ptr"], lambda e: mark[h["bn_dst"][e]], lambda e: h["bn_dst"][e])
    bnw = lay(h["bn_ptr"], lambda e: mark[h["bn_dst"][e]], lambda e: h["bn_w"][e])[1]
    bc = lay(h["bc_ptr"], lambda e: mark[row_pin[h["bc_row"][e]]], lambda e: cone_row[h["bc_row"][e]])
    pins = order[inpos]
    even = lv[pins] % 2 == 0
    return dict(mark=mark, base=base, count=C, order=pins, level_ptr=lp, cell_base=cb, f=f, bn=bn, bn_w=bnw, bc=bc,
                cell_pins=pins[even][::-1], net_pins=pins[~even][::-1], n_cell_rows_cone=Cc, cone_row=cone_row)


def _check_fanin(fc, h, endpoints, seed, what):
    ep = torch.as_tensor(np.asarray(endpoints), dtype=torch.int32).to(DEV)
    sd = torch.as_tensor(np.asarray(seed), dtype=torch.float32).to(DEV)
    ref = _ref_fanin(h, endpoints, seed)
    for k in range(2):                                     # a second build into the same buffers
        fc.build(ep, sd)
        torch.cuda.synchronize()
        cnt = _np(fc.counts)
        ns, base = h["ns"], ref["base"]
        assert cnt[0] == ref["count"], f"{what}: count {cnt[0]} != {ref['count']}"
        assert cnt[1] == len(ref["cell_pins"]) and cnt[2] == len(ref["net_pins"]), f"{what}: class counts {cnt}"
        np.testing.assert_array_equal(_np(fc.order)[base:ns], ref["order"], err_msg=f"{what}: order")
        np.testing.assert_array_equal(_np(fc.level_ptr), ref["level_ptr"], err_msg=f"{what}: level_ptr")
        np.testing.assert_array_equal(_np(fc.cell_base), ref["cell_base"], err_msg=f"{what}: cell_base")
        for name, ptr, vals, (rp, rv) in (("f", fc.f_ptr, fc.f_src, ref["f"]), ("bn", fc.bn_ptr, fc.bn_dst, ref["bn"]),
                                          ("bc", fc.bc_ptr, fc.bc_row, ref["bc"])):
            got_p = _np(ptr)[base:ns + 1]
            np.testing.assert_array_equal(got_p, rp, err_msg=f"{what}: {name}_ptr")
            np.testing.assert_array_equal(_np(vals)[rp[0]:rp[-1]], rv, err_msg=f"{what}: {name} edges")
        rp = ref["bn"][0]
        np.testing.assert_array_equal(fc.bn_w.cpu().numpy()[rp[0]:rp[-1]], ref["bn_w"], err_msg=f"{what}: bn_w")
        np.testing.assert_array_equal(_np(fc.cell_pins)[:cnt[1]], ref["cell_pins"], err_msg=f"{what}: cell_pins")
        np.testing.assert_array_equal(_np(fc.net_pins)[:cnt[2]], ref["net_pins"], err_msg=f"{what}: net_pins")
    return ref


def _layered_netlist(n_target, n_lv, rng):
    """A big layered netlist (level 0 PIs, odd levels net sinks, even levels cell outputs) with edges that skip levels."""
    per = n_target // n_lv
    ids = rng.permutation(per * n_lv).reshape(n_lv, per)
    net_s, net_d, cell_s, cell_d = [], [], [], []
    for l in range(1, n_lv):
        if l % 2:
            src_lv = 2 * rng.integers(0, (l + 1) // 2, size=per)
            net_s.append(ids[src_lv, rng.integers(0, per, size=per)])
            net_d.append(ids[l])
        else:
            for _ in range(2):
                src_lv = 2 * rng.integers(0, l // 2, size=per) + 1
                cell_s.append(ids[src_lv, rng.integers(0, per, size=per)])
                cell_d.append(ids[l])
    cat = lambda a: np.concatenate(a).astype(np.int64)               # noqa: E731
    return per * n_lv, (cat(net_s), cat(net_d)), (cat(cell_s), cat(cell_d)), ids[0], ids[-1]


def _gnn_params(model):
    import tm_ops
    sd = dict(model.gnn.named_parameters())
    return [sd[k].detach() for k in tm_ops.GNN_PARAM_NAMES]


def _edit_rows(b, pins, rng):
    cf, nf = b.cell_feat, b.net_feat
    for p in pins:
        row = cf[p]
        oh = row[:NUM_CTYPES]
        if float(oh.sum()) == 1.0:
            k = int(torch.argmax(oh))
            j = (k + 1 + int(rng.integers(0, NUM_CTYPES - 1))) % NUM_CTYPES
            oh.zero_()
            oh[j] = 1.0
            row[NUM_CTYPES:] = torch.tensor(rng.random(2), dtype=torch.float32, device=DEV)
        if float(nf[p].abs().sum()) > 0:
            nf[p] = torch.tensor(rng.random(2), dtype=torch.float32, device=DEV)


def _bits_equal(a, b, what):
    a, b = a.detach().contiguous(), b.detach().contiguous()
    assert a.shape == b.shape, what
    ne = int((a.view(torch.int32) != b.view(torch.int32)).sum())
    assert ne == 0, f"{what}: {ne} of {a.numel()} elements differ in their bits"


def _same_values(a, b, what):
    """Bitwise up to the sign of zeros (the cone drops edges that carry an exact zero)."""
    a, b = a.detach(), b.detach()
    assert a.shape == b.shape, what
    ne = int(((a != b) & ~(torch.isnan(a) & torch.isnan(b))).sum())
    assert ne == 0, f"{what}: {ne} of {a.numel()} elements differ"
    _bits_equal(torch.where(a == 0, torch.zeros_like(a), a), torch.where(b == 0, torch.zeros_like(b), b), what)


def _close(got, ref, what, rtol=1e-3, atol=2e-4):
    scale = max(float(ref.abs().max()), 1e-30)
    err = (got - ref).abs()
    bad = int((err > rtol * ref.abs() + atol * scale).sum())
    assert bad == 0, f"{what}: {bad} elements outside rtol {rtol} / atol {atol} x max|ref| (max err {float(err.max())})"


def _design(cnn, seed, n_cells=3000, T=200):
    kw = dict(img_channels=2, img_scale=4) if cnn == "layoutnet" else {}
    return tm_synth.make_design(seed=seed, n_cells=n_cells, n_lv=20, map_size=32, n_endpoints=T, **kw)


def _models(eng, cnn, seed=0):
    model, net = eng.build_models(32, seed=seed, device=DEV, cnn=cnn)
    if cnn == "layoutnet":
        net.math = "bf16"
    return model, net


def _state(model, net):
    named = [("m." + k, p) for k, p in model.named_parameters()] + [("c." + k, p) for k, p in net.named_parameters()]
    bufs = [("m." + k, v) for k, v in model.named_buffers()] + [("c." + k, v) for k, v in net.named_buffers()]
    return dict(params={k: p.detach().clone() for k, p in named},
                grads={k: (p.grad, None if p.grad is None else p.grad.clone()) for k, p in named},
                bufs={k: v.clone() for k, v in bufs})


def _assert_state(model, net, before):
    after = _state(model, net)
    for k, v in before["params"].items():
        _bits_equal(after["params"][k], v, f"parameter {k}")
    for k, (obj, val) in before["grads"].items():
        g_obj, _ = after["grads"][k]
        assert g_obj is obj, f".grad of {k} was replaced"
        if val is not None:
            _bits_equal(g_obj, val, f".grad of {k}")
    for k, v in before["bufs"].items():
        assert torch.equal(after["bufs"][k], v), f"buffer {k} changed"


def _seeds(T, rng):
    s1 = torch.zeros(T, dtype=torch.float32, device=DEV)
    s1[int(rng.integers(0, T))] = 1.0
    s7 = torch.zeros(T, dtype=torch.float32, device=DEV)
    s7[torch.as_tensor(rng.choice(T, 7, replace=False), device=DEV)] = torch.tensor(rng.standard_normal(7),
                                                                                     dtype=torch.float32, device=DEV)
    sa = torch.tensor(rng.standard_normal(T), dtype=torch.float32, device=DEV)
    return {"one": s1, "seven": s7, "all": sa}


def _reference(mods, step, inc, b, seed):
    """The persistent full forward + head data gradient + persistent full backward on b's current features:
    (G before the sweep, G after, dcell, dnet, saved, H)."""
    ops, lib = mods["ops"], mods["lib"]
    sched = b.graph.schedule()
    gp = _gnn_params(step.model)
    T, width = int(b.endpoints.numel()), inc.X.shape[1]
    old = lib.lib().tm_gnn_set_impl(3)
    try:
        H, saved = ops.gnn_forward(sched, b.cell_feat, b.net_feat, gp, save=True)
        f0, f2 = step.model.mlp_fuse.layers[0], step.model.mlp_fuse.layers[2]
        X = inc.X.clone()                                  # image-side columns: the frozen image branch's
        lib.call("tm_gather_cols", T, 128, H, 128, b.endpoints, X, width, 0, lib.stream())
        pred = torch.empty(T, 1, dtype=torch.float32, device=DEV)
        hf = ops.mlp2_forward(X, width, None, T, f0.weight.detach(), f0.bias.detach(), f2.weight.detach(),
                              f2.bias.detach(), pred, 1)
        dX = ops.mlp2_backward(X, width, None, T, f0.weight.detach(), f2.weight.detach(), hf,
                               seed.reshape(T, 1), 1, need_dx=True, need_wgrad=False)[4]
        G = torch.zeros(sched.n, 128, dtype=torch.float32, device=DEV)
        lib.call("tm_scatter_add_cols", T, 128, dX, width, 0, b.endpoints, G, 128, lib.stream())
        G0 = G.clone()
        _, dcf, dnf = ops.gnn_backward(sched, saved, gp, G, need_dx=True, need_wgrad=False)
    finally:
        lib.lib().tm_gnn_set_impl(old)
    return dict(G0=G0, G=G, dcf=dcf, dnf=dnf, saved=saved, H=H, X=X, hf=hf, pred=pred.squeeze(1))


def _check_against_reference(mods, step, inc, b, seed, what, check_saved=True):
    ops, lib = mods["ops"], mods["lib"]
    ref = _reference(mods, step, inc, b, seed)
    _bits_equal(inc.H, ref["H"], f"{what}: inc.H vs the persistent forward")
    _bits_equal(inc.X, ref["X"], f"{what}: inc.X vs the head's matrix on H")
    _bits_equal(inc._hf, ref["hf"], f"{what}: the head's hidden rows")
    _bits_equal(inc.pred, ref["pred"], f"{what}: inc.pred")
    g = inc.input_grads(seed)
    gs = inc._grad
    fc, sched = gs["cone"], b.graph.schedule()
    torch.cuda.synchronize()
    h = _host(sched)
    cr = _ref_fanin(h, _np(b.endpoints), seed.cpu().numpy())
    assert inc.grad_cone_size() == cr["count"], what
    cone_pins = torch.as_tensor(cr["order"], device=DEV)
    off = torch.as_tensor(h["order"][~cr["mark"][h["order"]]], device=DEV)
    _same_values(gs["G"][cone_pins], ref["G"][cone_pins], f"{what}: G on the cone")
    assert int((ref["G"][off] != 0).sum()) == 0, f"{what}: the reference's G is not zero off the cone"
    _bits_equal(g["cell_feat"], ref["dcf"], f"{what}: cell_feat gradient")
    _bits_equal(g["net_feat"], ref["dnf"], f"{what}: net_feat gradient")
    if check_saved and cr["n_cell_rows_cone"]:
        sc = ops.gnn_cone_scratch(sched, DEV)
        gp = [ops._f32c(p) for p in _gnn_params(step.model)]
        nb = lib.ws_bytes("tm_gnn_ws_bytes")
        lib.call("tm_gnn_save_cone", fc.struct, inc.H, ops.transpose(gp[8]), gp[9], ops.transpose(gp[10]), sc["A"],
                 sc["LSE"], sc["HID"], lib.workspace(nb, DEV), nb, lib.stream())
        cpins = cr["order"][(h["level"][cr["order"]] > 0) & (h["level"][cr["order"]] % 2 == 0)]
        prow = torch.as_tensor(h["crow"][cpins], device=DEV)
        crow = torch.as_tensor(cr["cone_row"][h["crow"][cpins]], device=DEV)
        for k in ("A", "LSE", "HID"):
            _bits_equal(sc[k][crow], ref["saved"][k][prow], f"{what}: recomputed {k}")
    return ref, g


# ------------------------------------------------------------------------------------------------------------------
# 1. tm_fanin_cone against numpy
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["tiny", "c1", "c2"])
def test_fanin_cone_matches_numpy_search(mods, cfg):
    d = tm_synth.make_design(seed=5, **tm_synth.CONFIGS[cfg])
    tg = mods["graph"].TimingGraph(d.n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis).to(DEV)
    h = _host(tg.schedule())
    fc = mods["graph"].FaninCone(tg)
    rng = np.random.default_rng(3)
    lv, order, lp, L = h["level"], h["order"], h["level_ptr"], h["L"]
    last = order[lp[L - 1]:lp[L]]
    ep = np.concatenate([rng.choice(last, 40), rng.choice(order, 40), [int(last[0])] * 3])
    if (lv < 0).any():
        ep = np.concatenate([ep, [int(np.nonzero(lv < 0)[0][0])]])
    T = ep.size
    cases = {"one": np.eye(1, T, 0)[0], "seven": np.isin(np.arange(T), rng.choice(T, 7, replace=False)) * 0.5,
             "all": rng.standard_normal(T), "zero": np.zeros(T),
             "duplicates": np.isin(np.arange(T), [T - 4, T - 3, T - 2]).astype(np.float64)}
    for name, seed in cases.items():
        ref = _check_fanin(fc, h, ep, seed, f"{cfg}/{name}")
        if name == "zero":
            assert ref["count"] == 0 and fc.size() == 0


@pytest.mark.gpu
def test_fanin_cone_bitmap_in_global_memory(mods):
    """1.7M pins: the membership bitmap (212 KB) lives in the workspace instead of shared memory."""
    rng = np.random.default_rng(7)
    n, net, cell, pis, last = _layered_netlist(1_700_000, 21, rng)
    tg = mods["graph"].TimingGraph(n, net, cell, pis=pis).to(DEV)
    h = _host(tg.schedule())
    fc = mods["graph"].FaninCone(tg)
    mid = h["order"][h["level_ptr"][10]:h["level_ptr"][11]]
    ep = np.concatenate([last[:50], mid[:50]])
    for name, seed in {"late2": np.isin(np.arange(100), [3, 40]) * 1.0, "mid1": np.eye(1, 100, 70)[0],
                       "all": np.ones(100)}.items():
        _check_fanin(fc, h, ep, seed, f"big/{name}")


# ------------------------------------------------------------------------------------------------------------------
# 2. bitwise against the persistent full backward
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_input_grads_bitwise(mods, cnn):
    eng = mods["engine"]
    model, net = _models(eng, cnn)
    b = eng.DesignBatch.from_synth(_design(cnn, 11), DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b)
    rng = np.random.default_rng(1)
    for name, seed in _seeds(int(b.endpoints.numel()), rng).items():
        _check_against_reference(mods, step, inc, b, seed, f"{cnn}/{name}")
    step.close()


@pytest.mark.gpu
def test_input_grads_joined_batch(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(_design("unet", 30 + k, n_cells=1500, T=100), DEV)
                                for k in range(3)])
    step = eng.DesignStep(model, net)
    inc = step.incremental(b)
    rng = np.random.default_rng(2)
    for name, seed in _seeds(int(b.endpoints.numel()), rng).items():
        _check_against_reference(mods, step, inc, b, seed, f"joined/{name}")
    # seeds in design 1 only: the other designs' rows are exactly zero
    seed = torch.zeros(int(b.endpoints.numel()), dtype=torch.float32, device=DEV)
    e0, e1 = int(b.ep_off_h[1]), int(b.ep_off_h[2])
    seed[e0:e1] = 1.0
    _, g = _check_against_reference(mods, step, inc, b, seed, "joined/design 1")
    p0, p1 = int(b.pin_off_h[1]), int(b.pin_off_h[2])
    for k in ("cell_feat", "net_feat"):
        assert int((g[k][:p0] != 0).sum()) == 0 and int((g[k][p1:] != 0).sum()) == 0, k
    step.close()


# ------------------------------------------------------------------------------------------------------------------
# 3. after edits: updates, captured updates, what-if commits
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_input_grads_after_edits(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 21), DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=4000)
    rng = np.random.default_rng(5)
    lv = b.graph.schedule().level.cpu().numpy()
    sched_pins = np.nonzero(lv >= 0)[0]
    T = int(b.endpoints.numel())
    seed = torch.tensor(rng.standard_normal(T), dtype=torch.float32, device=DEV)
    inc.input_grads(seed)
    pins = rng.choice(sched_pins, 6, replace=False)
    _edit_rows(b, pins, rng)
    inc.update(pins)
    cap_pins = rng.choice(sched_pins, 3, replace=False)
    replay = inc.capture_update(cap_pins)
    for _ in range(2):
        _edit_rows(b, cap_pins, rng)
        replay()
    _check_against_reference(mods, step, inc, b, seed, "after updates")
    wi = inc.what_if([list(rng.choice(sched_pins, 2, replace=False)) for _ in range(4)])
    for k in range(wi.K):
        _, cf, nf = wi.rows(k)
        cf[:, :NUM_CTYPES] = torch.roll(cf[:, :NUM_CTYPES], 1, dims=1)
    wi.run()
    wi.commit(2)
    ref, g = _check_against_reference(mods, step, inc, b, seed, "after a what-if commit")
    # the frozen step on the edited batch: other back ends, fp32 class
    b.input_grads = None
    step.run(b, input_grads=True, pred_grad=seed, param_grads=False)
    torch.cuda.synchronize()
    for k in ("cell_feat", "net_feat"):
        _close(g[k], b.input_grads[k], f"{k} vs the frozen step")
    step.close()


# ------------------------------------------------------------------------------------------------------------------
# 4. captured replays; 5. untouched state
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_capture_input_grads_and_state(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 41), DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=2000)
    T = int(b.endpoints.numel())
    rng = np.random.default_rng(6)
    seed = torch.zeros(T, dtype=torch.float32, device=DEV)
    seed[3] = 1.0
    replay = inc.capture_input_grads(seed)
    lv = b.graph.schedule().level.cpu().numpy()
    pins = rng.choice(np.nonzero(lv >= 0)[0], 4, replace=False)
    upd = inc.capture_update(pins)
    seeds = list(_seeds(T, rng).values()) + [torch.zeros(T, dtype=torch.float32, device=DEV)]
    for rnd, s in enumerate(seeds):
        if rnd == 2:                                       # feature edits and captured updates between replays
            _edit_rows(b, pins, rng)
            upd()
        seed.copy_(s)
        got = {k: v.clone() for k, v in replay().items()}
        size = inc.grad_cone_size()
        if rnd == len(seeds) - 1:
            assert size == 0
            for k in got:
                assert int((got[k] != 0).sum()) == 0, f"zero seed: {k}"
        eager = inc.input_grads(s.clone())
        assert inc.grad_cone_size() == size
        for k in got:
            _bits_equal(got[k], eager[k], f"replay {rnd}: {k}")

    # the call leaves the committed state, the batch and the model alone
    wi = inc.what_if([[int(pins[0])], [int(pins[1])]])
    wi.run()
    before = _state(model, net)
    keep = dict(H=inc.H.clone(), S=inc.S.clone(), pred=inc.pred.clone(), X=inc.X.clone(), cf=b.cell_feat.clone(),
                nf=b.net_feat.clone(), Hx=inc.H_ext.clone(), Sx=inc.S_ext.clone(), wp=wi.pred.clone())
    gen = inc.generation
    inc.input_grads(seeds[2])
    replay()
    torch.cuda.synchronize()
    _assert_state(model, net, before)
    for k, v in dict(H=inc.H, S=inc.S, pred=inc.pred, X=inc.X, cf=b.cell_feat, nf=b.net_feat, Hx=inc.H_ext,
                     Sx=inc.S_ext, wp=wi.pred).items():
        _bits_equal(v, keep[k], f"{k} after input_grads")
    assert inc.generation == gen
    wi.commit(1)                                           # the what-if is still valid
    step.close()


# ------------------------------------------------------------------------------------------------------------------
# 6. errors
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_input_grads_errors(mods):
    eng, lib, ops = mods["engine"], mods["lib"], mods["ops"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 50, n_cells=800, T=60), DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b)
    T = int(b.endpoints.numel())
    good = torch.ones(T, dtype=torch.float32, device=DEV)
    for bad in (torch.ones(T + 1, device=DEV), torch.ones(T, dtype=torch.float64, device=DEV), torch.ones(T),
                torch.ones(2 * T, device=DEV)[::2], torch.ones(T, 1, device=DEV), good.tolist()):
        with pytest.raises(ValueError, match="seed"):
            inc.input_grads(bad)
        with pytest.raises(ValueError, match="seed"):
            inc.capture_input_grads(bad)
    assert inc.grad_cone_size() == 0
    inc.input_grads(good)
    fc = inc._grad["cone"]
    with pytest.raises(ValueError):
        fc.build(b.endpoints.long(), good)
    sched = b.graph.schedule()
    with pytest.raises(RuntimeError, match="tm_fanin_cone.*workspace too small"):
        lib.call("tm_fanin_cone", sched.struct, T, b.endpoints, good, fc.order, fc.level_ptr, fc.cell_base, fc.f_ptr,
                 fc.f_src, fc.bn_ptr, fc.bn_dst, fc.bn_w, fc.bc_ptr, fc.bc_row, fc.cell_pins, fc.net_pins, fc.counts,
                 fc.ws, fc.nb - 1, lib.stream())
    with pytest.raises(RuntimeError, match="tm_fanin_cone.*NULL output"):
        lib.call("tm_fanin_cone", sched.struct, T, b.endpoints, good, fc.order, fc.level_ptr, None, fc.f_ptr,
                 fc.f_src, fc.bn_ptr, fc.bn_dst, fc.bn_w, fc.bc_ptr, fc.bc_row, fc.cell_pins, fc.net_pins, fc.counts,
                 fc.ws, fc.nb, lib.stream())
    with pytest.raises(RuntimeError, match="tm_fanin_cone.*endpoint"):
        lib.call("tm_fanin_cone", sched.struct, T, b.endpoints, None, fc.order, fc.level_ptr, fc.cell_base, fc.f_ptr,
                 fc.f_src, fc.bn_ptr, fc.bn_dst, fc.bn_w, fc.bc_ptr, fc.bc_row, fc.cell_pins, fc.net_pins, fc.counts,
                 fc.ws, fc.nb, lib.stream())
    bare = lib.tm_schedule()
    ctypes.memmove(ctypes.addressof(bare), ctypes.addressof(fc.struct), ctypes.sizeof(bare))
    bare.bc_row = None
    with pytest.raises(RuntimeError, match="tm_fanin_cone.*device arrays"):
        lib.call("tm_fanin_cone", bare, T, b.endpoints, good, fc.order, fc.level_ptr, fc.cell_base, fc.f_ptr,
                 fc.f_src, fc.bn_ptr, fc.bn_dst, fc.bn_w, fc.bc_ptr, fc.bc_row, fc.cell_pins, fc.net_pins, fc.counts,
                 fc.ws, fc.nb, lib.stream())
    gp = [ops._f32c(p) for p in _gnn_params(model)]
    w1t, w2t = ops.transpose(gp[8]), ops.transpose(gp[10])
    nb = lib.ws_bytes("tm_gnn_ws_bytes")
    ws = lib.workspace(nb, DEV)
    sc, G = inc._grad["scratch"], inc._grad["G"]
    with pytest.raises(RuntimeError, match="tm_gnn_save_cone.*NULL operand"):
        lib.call("tm_gnn_save_cone", fc.struct, inc.H, w1t, gp[9], w2t, None, sc["LSE"], sc["HID"], ws, nb, lib.stream())
    with pytest.raises(RuntimeError, match="tm_gnn_save_cone.*workspace too small"):
        lib.call("tm_gnn_save_cone", fc.struct, inc.H, w1t, gp[9], w2t, sc["A"], sc["LSE"], sc["HID"], ws, nb - 1,
                 lib.stream())
    with pytest.raises(RuntimeError, match="tm_gnn_backward_cone.*device arrays"):
        lib.call("tm_gnn_backward_cone", bare, inc.H, G, gp[8], gp[10], sc["A"], sc["LSE"], sc["HID"], sc["GA"], ws, nb,
                 lib.stream())
    with pytest.raises(RuntimeError, match="tm_gnn_backward_cone.*NULL operand"):
        lib.call("tm_gnn_backward_cone", fc.struct, inc.H, G, gp[8], gp[10], sc["A"], sc["LSE"], sc["HID"], None, ws,
                 nb, lib.stream())
    # the fan-in cone has no host level offsets: the full backward refuses it
    with pytest.raises(RuntimeError, match="tm_gnn_backward"):
        lib.call("tm_gnn_backward", fc.struct, inc.H, G, gp[8], gp[10], sc["A"], sc["LSE"], sc["HID"], sc["GA"], None,
                 None, ws, nb, lib.stream())
    dcf = torch.zeros_like(b.cell_feat)
    nb1 = lib.ws_bytes("tm_selfmlp_lin1_ws_bytes")
    with pytest.raises(RuntimeError, match="tm_selfmlp_lin1_relu_dcount.*NULL"):
        lib.call("tm_selfmlp_lin1_relu_dcount", fc.n_cell_cap, None, b.cell_feat, b.cell_feat.stride(0), fc.cell_pins,
                 b.cell_feat.shape[1], gp[0], gp[1], sc["HID"], 256, lib.workspace(nb1, DEV), nb1, lib.stream())
    nb2 = lib.ws_bytes("tm_selfmlp_rows_dh_ws_bytes")
    with pytest.raises(RuntimeError, match="tm_selfmlp_rows_dx_dcount.*workspace too small"):
        lib.call("tm_selfmlp_rows_dx_dcount", fc.n_cell_cap, fc.counts[1:], G, 128, fc.cell_pins, gp[2], sc["HID"], 256,
                 None, gp[0], b.cell_feat.shape[1], dcf, dcf.stride(0), fc.cell_pins, lib.workspace(nb2, DEV), nb2 - 1,
                 lib.stream())
    nb3 = lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")
    with pytest.raises(RuntimeError, match="tm_selfmlp_gen_bwd1_dx_dcount.*NULL"):
        lib.call("tm_selfmlp_gen_bwd1_dx_dcount", fc.n_net_cap, fc.counts[2:], G, 128, fc.net_pins, b.net_feat,
                 b.net_feat.stride(0), fc.net_pins, 2, gp[4], gp[5], gp[6], None, 2, lib.workspace(nb3, DEV), nb3,
                 lib.stream())
    torch.cuda.synchronize()
    step.close()
