"""Incremental evaluation: the forward cone of edited pins (``tm_forward_cone``), the propagation over it
(``tm_gnn_forward_cone``) and ``DesignStep.incremental`` / ``IncrementalEvaluation``.

1. ``tm_forward_cone`` against a numpy breadth-first search on tm_synth designs (shuffled ids, edges that skip levels)
   and on a 1.7M-pin netlist whose membership bitmap does not fit in shared memory: order, level_ptr, f_ptr, f_src
   and the count exactly, the same bits on a second call.
2. ``tm_gnn_forward_cone`` after the seeds' self terms changed: every H row the same bits as a full persistent forward
   over the edited features (cone levels tile cell pins at other widths than full levels).
3. ``IncrementalEvaluation`` with the U-Net and LayoutNet: pred / H bitwise against ``forward`` / ``gnn_forward`` after
   edits, after twenty successive updates, after edit-and-revert; the model left exactly as found.
4. A joined batch of three designs; 5. captured updates; 6. the errors.
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
def _graph(mods, d):
    tg = mods["graph"].TimingGraph(d.n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis).to(DEV)
    return tg, tg.schedule()


def _host(sched):
    return dict(level=sched.level.cpu().numpy(), order=sched.order.cpu().numpy(), level_ptr=sched.h_level_ptr.copy(),
                f_ptr=sched.f_ptr.cpu().numpy(), f_src=sched.f_src.cpu().numpy(), L=sched.num_levels)


def _ref_cone(h, edges, seeds):
    """Push search from the scheduled seeds over the edges the propagation reads (net edges into odd levels, cell edges
    into even levels > 0), then the sub-schedule laid out as tm_forward_cone documents it."""
    lv = h["level"]
    n = lv.size
    mark = np.zeros(n, bool)
    s = np.asarray(seeds, np.int64)
    s = s[(s >= 0) & (s < n)]
    mark[s[lv[s] >= 0]] = True
    src = np.concatenate([edges["net"][0], edges["cell"][0]]).astype(np.int64)
    dst = np.concatenate([edges["net"][1], edges["cell"][1]]).astype(np.int64)
    is_net = np.concatenate([np.ones(len(edges["net"][0]), bool), np.zeros(len(edges["cell"][0]), bool)])
    ld = lv[dst]
    ok = np.where(is_net, ld % 2 == 1, (ld > 0) & (ld % 2 == 0)) & (ld >= 0) & (lv[src] >= 0)
    src, dst = src[ok], dst[ok]
    while True:
        new = dst[mark[src] & ~mark[dst]]
        if new.size == 0:
            break
        mark[new] = True
    order, fp, fs = h["order"], h["f_ptr"], h["f_src"]
    inpos = mark[order]
    c_order = order[inpos]
    deg = (fp[1:len(order) + 1] - fp[:len(order)])[inpos]
    c_fptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    ns = len(order)
    pos_of_edge = np.repeat(np.arange(ns), fp[1:ns + 1] - fp[:ns])
    c_fsrc = fs[:fp[ns]][inpos[pos_of_edge]]
    cum = np.concatenate([[0], np.cumsum(inpos)])
    c_lptr = cum[h["level_ptr"]]
    return c_order, c_lptr, c_fptr, c_fsrc


def _check_cone(fc, h, edges, seeds, what):
    ref = _ref_cone(h, edges, seeds)
    for k in range(2):
        fc.build(torch.tensor(np.asarray(seeds, np.int64), dtype=torch.int32).to(DEV))
        cnt = fc.size()
        got = (fc.order[:cnt].cpu().numpy(), fc.level_ptr.cpu().numpy(), fc.f_ptr[:cnt + 1].cpu().numpy(),
               fc.f_src[:int(ref[2][-1])].cpu().numpy())
        assert cnt == len(ref[0]), f"{what}: count {cnt} != {len(ref[0])}"
        for name, g, r in zip(("order", "level_ptr", "f_ptr", "f_src"), got, ref):
            np.testing.assert_array_equal(g, np.asarray(r, np.int64), err_msg=f"{what} (call {k}): {name}")


def _seed_sets(h, rng):
    lv, order, lp, L = h["level"], h["order"], h["level_ptr"], h["L"]
    n = lv.size
    pis = order[lp[0]:lp[1]]
    mid = L // 2 if (L // 2) % 2 == 0 else L // 2 + 1              # an even level > 0: cell outputs
    cell_mid = order[lp[mid]:lp[mid + 1]]
    sinks = order[lp[1]:lp[2]]
    last = order[lp[L - 1]:lp[L]]
    outside = np.nonzero(lv < 0)[0]
    sets = {"pi": [int(pis[0])], "mid_cell": [int(rng.choice(cell_mid))], "net_sink": [int(rng.choice(sinks))],
            "last_level": [int(rng.choice(last))], "empty": [], "every_pin": list(range(n))}
    if outside.size:
        sets["outside"] = [int(outside[0])]
    sets["outside_and_dup"] = [int(outside[0]) if outside.size else int(last[0]), int(cell_mid[0]), int(cell_mid[0]),
                               int(sinks[-1]), int(sinks[-1])]
    sets["random64"] = [int(x) for x in rng.choice(n, 64)]
    return sets


def _layered_netlist(n_target, n_lv, rng):
    """A big layered netlist (level 0 PIs, odd levels net sinks, even levels cell outputs) with edges that skip levels."""
    per = n_target // n_lv
    ids = rng.permutation(per * n_lv).reshape(n_lv, per)
    net_s, net_d, cell_s, cell_d = [], [], [], []
    for l in range(1, n_lv):
        if l % 2:                                                     # every sink: one driver on an earlier even level
            src_lv = 2 * rng.integers(0, (l + 1) // 2, size=per)
            net_s.append(ids[src_lv, rng.integers(0, per, size=per)])
            net_d.append(ids[l])
        else:                                                         # every output: two inputs on earlier odd levels
            for _ in range(2):
                src_lv = 2 * rng.integers(0, l // 2, size=per) + 1
                cell_s.append(ids[src_lv, rng.integers(0, per, size=per)])
                cell_d.append(ids[l])
    cat = lambda a: np.concatenate(a).astype(np.int64)               # noqa: E731
    return per * n_lv, (cat(net_s), cat(net_d)), (cat(cell_s), cat(cell_d)), ids[0]


def _gnn_params(model):
    import tm_ops
    sd = dict(model.gnn.named_parameters())
    return [sd[k].detach() for k in tm_ops.GNN_PARAM_NAMES]


def _edit_rows(b, pins, rng):
    """Cell-type one-hot swaps on cell-output rows, new uniforms on net sinks, in place."""
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


def _scheduled(b):
    lv = b.graph.schedule().level.cpu().numpy()
    return np.nonzero(lv >= 0)[0]


def _bits_equal(a, b, what):
    a, b = a.detach().contiguous(), b.detach().contiguous()
    assert a.shape == b.shape, what
    ne = int((a.view(torch.int32) != b.view(torch.int32)).sum())
    assert ne == 0, f"{what}: {ne} of {a.numel()} elements differ in their bits"


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


def _reference(mods, step, b):
    """(pred, H) of a full forward on the persistent back end."""
    H, _ = mods["ops"].gnn_forward(b.graph.schedule(), b.cell_feat, b.net_feat, _gnn_params(step.model), save=False,
                                   impl=1)
    return step.forward(b), H


# ------------------------------------------------------------------------------------------------------------------
# 1. tm_forward_cone against numpy
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["tiny", "c1"])
def test_forward_cone_matches_numpy_search(mods, cfg):
    d = tm_synth.make_design(seed=5, **tm_synth.CONFIGS[cfg])
    tg, sched = _graph(mods, d)
    h = _host(sched)
    edges = {"net": (d.net_src, d.net_dst), "cell": (d.cell_src, d.cell_dst)}
    fc = mods["graph"].ForwardCone(tg)
    for name, seeds in _seed_sets(h, np.random.default_rng(1)).items():
        _check_cone(fc, h, edges, seeds, f"{cfg}/{name}")


@pytest.mark.gpu
def test_forward_cone_bitmap_in_global_memory(mods):
    """1.7M pins: the membership bitmap (212 KB) lives in the workspace instead of shared memory."""
    rng = np.random.default_rng(7)
    n, net, cell, pis = _layered_netlist(1_700_000, 21, rng)
    tg = mods["graph"].TimingGraph(n, net, cell, pis=pis).to(DEV)
    sched = tg.schedule()
    h = _host(sched)
    edges = {"net": net, "cell": cell}
    fc = mods["graph"].ForwardCone(tg)
    lp, order, L = h["level_ptr"], h["order"], h["L"]
    assert L >= 6
    for name, seeds in {"late": [int(order[lp[L - 3]]), int(order[lp[L - 2] + 5])],
                        "early": [int(order[lp[2] + 3])],
                        "random16": [int(x) for x in rng.choice(n, 16)]}.items():
        _check_cone(fc, h, edges, seeds, f"big/{name}")


# ------------------------------------------------------------------------------------------------------------------
# 2. tm_gnn_forward_cone against a full persistent forward
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cfg,n_seeds", [("tiny", 3), ("tiny", 40), ("c1", 1), ("c1", 50), ("c1", 600), ("c2", 64)])
def test_gnn_forward_cone_bitwise(mods, cfg, n_seeds):
    ops, eng = mods["ops"], mods["engine"]
    d = tm_synth.make_design(seed=11, **tm_synth.CONFIGS[cfg])
    model, _ = eng.build_models(d.map_size, seed=2, device=DEV)
    b = eng.DesignBatch.from_synth(d, DEV)
    sched = b.graph.schedule()
    gp = _gnn_params(model)
    S = torch.empty(sched.n, 128, dtype=torch.float32, device=DEV)
    ops.gnn_self_terms(S, b.cell_feat, b.net_feat, gp, sched.cell_class, sched.net_class)
    H = torch.zeros(sched.n, 128, dtype=torch.float32, device=DEV)
    ops.gnn_forward_cone(sched, H, S, gp)
    _bits_equal(H, ops.gnn_forward(sched, b.cell_feat, b.net_feat, gp, save=False, impl=1)[0], f"{cfg}: full pass")
    rng = np.random.default_rng(n_seeds)
    pins = np.unique(rng.choice(_scheduled(b), n_seeds, replace=False))
    _edit_rows(b, pins, rng)
    lv = sched.level.cpu().numpy()[pins]
    cell, net = pins[lv % 2 == 0], pins[lv % 2 == 1]
    ci = torch.tensor(cell, dtype=torch.int32, device=DEV)
    ni = torch.tensor(net, dtype=torch.int32, device=DEV)
    ops.gnn_self_terms(S, b.cell_feat, b.net_feat, gp, ci, ni)
    fc = mods["graph"].ForwardCone(b.graph)
    fc.build(torch.cat([ci, ni]))
    ops.gnn_forward_cone(fc, H, S, gp)
    assert 0 < fc.size() <= sched.n_sched
    ref = ops.gnn_forward(sched, b.cell_feat, b.net_feat, gp, save=False, impl=1)[0]
    _bits_equal(H, ref, f"{cfg}: {n_seeds} edited pins, cone of {fc.size()}")


# ------------------------------------------------------------------------------------------------------------------
# 3. IncrementalEvaluation
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cnn", ["unet", "layoutnet"])
def test_incremental_matches_forward_bitwise(mods, cnn):
    eng = mods["engine"]
    model, net = _models(eng, cnn)
    b = eng.DesignBatch.from_synth(_design(cnn, 21), DEV)
    step = eng.DesignStep(model, net)
    sched_pins = _scheduled(b)
    rng = np.random.default_rng(3)
    orig_cf, orig_nf = b.cell_feat.clone(), b.net_feat.clone()

    before = _state(model, net)                      # nothing of the model changes through any of this
    inc = step.incremental(b)
    pred0, H0 = inc.pred.clone(), inc.H.clone()
    for k in (1, 16, 256):
        pins = rng.choice(sched_pins, k, replace=False)
        _edit_rows(b, pins, rng)
        inc.update(list(pins) + list(pins[:2]))      # duplicates are dropped
        assert 0 < inc.cone_size() <= b.graph.schedule().n_sched
    rec = [(inc.pred.clone(), inc.H.clone())]
    for _ in range(20):
        pins = rng.choice(sched_pins, int(rng.integers(1, 9)), replace=False)
        _edit_rows(b, pins, rng)
        inc.update(torch.from_numpy(pins))
    rec.append((inc.pred.clone(), inc.H.clone()))
    cf20, nf20 = b.cell_feat.clone(), b.net_feat.clone()
    edited = np.nonzero(((b.cell_feat != orig_cf).any(1) | (b.net_feat != orig_nf).any(1)).cpu().numpy())[0]
    b.cell_feat.copy_(orig_cf)
    b.net_feat.copy_(orig_nf)
    inc.update(edited)                               # revert every edit: the original bits
    _bits_equal(inc.pred, pred0, "pred after edit and revert")
    _bits_equal(inc.H, H0, "H after edit and revert")
    inc.update([])
    assert inc.cone_size() == 0
    inc.refresh()
    _bits_equal(inc.pred, pred0, "pred after refresh")
    _assert_state(model, net, before)

    p_ref, H_ref = _reference(mods, step, b)
    _bits_equal(pred0, p_ref, "pred of the baseline vs forward")
    _bits_equal(H0, H_ref, "H of the baseline vs gnn_forward")
    b.cell_feat.copy_(cf20)
    b.net_feat.copy_(nf20)
    p_ref, H_ref = _reference(mods, step, b)
    _bits_equal(rec[1][0], p_ref, "pred after 20 successive updates vs one forward")
    _bits_equal(rec[1][1], H_ref, "H after 20 successive updates vs gnn_forward")

    # each edit checked on its own, against forward
    inc2 = step.incremental(b)
    for k in (1, 16, 256):
        pins = rng.choice(sched_pins, k, replace=False)
        _edit_rows(b, pins, rng)
        inc2.update(pins)
        p_ref, H_ref = _reference(mods, step, b)
        _bits_equal(inc2.pred, p_ref, f"pred after editing {k} pins")
        _bits_equal(inc2.H, H_ref, f"H after editing {k} pins")


# ------------------------------------------------------------------------------------------------------------------
# 4. joined batch
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_incremental_joined_batch(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(_design("unet", 30 + k, n_cells=1500, T=100), DEV)
                                for k in range(3)])
    step = eng.DesignStep(model, net)
    inc = step.incremental(b)
    pred0 = inc.pred.clone()
    p0, p1 = int(b.pin_off_h[1]), int(b.pin_off_h[2])
    e0, e1 = int(b.ep_off_h[1]), int(b.ep_off_h[2])
    lv = b.graph.schedule().level.cpu().numpy()
    cand = np.arange(p0, p1)[lv[p0:p1] >= 0]
    rng = np.random.default_rng(4)
    pins = rng.choice(cand, 32, replace=False)
    _edit_rows(b, pins, rng)
    inc.update(pins)
    _bits_equal(inc.pred[:e0], pred0[:e0], "design 0's predictions")
    _bits_equal(inc.pred[e1:], pred0[e1:], "design 2's predictions")
    assert not torch.equal(inc.pred[e0:e1], pred0[e0:e1])
    p_ref, H_ref = _reference(mods, step, b)
    _bits_equal(inc.pred, p_ref, "joined batch vs forward")
    _bits_equal(inc.H, H_ref, "joined batch H vs gnn_forward")


# ------------------------------------------------------------------------------------------------------------------
# 5. capture
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_capture_update(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 41), DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b)
    sched_pins = _scheduled(b)
    rng = np.random.default_rng(9)
    pa = rng.choice(sched_pins, 8, replace=False)
    pb = rng.choice(np.setdiff1d(sched_pins, pa), 64, replace=False)
    ra, rb = inc.capture_update(pa), inc.capture_update(pb)
    for rnd in range(3):
        for pins, replay in ((pa, ra), (pb, rb)):
            _edit_rows(b, pins, rng)
            pred = replay()
            assert pred is inc.pred
            got, gotH = pred.clone(), inc.H.clone()
            inc.update(pins)
            _bits_equal(got, inc.pred, f"replay vs eager update, round {rnd}")
            _bits_equal(gotH, inc.H, f"replay H vs eager update, round {rnd}")
            _bits_equal(got, step.forward(b), f"replay vs forward, round {rnd}")
    step.close()


# ------------------------------------------------------------------------------------------------------------------
# 6. errors
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_incremental_errors(mods):
    eng, lib, ops = mods["engine"], mods["lib"], mods["ops"]
    model, net = _models(eng, "unet")
    d = _design("unet", 50, n_cells=800, T=60)
    b = eng.DesignBatch.from_synth(d, DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b)
    n = b.graph.number_of_nodes()
    for bad in ([n], [-1], [0.5, 1.0], np.array([1.0]), ["a"], torch.tensor([1], device=DEV)):
        with pytest.raises(ValueError):
            inc.update(bad)
    with pytest.raises(ValueError):
        inc.capture_update([n + 3])
    bd = eng.DesignBatch.from_synth(d, DEV)
    bd.dynamic = True
    with pytest.raises(ValueError, match="dynamic"):
        step.incremental(bd)
    with pytest.raises(ValueError):
        inc.cone.build(torch.tensor([1, 2], dtype=torch.int64, device=DEV))

    sched = b.graph.schedule()
    gp = [ops._f32c(p) for p in _gnn_params(model)]
    w1t, w2t = ops.transpose(gp[8]), ops.transpose(gp[10])
    nb = lib.ws_bytes("tm_gnn_ws_bytes")
    ws = lib.workspace(nb, DEV)
    fc = inc.cone
    fc.build(torch.tensor([int(sched.order[0])], dtype=torch.int32, device=DEV))
    with pytest.raises(RuntimeError, match="tm_gnn_forward_cone.*workspace too small"):
        lib.call("tm_gnn_forward_cone", fc.struct, inc.H, inc.S, w1t, gp[9], w2t, gp[11], ws, nb - 1, lib.stream())
    bare = lib.tm_schedule()
    ctypes.memmove(ctypes.addressof(bare), ctypes.addressof(fc.struct), ctypes.sizeof(bare))
    bare.level_ptr = None
    with pytest.raises(RuntimeError, match="tm_gnn_forward_cone.*device arrays"):
        lib.call("tm_gnn_forward_cone", bare, inc.H, inc.S, w1t, gp[9], w2t, gp[11], ws, nb, lib.stream())
    seeds = torch.zeros(1, dtype=torch.int32, device=DEV)
    with pytest.raises(RuntimeError, match="tm_forward_cone.*workspace too small"):
        lib.call("tm_forward_cone", sched.struct, 1, seeds, fc.order, fc.level_ptr, fc.f_ptr, fc.f_src, fc.count, fc.ws,
                 fc.nb - 1, lib.stream())
    with pytest.raises(RuntimeError, match="tm_forward_cone.*device arrays"):
        lib.call("tm_forward_cone", bare, 1, seeds, fc.order, fc.level_ptr, fc.f_ptr, fc.f_src, fc.count, fc.ws,
                 fc.nb, lib.stream())
    # the cone has no host level offsets: the level-range entry points refuse it
    with pytest.raises(RuntimeError, match="tm_gnn_forward"):
        lib.call("tm_gnn_forward", fc.struct, 0, sched.num_levels, inc.H, inc.S, w1t, gp[9], w2t, gp[11], None, None,
                 None, ws, nb, lib.stream())
    G = torch.zeros_like(inc.H)
    with pytest.raises(RuntimeError, match="tm_gnn_backward"):
        lib.call("tm_gnn_backward", fc.struct, inc.H, G, gp[8], gp[10], None, None, None, G, None, None, ws, nb,
                 lib.stream())
    torch.cuda.synchronize()
