"""What-if evaluation: the joined forward cones of K candidate edits (``tm_forward_cones`` / ``tm_graph.ForwardCones``)
and ``IncrementalEvaluation.what_if`` / ``WhatIf``.

1. ``tm_forward_cones`` against a numpy search per candidate on tm_synth designs (tiny, c1, c2) and on a 1.7M-pin
   netlist whose bitmaps live in the workspace: membership, sizes, virtual rows by rank, each candidate's levels and
   remapped in-edge lists inside the joined schedule, the S copies.
2. ``run()`` bitwise per row against ``forward`` on the batch edited with that candidate alone (U-Net and LayoutNet,
   K = 1, 7, 33; late and uniform seeds, overlapping cones, shared pins, an empty set, unscheduled pins), the committed
   state and the model untouched.
3. A joined batch; 4. capture; 5. commit; 6. admission with too few rows; 7. the errors.
"""
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
# helpers (the reference search and the edits as in test_gpu_incremental.py)
# ------------------------------------------------------------------------------------------------------------------
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
    return per * n_lv, (cat(net_s), cat(net_d)), (cat(cell_s), cat(cell_d)), ids[0]


def _edit(cf, nf, rows, rng):
    """Cell-type one-hot swaps on rows carrying a cell type, new uniforms on rows carrying net features, in place."""
    for p in rows:
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


def _candidate_sets(b, K, rng, lo=0, hi=None):
    """K pin sets over pins [lo, hi): late single pins, late groups, uniform draws, overlapping and shared pins, an
    empty set and unscheduled pins."""
    sched = b.graph.schedule()
    lv = sched.level.cpu().numpy()
    hi = lv.size if hi is None else hi
    ids = np.arange(lo, hi)
    sch = ids[lv[lo:hi] >= 0]
    L = sched.num_levels
    late = sch[lv[sch] >= L - max(2, L // 4)]
    outside = ids[lv[lo:hi] < 0]
    shared = int(rng.choice(sch))
    kinds = ["late1", "late8", "uniform1", "shared", "empty", "outside", "uniform4", "overlap"]
    sets = []
    for k in range(K):
        kind = kinds[k % len(kinds)] if K > 1 else "uniform1"
        if kind == "late1":
            s = [int(rng.choice(late))]
        elif kind == "late8":
            s = [int(x) for x in rng.choice(late, 8, replace=False)]
        elif kind == "uniform1":
            s = [int(rng.choice(sch))]
        elif kind == "shared":
            s = [shared, int(rng.choice(late))]
        elif kind == "empty":
            s = []
        elif kind == "outside":
            s = [int(x) for x in outside[:3]] if outside.size else [shared]
        elif kind == "uniform4":
            s = [int(x) for x in rng.choice(sch, 4, replace=False)] + [shared]
        else:                                      # the previous set's pins plus one: overlapping cones, duplicates
            s = list(sets[-1]) + [int(rng.choice(sch))] + list(sets[-1][:1])
        sets.append(s)
    return sets


def _edit_candidates(wi, rng):
    for k in range(wi.K):
        pins, cf, nf = wi.rows(k)
        _edit(cf, nf, range(len(pins)), rng)


def _forward_with(step, b, wi, k):
    """step.forward(b) with candidate k's rows written into the batch, then the batch restored."""
    pins, cf, nf = wi.rows(k)
    cf0, nf0 = b.cell_feat.clone(), b.net_feat.clone()
    if len(pins):
        idx = torch.from_numpy(pins).to(DEV)
        b.cell_feat[idx] = cf
        b.net_feat[idx] = nf
    out = step.forward(b)
    b.cell_feat.copy_(cf0)
    b.net_feat.copy_(nf0)
    return out


def _base(inc, b):
    return dict(H=inc.H.clone(), S=inc.S.clone(), pred=inc.pred.clone(), cf=b.cell_feat.clone(), nf=b.net_feat.clone())


def _assert_base(inc, b, before, what):
    for k, t in (("H", inc.H), ("S", inc.S), ("pred", inc.pred), ("cf", b.cell_feat), ("nf", b.net_feat)):
        _bits_equal(t, before[k], f"{what}: committed {k}")


# ------------------------------------------------------------------------------------------------------------------
# 1. tm_forward_cones against numpy
# ------------------------------------------------------------------------------------------------------------------
def _check_cones(mods, tg, h, edges, sets, R, what):
    sched = tg.schedule()
    n = sched.n
    K = len(sets)
    ptr = np.concatenate([[0], np.cumsum([len(s) for s in sets])]).astype(np.int32)
    seeds = np.concatenate([np.asarray(s, np.int64) for s in sets]).astype(np.int32)
    ep = sched.order[-5:].contiguous()
    max_deg = int(np.max(h["f_ptr"][1:] - h["f_ptr"][:-1]))
    fc = mods["graph"].ForwardCones(tg, K, R, R * max_deg, ep, seeds.size)
    S = torch.randn(n + R + 1, 128, device=DEV)
    S0 = S[:n].clone()
    fc.build(torch.from_numpy(ptr).to(DEV), torch.from_numpy(seeds).to(DEV), None, S)
    _bits_equal(S[:n], S0, f"{what}: S rows of the pins")
    cnt = int(fc.count.item())
    order, lptr = fc.order[:cnt].cpu().numpy(), fc.level_ptr.cpu().numpy()
    fptr, vpin = fc.f_ptr[:cnt + 1].cpu().numpy(), fc.vpin[:cnt].cpu().numpy()
    fsrc = fc.f_src[:int(fptr[-1])].cpu().numpy()
    fitted, sizes, base = fc.fitted.cpu().numpy(), fc.sizes.cpu().numpy(), fc.row_base.cpu().numpy()
    head = fc.head_rows[:K * 5].cpu().numpy().reshape(K, 5)
    srows = fc.seed_rows[:seeds.size].cpu().numpy()
    assert lptr[0] == 0 and lptr[-1] == cnt and np.all(np.diff(lptr) >= 0)
    run = 0
    for k, s in enumerate(sets):
        c_order, c_lptr, c_fptr, c_fsrc = _ref_cone(h, edges, s)
        assert sizes[k] == len(c_order), f"{what}/{k}: size {sizes[k]} != {len(c_order)}"
        assert bool(fitted[k]) == (run + len(c_order) <= R and all(fitted[:k])), f"{what}/{k}: admission"
        if not fitted[k]:
            assert np.all(srows[ptr[k]:ptr[k + 1]] == n + R), f"{what}/{k}: seeds of a non-admitted candidate"
            continue
        assert base[k] == run
        lo, hi = n + run, n + run + len(c_order)
        np.testing.assert_array_equal(vpin[run:run + len(c_order)], np.sort(c_order), err_msg=f"{what}/{k}: rank")
        mine = (order >= lo) & (order < hi)
        np.testing.assert_array_equal(vpin[order[mine] - n], c_order, err_msg=f"{what}/{k}: order")
        cum = np.concatenate([[0], np.cumsum(mine)])
        np.testing.assert_array_equal(cum[lptr], c_lptr, err_msg=f"{what}/{k}: levels")
        pos = np.nonzero(mine)[0]
        got = np.concatenate([fsrc[fptr[p]:fptr[p + 1]] for p in pos]) if pos.size else np.zeros(0, np.int64)
        inside = got >= n
        assert np.all(got[inside] >= lo) and np.all(got[inside] < hi), f"{what}/{k}: a source in another candidate"
        mapped = np.where(inside, vpin[np.where(inside, got - n, 0)], got)
        np.testing.assert_array_equal(mapped, c_fsrc, err_msg=f"{what}/{k}: in-edges")
        mark = np.zeros(n, bool)
        mark[c_order] = True
        assert np.all(mark[got[~inside]] == False), f"{what}/{k}: a source in the cone kept its pin id"  # noqa: E712
        for i in range(ptr[k], ptr[k + 1]):
            u = int(seeds[i])
            want = n + run + int(np.searchsorted(np.sort(c_order), u)) if h["level"][u] >= 0 else n + R
            assert srows[i] == want, f"{what}/{k}: seed row of {u}"
        epn = ep.cpu().numpy()
        want = [n + run + int(np.searchsorted(np.sort(c_order), u)) if mark[u] else u for u in epn]
        np.testing.assert_array_equal(head[k], want, err_msg=f"{what}/{k}: head rows")
        _bits_equal(S[lo:hi], S0[vpin[run:run + len(c_order)]], f"{what}/{k}: S copies")
        run += len(c_order)
    assert cnt == run


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["tiny", "c1", "c2"])
def test_forward_cones_match_numpy_search(mods, cfg):
    d = tm_synth.make_design(seed=5, **tm_synth.CONFIGS[cfg])
    tg = mods["graph"].TimingGraph(d.n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis).to(DEV)
    h = _host(tg.schedule())
    edges = {"net": (d.net_src, d.net_dst), "cell": (d.cell_src, d.cell_dst)}
    rng = np.random.default_rng(1)
    lv, order, lp, L = h["level"], h["order"], h["level_ptr"], h["L"]
    late = order[lp[L - 2]:lp[L]]
    outside = np.nonzero(lv < 0)[0]
    sets = [[int(rng.choice(late))], [], [int(x) for x in rng.choice(d.n, 8)], [int(late[0]), int(late[0])],
            [int(outside[0])] if outside.size else [int(late[-1])], [int(order[lp[1]])], [int(late[0]), int(late[1])]]
    n_sched = int(lp[L])
    _check_cones(mods, tg, h, edges, sets, 4 * n_sched, f"{cfg}/all fit")
    sizes = [len(_ref_cone(h, edges, s)[0]) for s in sets]
    R = max(sizes[0] + sizes[1] + sizes[2], 1)     # the third fits exactly, the fourth may not
    _check_cones(mods, tg, h, edges, sets, R, f"{cfg}/R={R}")


@pytest.mark.gpu
def test_forward_cones_bitmaps_in_global_memory(mods):
    """1.7M pins: the candidates' bitmaps (212 KB each) live in the workspace instead of shared memory."""
    rng = np.random.default_rng(7)
    n, net, cell, pis = _layered_netlist(1_700_000, 21, rng)
    tg = mods["graph"].TimingGraph(n, net, cell, pis=pis).to(DEV)
    h = _host(tg.schedule())
    lp, order, L = h["level_ptr"], h["order"], h["L"]
    sets = [[int(order[lp[L - 3]]), int(order[lp[L - 2] + 5])], [int(order[lp[L - 2] + 7])],
            [int(x) for x in rng.choice(n, 4)], []]
    _check_cones(mods, tg, h, {"net": net, "cell": cell}, sets, 2 * n, "big")


# ------------------------------------------------------------------------------------------------------------------
# 2. predictions
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cnn,K", [("unet", 1), ("unet", 7), ("unet", 33), ("layoutnet", 7)])
def test_what_if_matches_forward_bitwise(mods, cnn, K):
    eng = mods["engine"]
    model, net = _models(eng, cnn)
    b = eng.DesignBatch.from_synth(_design(cnn, 21), DEV)
    step = eng.DesignStep(model, net)
    rng = np.random.default_rng(K)
    before = _state(model, net)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 4)
    base = _base(inc, b)
    wi = inc.what_if(_candidate_sets(b, K, rng))
    _edit_candidates(wi, rng)
    pred = wi.run()
    assert pred.shape == (K, int(b.endpoints.numel()))
    assert wi.fitted().all()
    _assert_base(inc, b, base, "after run")
    _assert_state(model, net, before)
    sizes = wi.cone_sizes()
    for k in range(K):
        pins = wi.rows(k)[0]
        if len(pins) == 0 or (inc._level[pins] < 0).all():
            assert sizes[k] == 0
            _bits_equal(pred[k], base["pred"], f"candidate {k}: nothing scheduled edited")
        else:
            assert sizes[k] > 0
        _bits_equal(pred[k], _forward_with(step, b, wi, k), f"{cnn} K={K}: candidate {k} vs forward")
    _assert_base(inc, b, base, "after the references")


# ------------------------------------------------------------------------------------------------------------------
# 3. joined batch
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_joined_batch(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(_design("unet", 30 + k, n_cells=1500, T=100), DEV)
                                for k in range(2)])
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes())
    rng = np.random.default_rng(4)
    p1 = int(b.pin_off_h[1])
    sets = _candidate_sets(b, 4, rng, 0, p1) + _candidate_sets(b, 4, rng, p1)
    wi = inc.what_if(sets)
    _edit_candidates(wi, rng)
    pred = wi.run()
    e1 = int(b.ep_off_h[1])
    for k in range(len(sets)):
        _bits_equal(pred[k], _forward_with(step, b, wi, k), f"joined batch: candidate {k}")
        other = slice(e1, None) if k < 4 else slice(0, e1)
        _bits_equal(pred[k][other], inc.pred[other], f"joined batch: candidate {k} leaves the other design alone")


# ------------------------------------------------------------------------------------------------------------------
# 4. capture
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_capture(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 41), DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 2)
    rng = np.random.default_rng(9)
    wi = inc.what_if(_candidate_sets(b, 9, rng))
    replay = wi.capture()
    for rnd in range(3):
        _edit_candidates(wi, rng)
        base = _base(inc, b)
        before = _state(model, net)                    # (forward below updates the U-Net's running statistics)
        got = replay().clone()
        _assert_base(inc, b, base, f"replay {rnd}")
        _assert_state(model, net, before)
        _bits_equal(got, wi.run(), f"replay vs eager run, round {rnd}")
        for k in (0, 3, 8):
            _bits_equal(got[k], _forward_with(step, b, wi, k), f"replay round {rnd}: candidate {k} vs forward")
        # the base moves: the next replay predicts against it
        pins = rng.choice(np.nonzero(inc._level >= 0)[0], 3, replace=False)
        _edit(b.cell_feat, b.net_feat, pins, rng)
        inc.update(pins)
    got = replay()
    for k in range(wi.K):
        _bits_equal(got[k], _forward_with(step, b, wi, k), f"replay after updates: candidate {k} vs forward")
    step.close()


# ------------------------------------------------------------------------------------------------------------------
# 5. commit
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_commit(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    d = _design("unet", 43)
    b = eng.DesignBatch.from_synth(d, DEV)
    b2 = eng.DesignBatch.from_synth(d, DEV)                # the same design, stepped with update
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 2)
    ref = step.incremental(b2)
    rng = np.random.default_rng(12)
    for rnd in range(3):
        wi = inc.what_if(_candidate_sets(b, 8, rng))
        _edit_candidates(wi, rng)
        wi.run()
        k = [0, 6, 2][rnd]
        pins, cf, nf = wi.rows(k)
        wi.commit(k)
        idx = torch.from_numpy(pins).to(DEV)
        b2.cell_feat[idx] = cf
        b2.net_feat[idx] = nf
        ref.update(pins)
        assert inc.cone_size() == ref.cone_size()
        _bits_equal(b.cell_feat, b2.cell_feat, f"commit {rnd}: cell_feat")
        _bits_equal(b.net_feat, b2.net_feat, f"commit {rnd}: net_feat")
        _bits_equal(inc.pred, ref.pred, f"commit {rnd}: pred vs update")
        _bits_equal(inc.H, ref.H, f"commit {rnd}: H vs update")
        _bits_equal(inc.S, ref.S, f"commit {rnd}: S vs update")
        _bits_equal(inc.pred, step.forward(b), f"commit {rnd}: pred vs forward")
        with pytest.raises(ValueError, match="base changed"):
            wi.commit(k)                                   # the commit itself moved the base
    wi = inc.what_if([[int(np.nonzero(inc._level >= 0)[0][-1])]])
    wi.run()
    inc.update([int(np.nonzero(inc._level >= 0)[0][0])])
    with pytest.raises(ValueError, match="base changed"):
        wi.commit(0)
    wi.run()
    wi2 = inc.what_if([[]])
    wi2.run()
    with pytest.raises(ValueError, match="another what-if"):
        wi.commit(0)
    inc.refresh()
    with pytest.raises(ValueError):
        wi2.commit(0)


# ------------------------------------------------------------------------------------------------------------------
# 6. admission
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_admission(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 45), DEV)
    step = eng.DesignStep(model, net)
    rng = np.random.default_rng(13)
    sets = _candidate_sets(b, 10, rng)
    probe = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 3).what_if(sets)
    probe.run()
    sizes = probe.cone_sizes()
    cut = 4
    R = int(sizes[:cut].sum()) + int(sizes[cut]) // 2 if sizes[cut] > 1 else int(sizes[:cut].sum())
    R = max(R, 1)
    inc = step.incremental(b, what_if_rows=R)
    n, G = inc.n, 7
    # guard rows after the (n + R + 1)-row buffers
    for name in ("H_ext", "S_ext"):
        big = torch.full((n + R + 1 + G, 128), 3.25, device=DEV)
        big[:n + R + 1] = getattr(inc, name)
        setattr(inc, name, big[:n + R + 1])
        setattr(inc, "_big_" + name, big)
    inc.H, inc.S = inc.H_ext[:n], inc.S_ext[:n]
    wi = inc.what_if(sets)
    _edit_candidates(wi, rng)
    base = _base(inc, b)
    pred = wi.run()
    fit = wi.fitted()
    np.testing.assert_array_equal(wi.cone_sizes(), probe.cone_sizes())
    run, open_ = 0, True
    for k in range(len(sets)):
        open_ = open_ and run + int(sizes[k]) <= R
        assert fit[k] == open_, f"candidate {k}: fitted {fit[k]}, expected {open_}"
        run += int(sizes[k]) if open_ else 0
        if fit[k]:
            _bits_equal(pred[k], _forward_with(step, b, wi, k), f"admitted candidate {k}")
        else:
            assert torch.isnan(pred[k]).all(), f"candidate {k} not admitted but not NaN"
            with pytest.raises(ValueError, match="not admitted"):
                wi.commit(k)
    assert not fit.all() and fit[0]
    _assert_base(inc, b, base, "with too few rows")
    for name in ("H_ext", "S_ext"):
        assert bool((getattr(inc, "_big_" + name)[n + R + 1:] == 3.25).all()), f"{name}: guard rows written"


# ------------------------------------------------------------------------------------------------------------------
# 7. errors
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_errors(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 50, n_cells=800, T=60), DEV)
    step = eng.DesignStep(model, net)
    with pytest.raises(ValueError, match="what_if_rows=0"):
        step.incremental(b).what_if([[1]])
    for bad in (-1, 1.5, True):
        with pytest.raises(ValueError):
            step.incremental(b, what_if_rows=bad)
    inc = step.incremental(b, what_if_rows=1000)
    n = b.graph.number_of_nodes()
    for bad in ([[n]], [[0], [-1]], [[0.5]], [["a"]], [torch.tensor([1], device=DEV)], [], torch.tensor([[1]])):
        with pytest.raises(ValueError):
            inc.what_if(bad)
    wi = inc.what_if([[1], [2, 2]])
    with pytest.raises(ValueError):
        wi.commit(0)                                       # never ran
    wi.run()
    for bad in (2, -1, 0.0):
        with pytest.raises(ValueError):
            wi.commit(bad)
    with pytest.raises(ValueError):
        wi.rows(2)
    torch.cuda.synchronize()
