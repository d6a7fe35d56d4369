"""What-if evaluation restricted to chosen endpoints: ``IncrementalEvaluation.what_if(pin_sets, endpoints=E)``, the fan-in
cone's bitmap (``tm_fanin_cone_bits`` / ``FaninCone(keep_bits=True)``) and the restricted joined cones
(``tm_forward_cones_within`` / ``ForwardCones(within=...)``).

1. R(E) against reverse reachability over the forward's in-edges (f_src) -- the closure the restriction relies on --
   and each candidate's restricted cone against numpy (its forward cone intersected with R(E)): tiny, c1, c2 and a
   1.7M-pin netlist; E shallow, deep and all endpoints.
2. ``run()`` bitwise per row against ``forward`` at E and against the unrestricted ``run()`` at E (U-Net and LayoutNet,
   K = 1, 7, 33; pins inside and outside R(E), unscheduled pins, empty sets, shared pins), the state untouched.
3. A joined batch with E in both designs; 4. admission; 5. ``commit`` against ``update``; 6. captured replays;
7. the errors.
"""
import numpy as np
import pytest
import torch

import tm_synth
from test_gpu_what_if import (_assert_base, _assert_state, _base, _bits_equal, _candidate_sets, _design, _edit,
                              _edit_candidates, _forward_with, _host, _layered_netlist, _models, _ref_cone, _state)

DEV = "cuda"


@pytest.fixture(scope="module")
def mods(pkg):
    import tm_engine, tm_graph, tm_lib, tm_ops  # noqa: E401
    yield dict(engine=tm_engine, graph=tm_graph, lib=tm_lib, ops=tm_ops)
    if torch.cuda.is_available():
        tm_lib.check_err_flags()


# ------------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------------
def _ref_within(h, pins):
    """R(E): the scheduled pins from which a scheduled pin of ``pins`` is reachable over the forward's in-edges (f_src),
    as a bool mask over the pins."""
    lv, order, fp, fs = h["level"], h["order"], h["f_ptr"], h["f_src"]
    ns = len(order)
    mark = np.zeros(lv.size, bool)
    p = np.asarray(pins, np.int64)
    mark[p[lv[p] >= 0]] = True
    dst = order[np.repeat(np.arange(ns), fp[1:ns + 1] - fp[:ns])].astype(np.int64)
    src = fs[:fp[ns]].astype(np.int64)
    keep = lv[src] >= 0                                    # an unscheduled source is in no forward cone
    src, dst = src[keep], dst[keep]
    while True:
        new = src[mark[dst] & ~mark[src]]
        if new.size == 0:
            break
        mark[new] = True
    return mark


def _unpack(bits, n):
    w = bits.cpu().numpy().view(np.uint32)
    return ((w[np.arange(n) >> 5] >> (np.arange(n) & 31).astype(np.uint32)) & 1).astype(bool)


def _ref_restricted(h, edges, seeds, rmask):
    """The restricted cone of ``seeds`` laid out as tm_forward_cones lays out a cone: (order, level_ptr counts, f_ptr,
    f_src) of fwdcone(seeds) intersected with R(E), in the parent's order."""
    c_order = _ref_cone(h, edges, seeds)[0]
    mark = np.zeros(h["level"].size, bool)
    mark[c_order] = True
    mark &= rmask
    order, fp, fs = h["order"], h["f_ptr"], h["f_src"]
    ns = len(order)
    inpos = mark[order]
    deg = (fp[1:ns + 1] - fp[:ns])[inpos]
    pos_of_edge = np.repeat(np.arange(ns), fp[1:ns + 1] - fp[:ns])
    cum = np.concatenate([[0], np.cumsum(inpos)])
    return order[inpos], cum[h["level_ptr"]], np.concatenate([[0], np.cumsum(deg)]), fs[:fp[ns]][inpos[pos_of_edge]]


def _check_restricted(mods, tg, h, edges, sets, E, R, what):
    """FaninCone(keep_bits) of E against numpy (membership and the f_src closure), then ForwardCones(within=...)."""
    g = mods["graph"]
    sched = tg.schedule()
    n = sched.n
    E = np.asarray(E, np.int64)
    ep = torch.from_numpy(E.astype(np.int32)).to(DEV)
    fan = g.FaninCone(tg, keep_bits=True)
    fan.build(ep, torch.ones(E.size, dtype=torch.float32, device=DEV))
    rmask = _ref_within(h, E)
    got = _unpack(fan.bits, n)
    np.testing.assert_array_equal(got, rmask, err_msg=f"{what}: R(E) bitmap vs reverse reachability over f_src")
    assert fan.size() == int(rmask.sum()), f"{what}: |R(E)|"
    K = len(sets)
    ptr = np.concatenate([[0], np.cumsum([len(s) for s in sets])]).astype(np.int32)
    seeds = np.concatenate([np.asarray(s, np.int64) for s in sets]).astype(np.int32)
    max_deg = int(np.max(h["f_ptr"][1:] - h["f_ptr"][:-1]))
    fc = g.ForwardCones(tg, K, R, R * max_deg, ep, seeds.size, within=fan)
    S = torch.randn(n + R + 1, 128, device=DEV)
    S0 = S[:n].clone()
    fc.build(torch.from_numpy(ptr).to(DEV), torch.from_numpy(seeds).to(DEV), None, S)
    _bits_equal(S[:n], S0, f"{what}: S rows of the pins")
    cnt = int(fc.count.item())
    order, lptr = fc.order[:cnt].cpu().numpy(), fc.level_ptr.cpu().numpy()
    fptr, vpin = fc.f_ptr[:cnt + 1].cpu().numpy(), fc.vpin[:cnt].cpu().numpy()
    fsrc = fc.f_src[:int(fptr[-1])].cpu().numpy()
    fitted, sizes, base = fc.fitted.cpu().numpy(), fc.sizes.cpu().numpy(), fc.row_base.cpu().numpy()
    head = fc.head_rows[:K * E.size].cpu().numpy().reshape(K, E.size)
    srows = fc.seed_rows[:seeds.size].cpu().numpy()
    assert lptr[0] == 0 and lptr[-1] == cnt and np.all(np.diff(lptr) >= 0)
    run = 0
    for k, s in enumerate(sets):
        c_order, c_lptr, c_fptr, c_fsrc = _ref_restricted(h, edges, s, rmask)
        assert sizes[k] == len(c_order), f"{what}/{k}: size {sizes[k]} != {len(c_order)}"
        assert bool(fitted[k]) == (run + len(c_order) <= R and all(fitted[:k])), f"{what}/{k}: admission"
        if not fitted[k]:
            assert np.all(srows[ptr[k]:ptr[k + 1]] == n + R), f"{what}/{k}: seeds of a non-admitted candidate"
            continue
        assert base[k] == run
        lo, hi = n + run, n + run + len(c_order)
        srt = np.sort(c_order)
        np.testing.assert_array_equal(vpin[run:run + len(c_order)], srt, err_msg=f"{what}/{k}: rank")
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
        assert not mark[got[~inside]].any(), f"{what}/{k}: a source in the cone kept its pin id"
        for i in range(ptr[k], ptr[k + 1]):
            u = int(seeds[i])
            want = n + run + int(np.searchsorted(srt, u)) if mark[u] else n + R
            assert srows[i] == want, f"{what}/{k}: seed row of {u}"
        want = [n + run + int(np.searchsorted(srt, u)) if mark[u] else u for u in E]
        np.testing.assert_array_equal(head[k], want, err_msg=f"{what}/{k}: head rows")
        _bits_equal(S[lo:hi], S0[vpin[run:run + len(c_order)]], f"{what}/{k}: S copies")
        run += len(c_order)
    assert cnt == run
    return rmask


def _endpoint_kinds(lv, endpoints, rng):
    """Positions of shallow endpoints, deep endpoints and all endpoints."""
    ep_lv = lv[endpoints]
    by = np.argsort(ep_lv, kind="stable")
    sch = by[ep_lv[by] >= 0]
    return {"shallow": sch[:5], "deep": sch[-9:], "all": np.arange(endpoints.size)}


# ------------------------------------------------------------------------------------------------------------------
# 1. cones against numpy
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["tiny", "c1", "c2"])
def test_restricted_cones_match_numpy(mods, cfg):
    d = tm_synth.make_design(seed=5, **tm_synth.CONFIGS[cfg])
    tg = mods["graph"].TimingGraph(d.n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis).to(DEV)
    h = _host(tg.schedule())
    edges = {"net": (d.net_src, d.net_dst), "cell": (d.cell_src, d.cell_dst)}
    rng = np.random.default_rng(3)
    lv, order, lp, L = h["level"], h["order"], h["level_ptr"], h["L"]
    endpoints = np.asarray(d.endpoints, np.int64)
    n_sched = int(lp[L])
    for kind, pos in _endpoint_kinds(lv, endpoints, rng).items():
        E = endpoints[pos]
        rmask = _ref_within(h, E)
        inside = np.nonzero(rmask)[0]
        outside = np.nonzero(~rmask & (lv >= 0))[0]
        unsched = np.nonzero(lv < 0)[0]
        pick = lambda a, m: [int(x) for x in rng.choice(a, min(m, a.size), replace=False)] if a.size else []  # noqa
        sets = [pick(inside, 1), [], pick(outside, 2), pick(inside, 3) + pick(outside, 2), pick(unsched, 1),
                [int(x) for x in rng.choice(d.n, 8)], pick(inside, 1) * 2, [int(order[lp[1]])]]
        _check_restricted(mods, tg, h, edges, sets, E, 4 * n_sched, f"{cfg}/{kind}/all fit")
        sizes = [int(_ref_restricted(h, edges, s, rmask)[0].size) for s in sets]
        R = max(sizes[0] + sizes[1] + sizes[2] + sizes[3] // 2, 1)
        _check_restricted(mods, tg, h, edges, sets, E, R, f"{cfg}/{kind}/R={R}")


@pytest.mark.gpu
def test_restricted_cones_bitmaps_in_global_memory(mods):
    """1.7M pins: the candidates' bitmaps live in the workspace, R(E)'s in its caller buffer."""
    rng = np.random.default_rng(8)
    n, net, cell, pis = _layered_netlist(1_700_000, 21, rng)
    tg = mods["graph"].TimingGraph(n, net, cell, pis=pis).to(DEV)
    h = _host(tg.schedule())
    lp, order, L = h["level_ptr"], h["order"], h["L"]
    edges = {"net": net, "cell": cell}
    top = order[lp[L - 3]:lp[L]]                           # the last three levels
    for kind, E in (("shallow", order[lp[4]:lp[4] + 3]), ("deep", top[-6:]), ("all", top)):
        rmask = _ref_within(h, E)
        inside = np.nonzero(rmask)[0]
        sets = [[int(top[0]), int(top[min(5, top.size - 1)])], [int(x) for x in rng.choice(inside, 2)],
                [int(x) for x in rng.choice(n, 4)], []]
        _check_restricted(mods, tg, h, edges, sets, E, 2 * n, f"big/{kind}")


# ------------------------------------------------------------------------------------------------------------------
# 2. predictions
# ------------------------------------------------------------------------------------------------------------------
def _mixed_sets(b, K, rng, rmask, lo=0, hi=None):
    """_candidate_sets with pins inside R(E) and scheduled pins outside it mixed in."""
    sets = _candidate_sets(b, K, rng, lo, hi)
    lv = b.graph.schedule().level.cpu().numpy()
    hi = lv.size if hi is None else hi
    ids = np.arange(lo, hi)
    inside = ids[rmask[lo:hi]]
    outside = ids[~rmask[lo:hi] & (lv[lo:hi] >= 0)]
    for k in range(K):
        if k % 3 == 1 and inside.size:
            sets[k] = [int(x) for x in rng.choice(inside, min(2, inside.size), replace=False)]
        elif k % 5 == 2 and outside.size:
            sets[k] = [int(x) for x in rng.choice(outside, min(3, outside.size), replace=False)]
        elif k % 7 == 3 and inside.size and outside.size:
            sets[k] = sets[k] + [int(rng.choice(inside)), int(rng.choice(outside))]
    if K == 1 and inside.size:
        sets[0] = [int(rng.choice(inside))]
    return sets


def _positions(b, kind, rng):
    T = int(b.endpoints.numel())
    lv = b.graph.schedule().level.cpu().numpy()
    if kind == "random":
        return np.sort(rng.choice(T, max(1, T // 15), replace=False))
    if kind == "all":
        return np.arange(T)
    return _endpoint_kinds(lv, b.endpoints.cpu().numpy().astype(np.int64), rng)[kind]


def _rmask(b, E):
    return _ref_within(_host(b.graph.schedule()), b.endpoints.cpu().numpy().astype(np.int64)[E])


@pytest.mark.gpu
@pytest.mark.parametrize("cnn,K,kind", [("unet", 1, "shallow"), ("unet", 7, "random"), ("unet", 33, "deep"),
                                        ("unet", 7, "all"), ("layoutnet", 1, "random"), ("layoutnet", 7, "deep"),
                                        ("layoutnet", 33, "random")])
def test_what_if_endpoints_match_forward_bitwise(mods, cnn, K, kind):
    eng = mods["engine"]
    model, net = _models(eng, cnn)
    b = eng.DesignBatch.from_synth(_design(cnn, 21), DEV)
    step = eng.DesignStep(model, net)
    rng = np.random.default_rng(100 + K)
    E = _positions(b, kind, rng)
    rmask = _rmask(b, E)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 4)
    sets = _mixed_sets(b, K, rng, rmask)
    full = inc.what_if(sets)
    wi = inc.what_if(sets, endpoints=E)
    np.testing.assert_array_equal(wi.endpoints, E)
    assert wi.within_size() == int(rmask.sum())
    _edit_candidates(wi, rng)                             # the same edited rows in both objects
    full.cell_feat.copy_(wi.cell_feat)
    full.net_feat.copy_(wi.net_feat)
    ref_all = full.run().clone()
    full_sizes, full_fit = full.cone_sizes(), full.fitted()
    before = _state(model, net)
    base = _base(inc, b)
    pred = wi.run()
    assert pred.shape == (K, E.size)
    assert wi.fitted().all()
    _assert_base(inc, b, base, "after run")
    _assert_state(model, net, before)
    sizes = wi.cone_sizes()
    Et = torch.from_numpy(E).to(DEV)
    h = _host(b.graph.schedule())
    edges = {"net": b.graph._edges["net"], "cell": b.graph._edges["cell"]}
    edges = {k: (v[0].cpu().numpy(), v[1].cpu().numpy()) for k, v in edges.items()}
    for k in range(K):
        pins = wi.rows(k)[0]
        want = _ref_restricted(h, edges, pins, rmask)[0].size
        assert sizes[k] == want, f"candidate {k}: restricted cone {sizes[k]} != {want}"
        assert sizes[k] <= full_sizes[k]
        if want == 0:
            _bits_equal(pred[k], base["pred"][Et], f"candidate {k}: nothing inside R(E) edited")
        if full_fit[k]:                                   # rows the unrestricted call admitted
            _bits_equal(pred[k], ref_all[k][Et], f"{cnn} K={K} {kind}: candidate {k} vs unrestricted run")
        _bits_equal(pred[k], _forward_with(step, b, wi, k)[Et], f"{cnn} K={K} {kind}: candidate {k} vs forward")
    _assert_base(inc, b, base, "after the references")


# ------------------------------------------------------------------------------------------------------------------
# 3. joined batch
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_endpoints_joined_batch(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.concat([eng.DesignBatch.from_synth(_design("unet", 30 + k, n_cells=1500, T=100), DEV)
                                for k in range(2)])
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes())
    rng = np.random.default_rng(5)
    e1, T = int(b.ep_off_h[1]), int(b.endpoints.numel())
    E = np.concatenate([rng.choice(e1, 6, replace=False), e1 + rng.choice(T - e1, 6, replace=False)])
    rmask = _rmask(b, np.sort(E))
    p1 = int(b.pin_off_h[1])
    sets = _mixed_sets(b, 4, rng, rmask, 0, p1) + _mixed_sets(b, 4, rng, rmask, p1)
    wi = inc.what_if(sets, endpoints=list(E) + list(E[:3]))
    np.testing.assert_array_equal(wi.endpoints, np.sort(E))
    _edit_candidates(wi, rng)
    full = inc.what_if(sets)
    full.cell_feat.copy_(wi.cell_feat)
    full.net_feat.copy_(wi.net_feat)
    ref_all = full.run().clone()
    pred = wi.run()
    Et = torch.from_numpy(wi.endpoints).to(DEV)
    other = [(wi.endpoints >= e1), (wi.endpoints < e1)]
    for k in range(len(sets)):
        _bits_equal(pred[k], ref_all[k][Et], f"joined batch: candidate {k} vs unrestricted run")
        _bits_equal(pred[k], _forward_with(step, b, wi, k)[Et], f"joined batch: candidate {k} vs forward")
        o = torch.from_numpy(other[0 if k < 4 else 1]).to(DEV)
        _bits_equal(pred[k][o], inc.pred[Et][o], f"joined batch: candidate {k} leaves the other design alone")


# ------------------------------------------------------------------------------------------------------------------
# 4. admission
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_endpoints_admission(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 45), DEV)
    step = eng.DesignStep(model, net)
    rng = np.random.default_rng(14)
    E = _positions(b, "shallow", rng)
    rmask = _rmask(b, E)
    inside = np.nonzero(rmask)[0]
    K = 12
    sets = [[int(x)] for x in rng.choice(inside, K, replace=inside.size < K)]
    probe = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 3)
    pu, pr = probe.what_if(sets), probe.what_if(sets, endpoints=E)
    pu.run()
    pr.run()
    su, sr = pu.cone_sizes(), pr.cone_sizes()
    R = int(sr.sum())
    assert su.sum() > R, "the test needs candidates whose forward cones leave R(E)"
    inc = step.incremental(b, what_if_rows=R)
    full, wi = inc.what_if(sets), inc.what_if(sets, endpoints=E)
    _edit_candidates(wi, rng)
    full.cell_feat.copy_(wi.cell_feat)
    full.net_feat.copy_(wi.net_feat)
    full.run()
    assert not full.fitted().all(), "the unrestricted call admits every candidate"
    pred = wi.run()
    assert wi.fitted().all(), "the restricted call leaves candidates out"
    Et = torch.from_numpy(E).to(DEV)
    for k in range(K):
        _bits_equal(pred[k], _forward_with(step, b, wi, k)[Et], f"R={R}: candidate {k}")
    # too small even restricted: the prefix rule
    cut = 5
    R2 = max(int(sr[:cut].sum()) + int(sr[cut]) // 2, 1)
    inc2 = step.incremental(b, what_if_rows=R2)
    wi2 = inc2.what_if(sets, endpoints=E)
    wi2.cell_feat.copy_(wi.cell_feat)
    wi2.net_feat.copy_(wi.net_feat)
    base = _base(inc2, b)
    pred2 = wi2.run()
    fit = wi2.fitted()
    np.testing.assert_array_equal(wi2.cone_sizes(), sr)
    run, open_ = 0, True
    for k in range(K):
        open_ = open_ and run + int(sr[k]) <= R2
        assert fit[k] == open_, f"candidate {k}: fitted {fit[k]}, expected {open_}"
        run += int(sr[k]) if open_ else 0
        if fit[k]:
            _bits_equal(pred2[k], pred[k], f"R={R2}: admitted candidate {k}")
        else:
            assert torch.isnan(pred2[k]).all(), f"candidate {k} not admitted but not NaN"
            with pytest.raises(ValueError, match="not admitted"):
                wi2.commit(k)
    assert not fit.all() and fit[0]
    _assert_base(inc2, b, base, "with too few rows")


# ------------------------------------------------------------------------------------------------------------------
# 5. commit
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_endpoints_commit(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    d = _design("unet", 43)
    b = eng.DesignBatch.from_synth(d, DEV)
    b2 = eng.DesignBatch.from_synth(d, DEV)                # the same design, stepped with update
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 2)
    ref = step.incremental(b2)
    rng = np.random.default_rng(15)
    E = _positions(b, "random", rng)
    rmask = _rmask(b, E)
    for rnd in range(4):
        wi = inc.what_if(_mixed_sets(b, 8, rng, rmask), endpoints=E)
        _edit_candidates(wi, rng)
        wi.run()
        k = [1, 2, 5, 0][rnd]                              # inside R(E), outside it, unscheduled pins, late pins
        pins, cf, nf = wi.rows(k)
        wi.commit(k)
        idx = torch.from_numpy(pins).to(DEV)
        b2.cell_feat[idx] = cf
        b2.net_feat[idx] = nf
        ref.update(pins)
        assert inc.cone_size() == ref.cone_size()
        assert inc.generation == ref.generation
        _bits_equal(b.cell_feat, b2.cell_feat, f"commit {rnd}: cell_feat")
        _bits_equal(b.net_feat, b2.net_feat, f"commit {rnd}: net_feat")
        _bits_equal(inc.pred, ref.pred, f"commit {rnd}: pred vs update")
        _bits_equal(inc.H, ref.H, f"commit {rnd}: H vs update")
        _bits_equal(inc.S, ref.S, f"commit {rnd}: S vs update")
        with pytest.raises(ValueError, match="base changed"):
            wi.commit(k)                                   # the commit itself moved the base
    sch = np.nonzero(inc._level >= 0)[0]
    wi = inc.what_if([[int(sch[-1])]], endpoints=E)
    wi.run()
    inc.update([int(sch[0])])
    with pytest.raises(ValueError, match="base changed"):
        wi.commit(0)
    wi.run()
    wi2 = inc.what_if([[]], endpoints=E[:1])
    wi2.run()
    with pytest.raises(ValueError, match="another what-if"):
        wi.commit(0)


# ------------------------------------------------------------------------------------------------------------------
# 6. capture
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_endpoints_capture(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 41), DEV)
    step = eng.DesignStep(model, net)
    inc = step.incremental(b, what_if_rows=b.graph.number_of_nodes() * 2)
    rng = np.random.default_rng(16)
    E = _positions(b, "random", rng)
    Et = torch.from_numpy(E).to(DEV)
    wi = inc.what_if(_mixed_sets(b, 9, rng, _rmask(b, E)), endpoints=E)
    replay = wi.capture()
    for rnd in range(3):
        _edit_candidates(wi, rng)
        base = _base(inc, b)
        before = _state(model, net)
        got = replay().clone()
        _assert_base(inc, b, base, f"replay {rnd}")
        _assert_state(model, net, before)
        _bits_equal(got, wi.run(), f"replay vs eager run, round {rnd}")
        for k in (0, 1, 8):
            _bits_equal(got[k], _forward_with(step, b, wi, k)[Et], f"replay round {rnd}: candidate {k} vs forward")
        pins = rng.choice(np.nonzero(inc._level >= 0)[0], 3, replace=False)
        _edit(b.cell_feat, b.net_feat, pins, rng)
        inc.update(pins)
    got = replay()
    for k in range(wi.K):
        _bits_equal(got[k], _forward_with(step, b, wi, k)[Et], f"replay after updates: candidate {k} vs forward")
    step.close()


# ------------------------------------------------------------------------------------------------------------------
# 7. errors
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_what_if_endpoints_errors(mods):
    eng = mods["engine"]
    model, net = _models(eng, "unet")
    b = eng.DesignBatch.from_synth(_design("unet", 50, n_cells=800, T=60), DEV)
    step = eng.DesignStep(model, net)
    with pytest.raises(ValueError, match="what_if_rows=0"):
        step.incremental(b).what_if([[1]], endpoints=[0])
    inc = step.incremental(b, what_if_rows=1000)
    T = int(b.endpoints.numel())
    for bad in ([], np.zeros(0, np.int64), [T], [-1], [0, T + 3], [0.5], ["a"], [True],
                torch.tensor([1], device=DEV)):
        with pytest.raises(ValueError):
            inc.what_if([[1]], endpoints=bad)
    for ok in ([5, 3, 3], np.array([5, 3]), torch.tensor([3, 5, 5])):
        wi = inc.what_if([[1], [2]], endpoints=ok)
        assert wi.endpoints.dtype == np.int64
        np.testing.assert_array_equal(wi.endpoints, [3, 5])
        assert wi.run().shape == (2, 2)
    wi = inc.what_if([[1], [2, 2]], endpoints=[0, 1])
    with pytest.raises(ValueError):
        wi.commit(0)                                       # never ran
    wi.run()
    for bad in (2, -1, 0.0):
        with pytest.raises(ValueError):
            wi.commit(bad)
    torch.cuda.synchronize()
