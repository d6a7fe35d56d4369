"""Development probe for the persistent propagation kernels (tm_gnn_persist.cu): compares them with
the per-level kernels (impl 0) on small designs and times both on configs 2 / 3.
Usage: python profiles/dev_gnn_persist.py [c2] [c3] [batch8]   -> JSON lines on stdout."""
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_NAME = "multimodal-fusion-based-pre-routing-timing-prediction-_b200"
for p in (ROOT, os.path.join(ROOT, PKG_NAME)):
    sys.path.insert(0, p)
importlib.import_module(PKG_NAME)
import tm_graph  # noqa: E402
import tm_lib  # noqa: E402
import tm_ops  # noqa: E402
import tm_synth  # noqa: E402

DEV = "cuda"


def graph_of(d):
    g = tm_graph.TimingGraph(d.n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis)
    g.ndata["cell_feat"] = torch.from_numpy(d.cell_feat)
    g.ndata["net_feat"] = torch.from_numpy(d.net_feat)
    return g.to(DEV)


def params(seed=0):
    import model as M
    torch.manual_seed(seed)
    gnn = M.PathConv(out_feat_dim=128, hidden_feat_dim=128, cell_feat_dim=36, net_feat_dim=2).to(DEV)
    sd = dict(gnn.named_parameters())
    return [sd[k].detach() for k in tm_ops.GNN_PARAM_NAMES]


def run(sched, g, ps, G0, impl):
    tm_lib.lib().tm_gnn_set_impl(impl)
    H, saved = tm_ops.gnn_forward(sched, g.ndata["cell_feat"], g.ndata["net_feat"], ps, save=True)
    G = G0.clone()
    grads = tm_ops.gnn_backward(sched, saved, ps, G)
    torch.cuda.synchronize()
    return H, saved, G, grads


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def compare(cfg, seed):
    d = tm_synth.make_design(seed=seed, **tm_synth.CONFIGS[cfg])
    g = graph_of(d)
    sched = g.schedule()
    ps = params(seed)
    torch.manual_seed(seed)
    G0 = (0.01 * torch.randn(d.n, 128)).to(DEV)
    H0, s0, Gz0, gr0 = run(sched, g, ps, G0, 0)
    H1, s1, Gz1, gr1 = run(sched, g, ps, G0, 3)
    out = dict(kind="compare", cfg=cfg, seed=seed, n=d.n, levels=sched.num_levels, H=rel(H1, H0), A=rel(s1["A"], s0["A"]),
               LSE=rel(s1["LSE"], s0["LSE"]), HID=rel(s1["HID"], s0["HID"]), Gz=rel(Gz1, Gz0),
               grads=max(rel(a, b) for a, b in zip(gr1, gr0)))
    H1b, _, Gz1b, _ = run(sched, g, ps, G0, 3)
    out["deterministic"] = bool(torch.equal(H1, H1b) and torch.equal(Gz1, Gz1b))
    H16, s16, Gz16, gr16 = run(sched, g, ps, G0, 16)  # per-level kernels, fp16 two-term split cell MLP
    out["h16"] = dict(H=rel(H16, H0), A=rel(s16["A"], s0["A"]), HID=rel(s16["HID"], s0["HID"]), Gz=rel(Gz16, Gz0),
                      grads=max(rel(a, b) for a, b in zip(gr16, gr0)))
    print(json.dumps(out), flush=True)


def timeit(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(iters):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / iters


def concat_designs(ds):
    """Block-diagonal union of designs: one level schedule with wider levels."""
    off = 0
    ns, nd, cs, cd, cf, nf, pis = [], [], [], [], [], [], []
    for d in ds:
        ns.append(d.net_src + off); nd.append(d.net_dst + off)
        cs.append(d.cell_src + off); cd.append(d.cell_dst + off)
        cf.append(d.cell_feat); nf.append(d.net_feat); pis.append(np.asarray(d.pis) + off)
        off += d.n
    g = tm_graph.TimingGraph(off, (np.concatenate(ns), np.concatenate(nd)), (np.concatenate(cs), np.concatenate(cd)),
                             pis=np.concatenate(pis))
    g.ndata["cell_feat"] = torch.from_numpy(np.concatenate(cf))
    g.ndata["net_feat"] = torch.from_numpy(np.concatenate(nf))
    return g.to(DEV), off


def time_cfg(name, g, n):
    sched = g.schedule()
    ps = params(0)
    dev = torch.device(DEV)
    S = torch.randn(n, 128, device=dev) * 0.1
    H = torch.zeros(n, 128, device=dev)
    ncr = sched.n_cell_rows
    A = torch.empty(ncr, 128, device=dev); LSE = torch.empty(ncr, 128, device=dev); HID = torch.empty(ncr, 256, device=dev)
    GA = torch.empty(ncr, 128, device=dev); GHID = torch.empty(ncr, 256, device=dev); GZC = torch.empty(ncr, 128, device=dev)
    G = torch.zeros(n, 128, device=dev)
    cn1w, cn1b, cn2w, cn2b = ps[8], ps[9], ps[10], ps[11]
    w1t, w2t = tm_ops.transpose(cn1w), tm_ops.transpose(cn2w)
    nb = tm_lib.ws_bytes("tm_gnn_ws_bytes")
    ws = tm_lib.workspace(nb, dev)
    st = tm_lib.stream()
    peak = 6544.0
    for impl in (0, 16, 3):
        tm_lib.lib().tm_gnn_set_impl(impl)
        fwd = lambda: tm_lib.call("tm_gnn_forward", sched.struct, 0, sched.num_levels, H, S, w1t, cn1b, w2t, cn2b, A, LSE, HID, ws, nb, st)
        bwd = lambda: tm_lib.call("tm_gnn_backward", sched.struct, H, G, cn1w, cn2w, A, LSE, HID, GA, GHID, GZC, ws, nb, st)
        tf = timeit(fwd)
        G.normal_(std=1e-3)
        tb = timeit(bwd)
        bf, bb = sched.algorithmic_bytes_fwd(), sched.algorithmic_bytes_bwd()
        print(json.dumps(dict(kind="time", cfg=name, impl=impl, n=n, levels=sched.num_levels, fwd_ms=tf, bwd_ms=tb,
                              fwd_gbs=bf / tf / 1e6, bwd_gbs=bb / tb / 1e6, fwd_frac=bf / tf / 1e6 / peak,
                              bwd_frac=bb / tb / 1e6 / peak, barriers=int(tm_lib.lib().tm_gnn_last_barriers()))), flush=True)
    tm_lib.lib().tm_gnn_set_impl(3)
    # phase clocks of one forward and one backward pass (thread 0 of every CTA)
    names = ["setup", "cell_pre", "gather", "mma1", "epi1", "mma2", "exch", "cell_pub", "net_pre", "net_body", "net_tail"]
    for what, fn in (("fwd", fwd), ("bwd", bwd)):
        prof = torch.zeros(148, 16, dtype=torch.int64, device=dev)
        tm_lib.call("tm_gnn_set_profile", prof)
        fn()
        torch.cuda.synchronize()
        tm_lib.call("tm_gnn_set_profile", None)
        pm = prof.double().cpu().numpy()
        print(json.dumps(dict(kind="phases", cfg=name, what=what,
                              mean_us={k: round(float(pm[:, i].mean()) / 1965.0, 1) for i, k in enumerate(names)},
                              max_us={k: round(float(pm[:, i].max()) / 1965.0, 1) for i, k in enumerate(names)},
                              total_us=round(float(pm.sum(1).mean()) / 1965.0, 1))), flush=True)


if __name__ == "__main__":
    what = sys.argv[1:] or ["compare"]
    if "compare" in what:
        for cfg, seed in (("tiny", 0), ("tiny", 5), ("c1", 1)):
            compare(cfg, seed)
    for cfg in ("c2", "c3"):
        if cfg in what:
            d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS[cfg])
            time_cfg(cfg, graph_of(d), d.n)
    if "batch8" in what:
        ds = [tm_synth.make_design(seed=s, **tm_synth.CONFIGS["c2"]) for s in range(8)]
        g, n = concat_designs(ds)
        time_cfg("c2x8", g, n)
