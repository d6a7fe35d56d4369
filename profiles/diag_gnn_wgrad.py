"""Warm timings of the non-propagation pieces of the netlist branch (hoisted self MLPs forward, weight gradients
backward) on config 2, one piece at a time.  Usage: python profiles/diag_gnn_wgrad.py -> JSON."""
import importlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_NAME = "multimodal-fusion-based-pre-routing-timing-prediction-_b200"
for p in (ROOT, os.path.join(ROOT, PKG_NAME)):
    sys.path.insert(0, p)
importlib.import_module(PKG_NAME)
import tm_ops  # noqa: E402
import tm_synth  # noqa: E402
from dev_gnn_persist import graph_of, params, timeit  # noqa: E402

D = 128


def main():
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS[os.environ.get("TM_DIAG_CFG", "c2")])
    g = graph_of(d)
    sched = g.schedule()
    ps = params(0)
    (cs1w, cs1b, cs2w, cs2b, ns1w, ns1b, ns2w, ns2b, cn1w, cn1b, cn2w, cn2b) = ps
    dev = torch.device("cuda")
    cf, nf = g.ndata["cell_feat"], g.ndata["net_feat"]
    nc, nn_ = int(sched.cell_class.numel()), int(sched.net_class.numel())
    ncr = sched.n_cell_rows
    n = sched.n
    out = dict(n=n, nc=nc, nn=nn_, ncr=ncr)
    S = torch.empty(n, D, device=dev)
    hc = tm_ops.mlp2_forward(cf, cf.stride(0), sched.cell_class, nc, cs1w, cs1b, cs2w, cs2b, S, D, out_rows=sched.cell_class)
    out["fwd_cell_self_ms"] = timeit(lambda: tm_ops.mlp2_forward(cf, cf.stride(0), sched.cell_class, nc, cs1w, cs1b, cs2w, cs2b, S, D,
                                                                 out_rows=sched.cell_class))
    out["fwd_net_self_ms"] = timeit(lambda: tm_ops.mlp2_forward(nf, nf.stride(0), sched.net_class, nn_, ns1w, ns1b, ns2w, ns2b, S, D,
                                                                out_rows=sched.net_class))
    G = torch.randn(n, D, device=dev) * 1e-3
    GZC = torch.randn(ncr, D, device=dev) * 1e-3
    GHID = torch.randn(ncr, 256, device=dev) * 1e-3
    HID = torch.randn(ncr, 256, device=dev).relu_()
    A = torch.randn(ncr, D, device=dev)
    w = torch.empty(D, 256, device=dev); b = torch.empty(D, device=dev)
    w1 = torch.empty(256, D, device=dev); b1 = torch.empty(256, device=dev)

    def neigh():
        tm_ops.gemm_tn(D, 256, ncr, GZC, D, HID, 256, w, 256, colsum_a=b)
        tm_ops.gemm_tn(256, D, ncr, GHID, 256, A, D, w1, D, colsum_a=b1)
        tm_ops.aux_join()
    out["bwd_cell_neigh_wgrads_ms"] = timeit(neigh)
    out["bwd_cell_neigh_gemm_only_ms"] = timeit(lambda: (tm_ops.gemm_tn(D, 256, ncr, GZC, D, HID, 256, w, 256),
                                                         tm_ops.gemm_tn(256, D, ncr, GHID, 256, A, D, w1, D)))
    out["colsum_256_ms"] = timeit(lambda: tm_ops.colsum(GHID, ncr, 256, 256))
    out["colsum_128_ms"] = timeit(lambda: tm_ops.colsum(GZC, ncr, D, D))
    out["bwd_cell_self_ms"] = timeit(lambda: tm_ops.mlp2_backward(cf, cf.stride(0), sched.cell_class, nc, cs1w, cs2w, hc, G, D,
                                                                  g_rows=sched.cell_class, b1=cs1b))
    out["bwd_net_self_ms"] = timeit(lambda: tm_ops.mlp2_backward(nf, nf.stride(0), sched.net_class, nn_, ns1w, ns2w, None, G, D,
                                                                 g_rows=sched.net_class, b1=ns1b))
    # the pieces of the cell-self backward
    hid = 256
    dw2 = torch.empty(D, hid, device=dev); db2 = torch.empty(D, device=dev)
    out["cs_dw2_ms"] = timeit(lambda: tm_ops.gemm_tn(D, hid, nc, G, D, hc, hid, dw2, hid, a_rows=sched.cell_class))
    dh = torch.empty(nc, hid, device=dev)
    out["cs_dh_ms"] = timeit(lambda: tm_ops.gemm_nn(nc, hid, D, G, D, cs2w, hid, dh, hid, a_rows=sched.cell_class, mask=hc, ldmask=hid))
    dw1 = torch.empty(hid, cf.shape[1], device=dev)
    out["cs_dw1_ms"] = timeit(lambda: tm_ops.gemm_tn(hid, cf.shape[1], nc, dh, hid, cf, cf.stride(0), dw1, cf.shape[1], b_rows=sched.cell_class))
    print(json.dumps({k: (round(v, 4) if isinstance(v, float) else v) for k, v in out.items()}), flush=True)


if __name__ == "__main__":
    main()
