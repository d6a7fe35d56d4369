"""What compute-sanitizer runs (memcheck / racecheck, one tool per gpurun call): smoke() -- schedule build incl. the
cooperative levelizer, the PDL-chained per-level kernels, tcgen05 GEMMs with their mbarrier rings and TMEM
alloc/dealloc, fusion, head -- plus the persistent cluster kernels on a tiny design."""
import importlib, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "multimodal-fusion-based-pre-routing-timing-prediction-_b200"
for p in (ROOT, os.path.join(ROOT, PKG)):
    sys.path.insert(0, p)
import __graft_entry__ as g
g.smoke()
importlib.import_module(PKG)
import model as M, tm_graph, tm_lib, tm_ops, tm_synth
d = tm_synth.make_design(seed=1, **tm_synth.CONFIGS["tiny"])
gr = tm_graph.TimingGraph(d.n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis)
gr.ndata["cell_feat"], gr.ndata["net_feat"] = torch.from_numpy(d.cell_feat), torch.from_numpy(d.net_feat)
gr = gr.to("cuda")
torch.manual_seed(0)
gnn = M.PathConv(out_feat_dim=128, hidden_feat_dim=128, cell_feat_dim=36, net_feat_dim=2).to("cuda")
tm_lib.lib().tm_gnn_set_impl(3)
H = gnn.propagate(gr)
H.backward(torch.randn_like(H))
torch.cuda.synchronize()
print("persistent kernels ok", float(H.abs().sum()))
tm_lib.check_err_flags()
