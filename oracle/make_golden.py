"""Generate ``tests/golden/*.npz`` by running the UNMODIFIED reference here.

Oracle / test infrastructure only.  Needs a checkout of the original project:
``TM_REFERENCE_SRC=<reference>/src python oracle/make_golden.py``.

* ``step_<cfg>.npz``   one design step of the reference's own ``PathModel`` /
  ``PathConv`` / ``MLP`` (``src/model.py``) + ``UNet`` (``src/Unet.py``) driven
  exactly like ``src/train.py:465,490-522,552-553`` through ``fake_dgl``:
  inputs, initial weights, predictions, loss, H, feature map, every parameter
  gradient, BN running statistics after the step.
* ``levels_<cfg>.npz`` the reference's own ``cal_topo_level`` and
  ``find_critical_path`` (``verilog_parser_asap7.py:1433-1517``) executed on a
  networkx graph of the same design: pin->level map and critical paths.
* ``layoutnet.npz``    reference ``LayoutNet`` forward/backward on a small image.
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG = os.path.join(ROOT, "multimodal-fusion-based-pre-routing-timing-prediction-_b200")
sys.path.insert(0, ROOT)
sys.path.insert(0, PKG)

import tm_synth  # noqa: E402
from oracle import fake_dgl, ref_loader  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def build_reference_models(map_size, seed):
    m, u = ref_loader.ref_model(), ref_loader.ref_unet()
    torch.manual_seed(seed)
    gnn = m.PathConv(out_feat_dim=128, hidden_feat_dim=128, cell_feat_dim=36, net_feat_dim=2)
    fcn = torch.nn.Linear(map_size * map_size, 128)                       # train.py:71-73
    torch.nn.init.xavier_uniform_(fcn.weight, gain=torch.nn.init.calculate_gain("relu"))
    model = m.PathModel(gnn, None, fcn, None, None, m.MLP(128 + 128 + 32, 2 * (128 + 128 + 32), 1))
    cnn = u.UNet("max")
    model.train(); cnn.train()
    return model, cnn


def reference_step(model, cnn, d):
    """The loop of train.py:465,490-522,552-553 on one design, all endpoints in one batch."""
    g = fake_dgl.FakeGraph(d.n, {"net": (d.net_src, d.net_dst), "cell": (d.cell_src, d.cell_dst)})
    g.ndata["cell_feat"] = torch.from_numpy(d.cell_feat)
    g.ndata["net_feat"] = torch.from_numpy(d.net_feat)
    g.ndata["h"] = torch.zeros(d.n, 128)
    feat_map = cnn(torch.from_numpy(d.image).unsqueeze(0))                # 4-D like train.py:178
    flat = feat_map.reshape(1, -1)
    width = d.map_size * d.map_size
    rows = np.repeat(np.arange(d.endpoints.size), np.diff(d.mask_indptr))
    path_masks = torch.sparse_coo_tensor(np.stack([rows, d.mask_cols.astype(np.int64)]),
                                         torch.ones(d.mask_cols.size, dtype=torch.int64),
                                         (d.endpoints.size, width))
    hats = None
    for level_id, (nodes, targets, paths) in enumerate(d.topo_levels()):
        if len(paths) == 0:
            path_map = None
        else:
            path_map = torch.index_select(path_masks, 0, torch.tensor(paths)).to_dense() * flat
        cur = model(g, nodes, targets, targets, level_id,
                    torch.tensor(level_id, dtype=torch.float).unsqueeze(0), path_map)
        if len(paths) == 0:
            continue
        hats = cur if hats is None else torch.cat((hats, cur), 0)
    loss = torch.nn.MSELoss()(hats, torch.from_numpy(d.arrival_time))
    loss.backward()
    return hats.detach(), loss.detach(), g.ndata["h"].detach(), feat_map.detach()


def dump_step(cfg, seed=0):
    d = tm_synth.make_design(seed=seed, **tm_synth.CONFIGS[cfg])
    model, cnn = build_reference_models(d.map_size, seed)
    sd_m = {k: v.detach().clone().numpy() for k, v in model.state_dict().items()}
    sd_c = {k: v.detach().clone().numpy() for k, v in cnn.state_dict().items()}
    pred, loss, H, fmap = reference_step(model, cnn, d)
    out = {"pred": pred.numpy(), "loss": loss.numpy(), "H": H.numpy(), "feat_map": fmap.numpy()}
    for k, v in sd_m.items():
        out["model." + k] = v
    for k, v in sd_c.items():
        out["cnn." + k] = v
    for k, p in model.named_parameters():
        out["grad.model." + k] = (p.grad.numpy() if p.grad is not None else np.zeros(0, np.float32))
    for k, p in cnn.named_parameters():
        out["grad.cnn." + k] = p.grad.numpy()
    for k, v in cnn.state_dict().items():
        if "running" in k or "num_batches" in k:
            out["after.cnn." + k] = v.numpy()
    np.savez_compressed(os.path.join(GOLD, f"step_{cfg}.npz"), **out)
    print("step", cfg, "n", d.n, "loss", float(loss), "pred[:3]", pred[:3].tolist())


def dump_levels(cfg, seed=0):
    import networkx as nx
    cal_topo_level, find_critical_path = ref_loader.ref_parser_funcs()
    d = tm_synth.make_design(seed=seed, **tm_synth.CONFIGS[cfg])
    name = lambda i: f"p{int(i)}"                                          # noqa: E731
    G = nx.DiGraph()
    G.add_nodes_from(name(i) for i in range(d.n))
    # an unreachable island to exercise node removal (verilog_parser_asap7.py:1513-1515)
    extra = d.n
    G.add_edge(name(extra), name(extra + 1))
    for s, t in zip(np.concatenate([d.net_src, d.cell_src]), np.concatenate([d.net_dst, d.cell_dst])):
        G.add_edge(name(s), name(t))
    pos = {name(e) for e in d.endpoints}
    po2path = {name(e): i for i, e in enumerate(d.endpoints)}
    me = SimpleNamespace(graph=G)
    levels = cal_topo_level(me, {name(p) for p in d.pis}, pos, po2path)
    node_level = np.full(d.n + 2, -1, np.int32)
    targets_level = np.full(d.endpoints.size, -1, np.int32)
    for lid, (nodes, targets, path_ids) in enumerate(levels):
        node_level[[int(x[1:]) for x in nodes]] = lid
        targets_level[path_ids] = lid
        assert [po2path[t] for t in targets] == path_ids
    me.node2level = {name(i): int(l) for i, l in enumerate(node_level)}
    paths = [np.array([int(x[1:]) for x in find_critical_path(me, name(e))], np.int64)
             for e in d.endpoints]
    plen = np.array([len(p) for p in paths], np.int64)
    np.savez_compressed(os.path.join(GOLD, f"levels_{cfg}.npz"), node_level=node_level,
                        targets_level=targets_level, remaining=np.array(sorted(int(x[1:]) for x in G.nodes())),
                        path_len=plen, path_flat=np.concatenate(paths))
    print("levels", cfg, "num_levels", len(levels), "removed", d.n + 2 - G.number_of_nodes())


def dump_layoutnet(seed=0):
    m = ref_loader.ref_model()
    torch.manual_seed(seed)
    net = m.LayoutNet("max")
    x = torch.rand(2, 2, 32, 32)
    y = net(x)
    y.square().sum().backward()
    out = {"x": x.numpy(), "y": y.detach().numpy()}
    for k, p in net.named_parameters():
        out["p." + k] = p.detach().numpy()
        out["g." + k] = p.grad.numpy()
    np.savez_compressed(os.path.join(GOLD, "layoutnet.npz"), **out)
    print("layoutnet", tuple(y.shape))


if __name__ == "__main__":
    assert ref_loader.available(), "set TM_REFERENCE_SRC to the original project's src/ directory"
    os.makedirs(GOLD, exist_ok=True)
    dump_step("tiny")
    dump_levels("tiny")
    dump_levels("c1")
    dump_layoutnet()
