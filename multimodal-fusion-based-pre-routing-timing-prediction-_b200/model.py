"""Drop-in ``model`` module: MLP, PathConv, LayoutNet, PathModel on libtm_b200 (sm_100a).

Same module name, class names, constructor / ``forward`` signatures and parameter names as the
reference's ``src/model.py`` (pickles made by ``src/train.py:86-89`` resolve ``model.PathModel``
etc.; ``state_dict`` keys are interchangeable), so ``train.py`` / ``test.py`` can import it
unchanged (``from model import *`` also re-exports ``th``, ``nn``, ``fn``, ``F`` as they rely on).
The arithmetic runs in hand-written CUDA kernels through the C ABI of ``include/tm_b200.h``;
there is no CPU or library fallback -- inputs must live on a CUDA device.

What differs from the reference on purpose (SURVEY.md 2.3):
* ``PathConv.forward`` runs the WHOLE level-wise propagation when it is called for level 0 (one
  pass over a precomputed level schedule) and later level calls only gather rows, which is
  equivalent because every pin is written exactly once, on its own level (model.py:158-213);
* ``PathModel`` also accepts the legacy ``PathModel(gnn, fcn, mlp)`` call of train.py:81 (D1/D2);
* ``path_map`` may be a ``MaskedFeatureMap`` (sparse mask rows + feature map) instead of the
  dense (T, map^2) product of train.py:500-501;
* the unrunnable attention variant (``flag_attn``: needs ``ndata['key']`` that nothing creates)
  raises ``NotImplementedError``.
"""
import torch as th
from torch import nn
import torch.nn.functional as F

try:                                            # train.py only needs the name to exist
    from dgl import function as fn
except Exception:                               # DGL is optional: TimingGraph replaces it
    class _NoDGL:
        def __getattr__(self, name):
            raise ImportError("dgl is not installed; PathConv does not need it")
    fn = _NoDGL()

import tm_ops
import tm_unet
from tm_graph import as_timing_graph
from tm_ops import MaskedFeatureMap


def cell_msg_reduce(nodes):
    """Unused max-reduce UDF kept for ``from model import *`` parity (reference model.py:6-7)."""
    return {'h_neigh1': th.max(nodes.mailbox['m'], dim=1)}


class MLP(th.nn.Module):
    """Linear -> LeakyReLU(negative_slope) [-> Dropout(0.2)] [-> BatchNorm1d] ... -> Linear."""

    def __init__(self, *sizes, batchnorm=False, dropout=False, negative_slope=0):
        super().__init__()
        mods = []
        for i, (a, b) in enumerate(zip(sizes[:-1], sizes[1:])):
            mods.append(th.nn.Linear(a, b))
            if i < len(sizes) - 2:
                mods.append(th.nn.LeakyReLU(negative_slope=negative_slope))
                if dropout:
                    mods.append(th.nn.Dropout(p=0.2))
                if batchnorm:
                    mods.append(th.nn.BatchNorm1d(b))
        self.layers = th.nn.Sequential(*mods)

    def forward(self, x):
        mods = list(self.layers)
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, th.nn.Linear):
                nxt = mods[i + 1] if i + 1 < len(mods) else None
                fuse = isinstance(nxt, th.nn.LeakyReLU) and nxt.negative_slope == 0
                x = tm_ops.linear(x, m.weight, m.bias, relu=fuse)      # fused bias + ReLU epilogue
                i += 2 if fuse else 1
            else:                                                       # Dropout / BatchNorm1d / leaky
                x = m(x)
                i += 1
        return x


class PathConv(nn.Module):
    def __init__(self, out_feat_dim, hidden_feat_dim, cell_feat_dim, net_feat_dim, flag_attn=False,
                 num_heads=1, activation=th.nn.functional.relu, bias=True, norm=None):
        super(PathConv, self).__init__()
        self.flag_attn = flag_attn
        self.hidden_feat_dim = hidden_feat_dim
        self.out_feat_dim = out_feat_dim
        self.cell_feat_dim = cell_feat_dim
        self.net_feat_dim = net_feat_dim
        self.num_heads = num_heads
        # creation order == reference (model.py:48-54) so seeded initialisation matches
        self.fc_cell_neigh = MLP(hidden_feat_dim, 256, out_feat_dim)
        self.fc_cell_self = MLP(cell_feat_dim, 256, out_feat_dim)
        self.fc_net_self = MLP(net_feat_dim, 256, out_feat_dim)
        self.fc_net_drive = MLP(2, out_feat_dim)                 # never used (no gradient), kept for parity
        self.fc_attn2 = nn.Linear(out_feat_dim, 1, bias=False)   # never used, kept for parity
        if flag_attn:
            self.fc_key = nn.Linear(1, 256, bias=False)
            self.fc_attn = nn.Linear(2 * 256, 1, bias=False)
        self.activation = activation
        self.norm = norm
        self._prop = None

    def __getstate__(self):                                      # whole-module pickles (train.py:86-89)
        d = self.__dict__.copy()
        d["_prop"] = None
        return d

    def _params(self):
        sd = dict(self.named_parameters())
        return [sd[k] for k in tm_ops.GNN_PARAM_NAMES]

    def propagate(self, graph):
        """All levels in one pass; returns H (N, out_feat_dim) and caches it for the level calls."""
        if self.flag_attn:
            raise NotImplementedError("flag_attn=True is not runnable in the reference either "
                                      "(ndata['key'] is never created)")
        if self.activation is not th.nn.functional.relu or self.norm is not None:
            raise NotImplementedError("the CUDA propagation implements activation=relu, norm=None "
                                      "(the only configuration the reference constructs, train.py:56-63)")
        g = as_timing_graph(graph)
        sched = g.schedule()
        params = self._params()
        need = th.is_grad_enabled() and any(p.requires_grad for p in params)
        H = tm_ops.GnnPropagateFn.apply(sched, g.ndata['cell_feat'], g.ndata['net_feat'], need, *params)
        self._prop = (g, sched, H)
        g.ndata['h'] = H                                          # what model.py:208 leaves behind
        return H

    def forward(self, graph, cur_nodes, eids, targets, level_id):
        g = as_timing_graph(graph)
        if level_id == 0 or self._prop is None or self._prop[0] is not g:
            if level_id != 0:
                raise RuntimeError("PathConv must be called from level 0 upwards (train.py:489)")
            self.propagate(g)
        _, sched, H = self._prop
        if level_id >= sched.num_levels or \
                len(cur_nodes) != int(sched.h_level_ptr[level_id + 1] - sched.h_level_ptr[level_id]):
            raise RuntimeError(f"level {level_id}: the caller's node list does not match the level schedule; "
                               "pass the batch's own levels with graph.set_topo_levels(topo_levels)")
        if len(targets) == 0:                                     # most levels carry no sampled endpoint: no launch, no copy
            return H[:0]
        idx = th.as_tensor(targets, dtype=th.int64, device=H.device)
        return H[idx]


class LayoutNet(nn.Module):
    def __init__(self, pooling):
        super(LayoutNet, self).__init__()
        if pooling == 'max':
            pool = lambda: nn.MaxPool2d(2, 2, 0, 1)              # noqa: E731
        elif pooling == 'avg':
            pool = lambda: nn.AvgPool2d(2, 2, 0)                 # noqa: E731
        else:
            assert False, 'wrong pooling type for layoutnet!'
        self.pooling = pooling
        self.encode = nn.Sequential(
            nn.Conv2d(2, 32, 9, 1, 4), nn.ReLU(), pool(),
            nn.Conv2d(32, 64, 7, 1, 3), nn.ReLU(), pool(),
            nn.Conv2d(64, 32, 9, 1, 4), nn.ReLU(),
            nn.Conv2d(32, 1, 7, 1, 3), nn.LeakyReLU(negative_slope=0.1))

    def forward(self, x):
        params = list(self.parameters())
        need = th.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
        return tm_unet.LayoutNetFn.apply(self, x, need, *params)


class PathModel(nn.Module):
    def __init__(self, gnn, cnn, fcn, mlp_impact=None, mlp_weight=None, mlp_fuse=None, global_dim=32):
        super(PathModel, self).__init__()
        if mlp_fuse is None and mlp_impact is None and mlp_weight is None and isinstance(fcn, MLP):
            # legacy call PathModel(gnn, fcn, mlp) of train.py:81: rebind and size the level
            # embedding from the head the caller built (train.py:76 uses 64, not 32)
            cnn, fcn, mlp_fuse = None, cnn, fcn
            used = (gnn.out_feat_dim if gnn is not None else 0) + (fcn.out_features if fcn is not None else 0)
            global_dim = mlp_fuse.layers[0].in_features - used
        self.global_dim = global_dim
        self.gnn = gnn
        self.cnn = cnn
        self.mlp_impact = mlp_impact
        self.mlp_weight = mlp_weight
        self.fcn = fcn
        self.mlp_fuse = mlp_fuse
        self.mlp_alpha = MLP(1, global_dim * 2, global_dim)

    def forward(self, graph, nodes, eids, target_list, level_id, level_id_th, path_map):
        n_t = len(target_list)
        h_cnn = None
        if self.fcn is not None and n_t != 0:
            if isinstance(path_map, MaskedFeatureMap):
                h_cnn = tm_ops.MaskFusionFn.apply(path_map.mask_rows, path_map.feat_map,
                                                  self.fcn.weight, self.fcn.bias)
            else:
                h_cnn = tm_ops.linear(path_map, self.fcn.weight, self.fcn.bias)
        h_gnn = self.gnn(graph, nodes, eids, target_list, level_id) if self.gnn is not None else None
        if n_t == 0:
            return None
        h_global = self.mlp_alpha(level_id_th).expand(n_t, self.global_dim)
        parts = [p for p in (h_gnn, h_cnn) if p is not None] + [h_global]
        return self.mlp_fuse(th.cat(parts, dim=1)).squeeze(-1)
