"""Fused design step: image network (U-Net or LayoutNet) + level-wise GNN + mask fusion + head, forward and backward.

``DesignStep.run(batch)`` performs what one optimisation step of the reference does to one design
with all sampled endpoints in a batch (src/train.py:465 CNN forward, :490-511 level loop,
:513-522 MSE on arrival time, :552-553 backward) as a straight sequence of libtm_b200 launches
with no autograd graph, then leaves the gradients in ``param.grad`` (like ``optim.zero_grad();
loss.backward()``).  It is numerically the same computation the ``nn.Module`` surface
(``model.py`` / ``Unet.py``) performs through autograd; tests check both against the oracle.

Data parallelism (SURVEY.md 8e): designs are independent samples, so ranks own disjoint designs
and the only exchange is one gradient all-reduce per step.  ``DesignStep`` posts it in three
buckets on a side stream as soon as each group of gradients exists (head+fusion -> GNN ->
U-Net), so the NCCL transfers over NVLink overlap the remaining backward kernels.
"""
import os

import numpy as np
import torch

import tm_dp
import tm_lib
import tm_ops
import tm_unet
from tm_graph import ConeGraph, FaninCone, ForwardCone, ForwardCones, MaskCSR, TimingGraph
from tm_lib import call, stream
from tm_ops import D, RELU, gemm_nn, gemm_tn, transpose


def build_models(map_size, pooling="max", seed=0, device="cuda", cnn="unet"):
    """Reference wiring (train.py:56-81 with the head sized as model.py:267,280 produce it).  ``cnn``: "unet" (the
    reference's ``--unet``) or "layoutnet" (its default, train.py:70); LayoutNet takes a 2-channel image of 4x the
    map size.  ``TM_UNET_MATH`` sets the math mode of either network."""
    import model as M
    import Unet as U
    torch.manual_seed(seed)
    gnn = M.PathConv(out_feat_dim=128, hidden_feat_dim=128, cell_feat_dim=36, net_feat_dim=2)
    fcn = torch.nn.Linear(map_size * map_size, 128)
    torch.nn.init.xavier_uniform_(fcn.weight, gain=torch.nn.init.calculate_gain("relu"))
    mdl = M.PathModel(gnn, None, fcn, None, None, M.MLP(128 + 128 + 32, 2 * (128 + 128 + 32), 1))
    if cnn == "unet":
        net = U.UNet(pooling)
    elif cnn == "layoutnet":
        net = M.LayoutNet(pooling)
    else:
        raise ValueError(f"build_models: cnn must be 'unet' or 'layoutnet', not {cnn!r}")
    if os.environ.get("TM_UNET_MATH"):                 # e.g. "bf16": image branch on the TMA-fed bf16 tensor-core path
        net.math = os.environ["TM_UNET_MATH"]
    return mdl.to(device).train(), net.to(device).train()


class HostDesign:
    """A design in pinned host memory: what a data loader hands over each step."""

    FIELDS = ("net_src", "net_dst", "cell_src", "cell_dst", "cell_feat", "net_feat", "pis", "endpoints",
              "endpoint_level", "arrival_time", "mask_indptr", "mask_cols", "image")

    def __init__(self, d, pin=True):
        self.n, self.map_size = d.n, d.map_size
        t = {"net_src": d.net_src, "net_dst": d.net_dst, "cell_src": d.cell_src, "cell_dst": d.cell_dst,
             "cell_feat": d.cell_feat, "net_feat": d.net_feat, "pis": d.pis, "endpoints": d.endpoints.astype(np.int32),
             "endpoint_level": d.level[d.endpoints].astype(np.float32), "arrival_time": d.arrival_time,
             "mask_indptr": d.mask_indptr, "mask_cols": d.mask_cols, "image": d.image}
        self.t = {}
        for k, v in t.items():
            x = torch.from_numpy(np.ascontiguousarray(v))
            self.t[k] = x.pin_memory() if pin and torch.cuda.is_available() else x

    def nbytes(self, per_step_only=False):
        keys = ("cell_feat", "net_feat", "endpoints", "endpoint_level", "arrival_time", "mask_indptr",
                "mask_cols", "image") if per_step_only else self.FIELDS
        return int(sum(self.t[k].numel() * self.t[k].element_size() for k in keys))


class DesignBatch:
    """Device-resident batch of one design, or of K designs joined by ``DesignBatch.concat``."""

    def __init__(self, graph, mask_csr, endpoints, endpoint_level, arrival_time, image, cell_feat=None, net_feat=None,
                 rows=None, dynamic=False, mask_rows=None):
        self.graph, self.mask_csr = graph, mask_csr
        # per-batch feature tensors (a prefetched batch must not disturb the one in flight through
        # the shared graph object); default: whatever the graph carries
        self.cell_feat = cell_feat if cell_feat is not None else graph.ndata["cell_feat"]
        self.net_feat = net_feat if net_feat is not None else graph.ndata["net_feat"]
        self.endpoints = endpoints                 # int32 (T,)
        self.endpoint_level = endpoint_level       # float32 (T,)
        self.arrival_time = arrival_time           # float32 (T,)
        self.image = image                         # (C,H,W); (K,C,H,W) for K designs
        # rows: the mask row (path id) of every endpoint -- th.index_select(path_masks, 0, paths), train.py:500;
        # None: endpoint t owns row t (one design's endpoints in one batch, test.py:176)
        if mask_rows is None:
            mask_rows = [mask_csr.select(rows) if rows is not None else mask_csr.select_all()]
        # one MaskRows per design; design k owns endpoints ep_off[k]..ep_off[k+1] of this batch
        self.mask_rows_list = list(mask_rows)
        self.mask_rows = self.mask_rows_list[0] if len(self.mask_rows_list) == 1 else None
        self.K = len(self.mask_rows_list)
        self.width = self.mask_rows_list[0].csr.width
        self.ep_off_h = np.concatenate([[0], np.cumsum([r.T for r in self.mask_rows_list])]).astype(np.int64)
        self.ep_off = None                         # int32 (K+1,) on the device: set by concat (K > 1 only)
        self.pin_off_h = None                      # first pin of every design in the joined netlist (concat)
        self.design_losses = None                  # (K,) device tensor, rewritten by every step / replay (K > 1)
        self.input_grads = None                    # {"cell_feat", "net_feat", "image"}: DesignStep.run(input_grads=True)
        # per-endpoint required time (float32) and critical label (int64, 0 = non-critical), both (T,) on the device:
        # when set, DesignStep.evaluate counts judge_critical's confusion matrix (train.py:391-395)
        self.required = None
        self.label = None
        self._fuse_table = None
        self._segments = None
        # dynamic: the endpoint batch (endpoints / levels / labels / mask rows) is refreshed IN PLACE between steps, so
        # the step re-runs the on-device row selection every time (captured into its CUDA graph): one capture per
        # design serves every shuffled batch of the reference's DataLoader (train.py:470-486)
        self.dynamic = bool(dynamic)
        self._cone = None

    def cone(self):
        """``tm_graph.ConeGraph`` of this batch's endpoints (cached): the sub-netlist that can reach an endpoint, on
        which ``DesignStep(..., prune=True)`` runs -- same predictions, loss and gradients over a fraction of the pins.
        None for a dynamic batch, whose endpoints change between replays of one captured step (the step then runs on
        the whole netlist).  The endpoints of a non-dynamic batch must not be modified in place."""
        if self.dynamic:
            return None
        if self._cone is None:
            self._cone = ConeGraph(self.graph, self.endpoints)
        return self._cone

    def set_endpoints(self, endpoints, endpoint_level, arrival_time, rows, design=0):
        """Refresh the endpoint batch in place (same batch size): what changes between two DataLoader batches.
        ``design``: which design of a joined batch (its pin ids as in its own netlist)."""
        s, e = int(self.ep_off_h[design]), int(self.ep_off_h[design + 1])
        if self.pin_off_h is not None:
            endpoints = endpoints + int(self.pin_off_h[design])
        self.endpoints[s:e].copy_(endpoints, non_blocking=True)
        self.endpoint_level[s:e].copy_(endpoint_level, non_blocking=True)
        self.arrival_time[s:e].copy_(arrival_time, non_blocking=True)
        self.mask_rows_list[design].rows.copy_(rows, non_blocking=True)
        self._cone = None
        self._segments = None

    def fuse_table(self):
        """int64 (K, 5) device table of every design's mask-row buffers {run_ptr, run_lo, run_hi, csc_ptr, csc_t}
        (read by the batched fusion kernels).  The buffers are allocated once and rewritten in place by
        ``MaskRows.rebuild``, so the table stays valid under CUDA-graph replay."""
        if self._fuse_table is None:
            rows = []
            for r in self.mask_rows_list:
                run_ptr, run_lo, run_hi = r.runs()
                csc_ptr, csc_t = r.csc()
                rows.append([t.data_ptr() for t in (run_ptr, run_lo, run_hi, csc_ptr, csc_t)])
            self._fuse_table = torch.tensor(rows, dtype=torch.int64).to(self.endpoints.device)
        return self._fuse_table

    def eval_segments(self):
        """(seg_ptr, seg_idx, L): the int32 device CSR of ``DesignStep.evaluate``'s metric rows (cached).  Row 0 is the
        whole batch, rows 1..K the designs (``ep_off_h``), then K x L rows: design k's endpoints on endpoint level l at
        row 1 + K + k * L + l, L = the largest endpoint level + 1.  Inside a row the endpoints keep the batch's order.
        Built on the host from ``endpoint_level`` (one device-to-host read), so build it before a capture; a captured
        evaluation keeps the levels it was built with."""
        if self._segments is None:
            lv = self.endpoint_level.detach().cpu().numpy()
            if lv.size and (lv.min() < 0 or not np.all(lv == np.round(lv))):
                raise ValueError("DesignBatch.eval_segments: endpoint levels must be non-negative integers")
            lv = lv.astype(np.int64)
            T, K = int(lv.size), self.K
            L = int(lv.max()) + 1 if T else 1
            sizes, idx = [T], [np.arange(T)]
            for k in range(K):
                s, e = int(self.ep_off_h[k]), int(self.ep_off_h[k + 1])
                sizes.append(e - s)
                idx.append(np.arange(s, e))
            for k in range(K):
                s, e = int(self.ep_off_h[k]), int(self.ep_off_h[k + 1])
                sizes.extend(np.bincount(lv[s:e], minlength=L).tolist())
                idx.append(s + np.argsort(lv[s:e], kind="stable"))
            ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
            dev = self.endpoints.device
            self._segments = (torch.from_numpy(ptr).to(dev), torch.from_numpy(np.concatenate(idx).astype(np.int32)).to(dev), L)
        return self._segments

    @staticmethod
    def concat(batches):
        """One batch of K designs (same image size, same map size), stepped as one by ``DesignStep``: the loss is the
        mean of the designs' losses and every gradient the mean of their gradients (``DesignStep.run``).

        The netlists are joined into one ``TimingGraph`` (pin ids of design k offset by the pins before it), whose
        level schedule is every design's own schedule side by side (caller-supplied topological levels survive);
        features, endpoints (offset), levels and labels are concatenated, the images stacked to (K, C, H, W), and the
        designs' ``MaskRows`` kept as they are.  A batch is dynamic when one of its designs is."""
        batches = list(batches)
        if not batches:
            raise ValueError("DesignBatch.concat: no designs")
        b0 = batches[0]
        for k, b in enumerate(batches[1:], 1):
            for what, a, c in (("image", b0.image.shape, b.image.shape),
                               ("mask width", (b0.width,), (b.width,)),
                               ("cell_feat width", tuple(b0.cell_feat.shape[1:]), tuple(b.cell_feat.shape[1:])),
                               ("net_feat width", tuple(b0.net_feat.shape[1:]), tuple(b.net_feat.shape[1:]))):
                if tuple(a) != tuple(c):
                    raise ValueError(f"DesignBatch.concat: design {k} has {what} {tuple(c)} but design 0 has {tuple(a)}")
            if b.K != 1:
                raise ValueError(f"DesignBatch.concat: design {k} is already a batch of {b.K} designs")
        if b0.K != 1:
            raise ValueError(f"DesignBatch.concat: design 0 is already a batch of {b0.K} designs")
        dev = b0.endpoints.device
        ns = [b.graph.number_of_nodes() for b in batches]
        pin_off = np.concatenate([[0], np.cumsum(ns)]).astype(np.int64)
        scheds = [b.graph.schedule() for b in batches]
        edges = {}
        for et in ("net", "cell"):
            edges[et] = tuple(torch.cat([b.graph._edges[et][i].to(dev) + int(o) for b, o in zip(batches, pin_off)])
                              for i in range(2))
        g = TimingGraph(int(pin_off[-1]), edges["net"], edges["cell"])
        g._edges = edges                                                   # already on the device
        g._levels = (torch.cat([s.level for s in scheds]).contiguous(), max(s.num_levels for s in scheds))
        cell_feat = torch.cat([b.cell_feat for b in batches])
        net_feat = torch.cat([b.net_feat for b in batches])
        g.ndata["cell_feat"], g.ndata["net_feat"] = cell_feat, net_feat
        endpoints = torch.cat([b.endpoints + int(o) for b, o in zip(batches, pin_off)]).to(torch.int32)
        out = DesignBatch(g, None, endpoints, torch.cat([b.endpoint_level for b in batches]),
                          torch.cat([b.arrival_time for b in batches]), torch.stack([b.image for b in batches]),
                          cell_feat=cell_feat, net_feat=net_feat, dynamic=any(b.dynamic for b in batches),
                          mask_rows=[b.mask_rows for b in batches])
        out.pin_off_h = pin_off
        out.ep_off = torch.from_numpy(out.ep_off_h.astype(np.int32)).to(dev)
        if all(b.required is not None for b in batches):
            out.required = torch.cat([b.required for b in batches])
        if all(b.label is not None for b in batches):
            out.label = torch.cat([b.label for b in batches])
        return out

    @staticmethod
    def from_host(h, device, graph=None):
        """Upload a HostDesign.  With ``graph`` (a TimingGraph already on the device, schedule
        cached) only the per-step tensors move: features, endpoints, masks, labels, image."""
        dv = {k: v.to(device, non_blocking=True) for k, v in h.t.items()
              if graph is None or k not in ("net_src", "net_dst", "cell_src", "cell_dst", "pis")}
        if graph is None:
            graph = TimingGraph(h.n, (dv["net_src"], dv["net_dst"]), (dv["cell_src"], dv["cell_dst"]), pis=dv["pis"])
            graph.ndata["cell_feat"], graph.ndata["net_feat"] = dv["cell_feat"], dv["net_feat"]
        mask = MaskCSR(dv["mask_indptr"], dv["mask_cols"], h.map_size * h.map_size)
        return DesignBatch(graph, mask, dv["endpoints"], dv["endpoint_level"], dv["arrival_time"], dv["image"],
                           cell_feat=dv["cell_feat"], net_feat=dv["net_feat"])

    @staticmethod
    def from_synth(d, device):
        return DesignBatch.from_host(HostDesign(d, pin=False), device)


class EvalMetrics:
    """``DesignStep.evaluate``'s metrics: ONE (1 + K + K * L, 9) float32 tensor, columns ``tm_ops.EVAL_COLUMNS``
    ([mse, r2, correct, tp, fn, tn, fp, count, mape]), and views into it.  Under CUDA-graph replay the tensor is
    rewritten in place, and so are the views."""

    def __init__(self, table, K, L):
        self.table, self.K, self.L = table, K, L
        self.batch = table[0]                                    # (9,) the whole batch
        self.design = table[1:1 + K]                             # (K, 9) every design of a joined batch
        self.level = table[1 + K:].view(K, L, table.shape[1])    # (K, L, 9) design k's endpoints on endpoint level l

    def to_host(self):
        """The same views over one device-to-host copy of the table."""
        return EvalMetrics(self.table.cpu(), self.K, self.L)


class PreparedDesign:
    VALUE_FIELDS = ("cell_feat", "net_feat", "image", "arrival_time")

    def __init__(self, step, host, device, graph=None, pool=None, input_grads=False, param_grads=True, evaluate=False):
        _check_evaluate_options(evaluate, input_grads, param_grads)
        self.batch = DesignBatch.from_host(host, device, graph=graph)
        self.static = {"cell_feat": self.batch.cell_feat, "net_feat": self.batch.net_feat,
                       "image": self.batch.image, "arrival_time": self.batch.arrival_time}
        torch.cuda.synchronize()
        if evaluate:
            self.replay = step.capture_evaluate(self.batch, pool=pool)
        else:
            self.replay = step.capture(self.batch, pool=pool, input_grads=input_grads, param_grads=param_grads)

    def upload(self, host, stream=None):
        """Host -> device copy of the per-step values into the graph's static inputs."""
        ctx = torch.cuda.stream(stream) if stream is not None else torch.cuda.stream(torch.cuda.current_stream())
        with ctx:
            for k in self.VALUE_FIELDS:
                self.static[k].copy_(host.t[k], non_blocking=True)

    def nbytes(self):
        return int(sum(t.numel() * t.element_size() for t in self.static.values()))

    def step(self, host=None):
        if host is not None:
            self.upload(host)
        return self.replay()


class PreparedDesigns:
    """``DesignStep.prepare_many``: K resident designs, one captured step over all of them."""

    def __init__(self, step, hosts, device, pool=None, input_grads=False, param_grads=True, evaluate=False):
        _check_evaluate_options(evaluate, input_grads, param_grads)
        self.parts = [DesignBatch.from_host(h, device) for h in hosts]
        self.batch = DesignBatch.concat(self.parts)
        torch.cuda.synchronize()
        if evaluate:
            self.replay = step.capture_evaluate(self.batch, pool=pool)
        else:
            self.replay = step.capture(self.batch, pool=pool, input_grads=input_grads, param_grads=param_grads)

    def upload(self, hosts, stream=None):
        """Host -> device copy of every design's per-step values into its slices of the graph's static inputs."""
        if len(hosts) != len(self.parts):
            raise ValueError(f"PreparedDesigns.upload: {len(hosts)} designs given, {len(self.parts)} prepared")
        b = self.batch
        ctx = torch.cuda.stream(stream) if stream is not None else torch.cuda.stream(torch.cuda.current_stream())
        with ctx:
            for k, h in enumerate(hosts):
                p0, p1 = int(b.pin_off_h[k]), int(b.pin_off_h[k + 1])
                e0, e1 = int(b.ep_off_h[k]), int(b.ep_off_h[k + 1])
                b.cell_feat[p0:p1].copy_(h.t["cell_feat"], non_blocking=True)
                b.net_feat[p0:p1].copy_(h.t["net_feat"], non_blocking=True)
                b.image[k].copy_(h.t["image"], non_blocking=True)
                b.arrival_time[e0:e1].copy_(h.t["arrival_time"], non_blocking=True)

    def step(self, hosts=None):
        if hosts is not None:
            self.upload(hosts)
        return self.replay()


def _check_evaluate_options(evaluate, input_grads, param_grads):
    if evaluate and (input_grads or not param_grads):
        raise ValueError("DesignStep.prepare: evaluate=True is the forward alone; it takes neither input_grads nor "
                         "param_grads=False")


class DesignStep:
    def __init__(self, model, cnn, process_group=None, world_size=1, prune=None):
        """``prune`` (default: environment ``TM_CONE=1``, else off): run the netlist branch on the sub-netlist that can
        reach the batch's endpoints (``tm_graph.ConeGraph``) instead of the whole netlist.  Predictions, loss and every
        gradient are unchanged (``tests/test_gpu_parity.py::test_design_step_on_cone_subnetlist``); pins that no
        endpoint of the batch depends on are simply not evaluated.  Off by default: the headline step evaluates every
        pin, as the reference does."""
        self.model, self.cnn = model, cnn
        self.prune = (os.environ.get("TM_CONE", "0") == "1") if prune is None else bool(prune)
        self.pg, self.world = process_group, world_size
        self.comm_stream = torch.cuda.Stream() if world_size > 1 else None
        # The image branch (U-Net) and the netlist branch (GNN) are independent until the fusion, and
        # both are chains of small latency-bound kernels: they run on two streams, forward and backward.
        self.image_stream = torch.cuda.Stream() if torch.cuda.is_available() else None
        self.overlap = True
        self._buckets = {}            # name -> tm_dp.FlatBucket (persistent flat gradient buffers)
        self._graphs = []             # captured CUDA graphs (released by close())
        g = model.gnn
        sd = dict(g.named_parameters())
        self.gnn_params = [sd[k] for k in tm_ops.GNN_PARAM_NAMES]
        self.cnn_names = [k for k, _ in cnn.named_parameters()]
        self.cnn_params = dict(cnn.named_parameters())
        import model as M
        self.layoutnet = isinstance(cnn, M.LayoutNet)    # else the U-Net (LayoutNet has no BatchNorm statistics)

    # ---------------------------------------------------------------- image branch
    def _image_forward(self, image, need_bwd, update_stats=True):
        if self.layoutnet:
            return tm_unet.layoutnet_forward(self.cnn, image, need_bwd=need_bwd)
        # several designs: each image is normalised with its own statistics, as the reference's batch of one is
        return tm_unet.unet_forward(self.cnn, image, need_bwd=need_bwd, update_stats=update_stats and self.cnn.training,
                                    per_image=True)

    def _image_backward(self, st, gout, need_dx=False, need_wgrad=True):
        if self.layoutnet:
            return tm_unet.layoutnet_backward(self.cnn, st, gout, need_dx=need_dx, need_wgrad=need_wgrad)
        return tm_unet.unet_backward(self.cnn, st, gout, need_dx=need_dx, need_wgrad=need_wgrad)

    @staticmethod
    def _check_feature_map(fmap, b):
        per = fmap.numel() // b.K                        # one feature map per design
        if per * b.K != fmap.numel() or per != b.width:
            raise ValueError(f"the image network's feature map has {per} pixels per design ({tuple(fmap.shape)}) but the "
                             f"path masks are {b.width} columns wide (map_size**2): wrong image size for this CNN")

    # ---------------------------------------------------------------- forward pieces
    def _head_image_side(self, b, feat, X):
        """The head's inputs that do not depend on the propagation: mask fusion of the feature map and the level
        embedding (``mlp_alpha``), written into columns D.. of the head matrix X.  Runs on the image stream."""
        m = self.model
        T = int(b.endpoints.numel())
        width = X.shape[1]
        tab = b.fuse_table() if b.K > 1 else None
        wt = tm_ops.fusion_forward_multi(b.mask_rows_list, tab, b.ep_off, feat, m.fcn.weight.detach(),
                                         m.fcn.bias.detach(), X[:, D:], width)
        a0, a2 = m.mlp_alpha.layers[0], m.mlp_alpha.layers[2]
        lv = b.endpoint_level.reshape(T, 1)
        ha = tm_ops.mlp2_forward(lv, 1, None, T, a0.weight.detach(), a0.bias.detach(), a2.weight.detach(),
                                 a2.bias.detach(), X[:, 2 * D:], width)
        return dict(X=X, wt=wt, ha=ha, lv=lv, width=width, tab=tab)

    def _head_netlist_side(self, H, b, hs, endpoints=None, out=None, hf_out=None):
        """Endpoint rows of H into columns 0..D of X, then ``mlp_fuse`` (into ``out`` when given; its hidden rows into
        ``hf_out`` when given)."""
        m = self.model
        T = int(b.endpoints.numel())
        X, width = hs["X"], hs["width"]
        call("tm_gather_cols", T, D, H, D, b.endpoints if endpoints is None else endpoints, X, width, 0, stream())
        f0, f2 = m.mlp_fuse.layers[0], m.mlp_fuse.layers[2]
        pred = out if out is not None else torch.empty(T, f2.weight.shape[0], dtype=torch.float32, device=H.device)
        hs["hf"] = tm_ops.mlp2_forward(X, width, None, T, f0.weight.detach(), f0.bias.detach(), f2.weight.detach(),
                                       f2.bias.detach(), pred, pred.shape[1], h_out=hf_out)
        return pred

    def _head_forward(self, H, b, feat):
        T = int(b.endpoints.numel())
        X = torch.empty(T, D + D + self.model.global_dim, dtype=torch.float32, device=H.device)
        hs = self._head_image_side(b, feat, X)
        return self._head_netlist_side(H, b, hs), hs

    def forward(self, b):
        """Inference: predictions for the batch's endpoints (validate(), train.py:137-291); for a joined batch, every
        design's predictions one after the other."""
        fmap, _ = self._image_forward(b.image, need_bwd=False)
        self._check_feature_map(fmap, b)
        sched = b.graph.schedule()
        H, _ = tm_ops.gnn_forward(sched, b.cell_feat, b.net_feat,
                                  [p.detach() for p in self.gnn_params], save=False)
        pred, _ = self._head_forward(H, b, fmap.reshape(-1))
        return pred.squeeze(-1)

    def evaluate(self, b):
        """One evaluation step (validate(), train.py:137-291; test.py:124-318): the forward half of ``run``, laid out as
        ``run`` lays it out -- the netlist branch on the current stream with the per-level kernels, the image branch on
        the image stream, the head after the join -- followed by ONE ``tm_eval_metrics`` launch.  Returns ``(pred (T,),
        metrics)``; ``metrics`` is an ``EvalMetrics`` (``.batch``, ``.design``, ``.level``, ``.to_host()``) against the
        batch's labels, with the confusion counts when ``b.required`` / ``b.label`` are set.  Predictions are the same
        bits as ``run(b)``'s.  Nothing of the model is touched except what ``forward`` touches: U-Net batch norm in train
        mode updates its running statistics (the reference validates in train mode under ``no_grad``).  No ``.grad``, no
        parameter, no gradient bucket, no collective.  Joined batches give every design's and every level's row;
        ``prune`` does not apply (the cone of all endpoints is nearly the whole netlist)."""
        m = self.model
        dev = b.image.device
        main = torch.cuda.current_stream()
        if getattr(b, "dynamic", False):
            for r in b.mask_rows_list:
                r.rebuild()
        seg_ptr, seg_idx, L = b.eval_segments()
        side = self.image_stream if (self.overlap and self.image_stream is not None) else main
        side.wait_stream(main)
        sched = b.graph.schedule()
        gp = [p.detach() for p in self.gnn_params]
        T = int(b.endpoints.numel())
        X = torch.empty(T, D + D + m.global_dim, dtype=torch.float32, device=dev)
        H, _ = tm_ops.gnn_forward(sched, b.cell_feat, b.net_feat, gp, save=False,
                                  impl=16 if side is not main and os.environ.get("TM_GNN_IMPL") is None else None)
        img_cap = int(os.environ.get("TM_IMAGE_SM_CAP", "0")) if side is not main else 0
        with torch.cuda.stream(side):
            old_cap = tm_lib.lib().tm_tc_set_grid_cap(img_cap)
            fmap, _ = self._image_forward(b.image, need_bwd=False)
            tm_lib.lib().tm_tc_set_grid_cap(old_cap)
            self._check_feature_map(fmap, b)
            hs = self._head_image_side(b, fmap.reshape(-1), X)
        main.wait_stream(side)
        pred = self._head_netlist_side(H, b, hs).squeeze(-1)
        table = tm_ops.eval_metrics(pred, b.arrival_time, seg_ptr, seg_idx, b.required, b.label)
        # a tensor-core barrier timeout leaves garbage: the whole batch's mse becomes NaN (tm_lib.check_err_flags)
        call("tm_poison_on_error", table, tm_lib.err_flag(dev), stream())
        return pred, EvalMetrics(table, b.K, L)

    def incremental(self, b, what_if_rows=0):
        """An ``IncrementalEvaluation`` of batch ``b``: one full forward now, then re-prediction after feature edits by
        re-propagating only the edited pins' forward cone (see the class).  ``what_if_rows`` (default 0): rows reserved
        for ``what_if`` candidates' cone pins (see ``WhatIf``); 0 allocates nothing extra."""
        return IncrementalEvaluation(self, b, what_if_rows)

    # ---------------------------------------------------------------- full step
    def run(self, b, grad_scale=1.0, input_grads=False, pred_grad=None, param_grads=True):
        """Forward + backward.  Returns (loss (1,) device tensor, pred (T,)); fills ``.grad``.  A batch of K designs
        (``DesignBatch.concat``) gives loss = mean of the designs' MSEs (``b.design_losses``, (K,)) and every gradient
        the mean of their gradients; predictions are per design as the one-design step gives them.

        ``input_grads``: also fill ``b.input_grads`` = {"cell_feat", "net_feat", "image"}, the gradients of what the step
        differentiates with respect to the batch's inputs, shaped like ``b.cell_feat`` / ``b.net_feat`` / ``b.image``
        and rewritten by every run or replay.  Feature rows the propagation never reads (net-class pins in
        "cell_feat", cell-class pins in "net_feat", pins outside the schedule or, with ``prune``, outside the cone) are
        exactly zero.  In a joined batch design k owns the rows ``b.pin_off_h[k]:b.pin_off_h[k + 1]`` and ``image[k]``.
        With several ranks these gradients belong to the rank's own designs and are not all-reduced.
        ``pred_grad``: (T,) float32 device tensor, dObjective/dpred, that seeds the backward instead of the MSE's
        gradient, taken as given (no 1/T or 1/K factor; ``grad_scale`` must stay 1): every ``.grad`` and input gradient
        is then the vector-Jacobian product ``pred.backward(pred_grad)`` gives.  The loss is still computed.  Neither
        option changes the parameter gradients' arithmetic: with ``pred_grad`` unset they are the same bits.
        ``param_grads=False`` (needs ``input_grads``): a step against a frozen predictor, for layout optimisation or
        saliency.  The model is left exactly as it was: no ``.grad`` is touched, no parameter changes, U-Net batch norm
        normalises with the batch's statistics as the training step does but does not update its running statistics
        or ``num_batches_tracked``, and no gradient all-reduce is posted.  No parameter-gradient kernel runs.  Loss,
        predictions and the "net_feat" / "image" input gradients are the same bits as with ``param_grads=True``;
        "cell_feat" comes from a fused data-gradient kernel that sums in another order (fp32-class)."""
        if not param_grads and not input_grads:
            raise ValueError("DesignStep.run: param_grads=False computes input gradients only; pass input_grads=True")
        if pred_grad is not None:
            T = int(b.endpoints.numel())
            if grad_scale != 1.0:
                raise ValueError("DesignStep.run: pred_grad is taken as given; scale the seed instead of grad_scale")
            if (pred_grad.shape != (T,) or pred_grad.dtype != torch.float32 or not pred_grad.is_contiguous()
                    or pred_grad.device != b.endpoints.device):
                raise ValueError(f"DesignStep.run: pred_grad must be a contiguous float32 ({T},) tensor on "
                                 f"{b.endpoints.device}, got {pred_grad.dtype} {tuple(pred_grad.shape)} on {pred_grad.device}")
        m = self.model
        dev = b.image.device
        main = torch.cuda.current_stream()
        if getattr(b, "dynamic", False):
            for r in b.mask_rows_list:                       # this batch's mask-row selection (7 small kernels, no host sync)
                r.rebuild()
        side = self.image_stream if (self.overlap and self.image_stream is not None) else main
        side.wait_stream(main)                               # fork: inputs / parameters are ready on `main`
        # the netlist branch runs on the sub-netlist that can reach this batch's endpoints (tm_graph.ConeGraph)
        cone = b.cone() if self.prune else None
        sched = (cone.graph if cone is not None else b.graph).schedule()
        endpoints = cone.endpoints if cone is not None else b.endpoints
        x_rows = (cone.cell_x_rows, cone.net_x_rows) if cone is not None else None
        gp = [p.detach() for p in self.gnn_params]
        # the longer chain is enqueued first so the host's launch time for the other one overlaps it
        # (per-level kernels while the image stream runs next to them: measured 5.07 ms/step against 5.49 ms
        #  with the persistent forward, which owns all SMs for 0.9 ms and serialises the U-Net behind it)
        T = int(b.endpoints.numel())
        X = torch.empty(T, D + D + m.global_dim, dtype=torch.float32, device=dev)     # head input [H rows | fused map | level]
        G = torch.empty(sched.n, D, dtype=torch.float32, device=dev)                 # dLoss/dH, seeded at the endpoints
        H, saved = tm_ops.gnn_forward(sched, b.cell_feat, b.net_feat, gp, save=True, x_rows=x_rows,
                                      impl=16 if side is not main and os.environ.get("TM_GNN_IMPL") is None else None)
        img_cap = int(os.environ.get("TM_IMAGE_SM_CAP", "0")) if side is not main else 0
        with torch.cuda.stream(side):
            old_cap = tm_lib.lib().tm_tc_set_grid_cap(img_cap)
            fmap, ust = self._image_forward(b.image, need_bwd=True, update_stats=param_grads)
            tm_lib.lib().tm_tc_set_grid_cap(old_cap)
            self._check_feature_map(fmap, b)
            feat = fmap.reshape(-1)
            # everything of the head that does not read H runs here, off the netlist branch's critical path
            # (the image stream is idle long before the 101 levels finish): mask fusion, level embedding, G = 0
            hs = self._head_image_side(b, feat, X)
            G.zero_()
        main.wait_stream(side)                               # join: the head needs the fused feature map
        pred = self._head_netlist_side(H, b, hs, endpoints)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        gpred = torch.empty(T, 1, dtype=torch.float32, device=dev)
        if b.K == 1:
            call("tm_mse", T, pred, b.arrival_time, loss, gpred, float(grad_scale), stream())
        else:                                                # mean over designs: each design's gradient scaled by 1/K
            b.design_losses = torch.empty(b.K, dtype=torch.float32, device=dev)
            call("tm_mse_multi", b.K, b.ep_off, pred, b.arrival_time, b.design_losses, loss, gpred, float(grad_scale),
                 stream())
        if pred_grad is not None:
            gpred = pred_grad.reshape(T, 1)

        # ---- head backward: mlp_fuse on the netlist stream (its dX seeds the backward sweep) ...
        width = hs["width"]
        f0, f2 = m.mlp_fuse.layers[0], m.mlp_fuse.layers[2]
        dw1, db1, dw2, db2, dX = tm_ops.mlp2_backward(X, width, None, T, f0.weight.detach(), f2.weight.detach(),
                                                      hs["hf"], gpred, 1, need_dx=True,
                                                      wgrad_stream=side if side is not main else None,
                                                      need_wgrad=param_grads)
        side.wait_stream(main)                               # dX is ready
        # ... the level embedding and the mask fusion (whose dF starts the U-Net backward) on the image stream
        a0, a2 = m.mlp_alpha.layers[0], m.mlp_alpha.layers[2]
        with torch.cuda.stream(side):
            # (a frozen step: the level embedding's input has no gradient, so mlp_alpha has no backward at all)
            if param_grads:
                da1, dab1, da2, dab2, _ = tm_ops.mlp2_backward(hs["lv"], 1, None, T, a0.weight.detach(),
                                                               a2.weight.detach(), hs["ha"], dX[:, 2 * D:], width,
                                                               b1=a0.bias.detach())
            dF, dfw, dfb = tm_ops.fusion_backward_multi(b.mask_rows_list, hs["tab"], b.ep_off, feat, hs["wt"],
                                                        dX[:, D:], width, need_wgrad=param_grads)
            if param_grads:
                head = [(f0.weight, dw1), (f0.bias, db1), (f2.weight, dw2), (f2.bias, db2), (a0.weight, da1),
                        (a0.bias, dab1), (a2.weight, da2), (a2.bias, dab2), (m.fcn.weight, dfw), (m.fcn.bias, dfb)]
                self._assign(head)
                self._post_allreduce("head", [p for p, _ in head])

        # ---- GNN backward (main stream) next to the U-Net backward (image stream)
        call("tm_scatter_add_cols", T, D, dX, width, 0, endpoints, G, D, stream())
        if input_grads:
            ggrads, dcf, dnf = tm_ops.gnn_backward(sched, saved, gp, G, need_dx=True, need_wgrad=param_grads)
        else:
            ggrads = tm_ops.gnn_backward(sched, saved, gp, G)
        pairs = list(zip(self.gnn_params, ggrads)) if param_grads else []
        self._assign(pairs)
        with torch.cuda.stream(side):
            old_cap = tm_lib.lib().tm_tc_set_grid_cap(img_cap)
            ug = self._image_backward(ust, dF.reshape(fmap.shape), need_dx=input_grads, need_wgrad=param_grads)
            tm_lib.lib().tm_tc_set_grid_cap(old_cap)
            if input_grads:
                ug, dimg = ug
                b.input_grads = {"cell_feat": dcf, "net_feat": dnf, "image": dimg}
            upairs = [(self.cnn_params[k], ug[k]) for k in self.cnn_names] if param_grads else []
            self._assign(upairs)
        main.wait_stream(side)                               # join: every gradient exists on `main`
        if param_grads:
            # The GNN and U-Net gradients go out as ONE exchange after the join (2.5 MB): posted separately they were
            # two latency-bound all-reduces queued behind each other on the communication stream at the very end of
            # the step (the U-Net's could not start before the GNN's, which waits for the last weight-gradient kernel)
            self._post_allreduce("tail", [p for p, _ in pairs] + [p for p, _ in upairs])
            self._wait_allreduce()
        # a tensor-core kernel whose barrier timed out leaves garbage: the step's loss becomes NaN (loud in any
        # training loop, also under graph replay); tm_lib.check_err_flags() names the cause on the host
        call("tm_poison_on_error", loss, tm_lib.err_flag(dev), stream())
        return loss, pred.squeeze(-1)

    # ---------------------------------------------------------------- CUDA graph
    def capture(self, b, warmup=2, pool=None, input_grads=False, pred_grad=None, param_grads=True):
        """Capture ``run(b, input_grads=input_grads, pred_grad=pred_grad)`` (about 500 launches on two streams) into
        one CUDA graph.  The batch's tensors -- and ``pred_grad`` -- become the graph's static inputs: refresh them in
        place (``tensor.copy_``) and call the returned function, which replays the graph and returns the same (loss,
        pred) tensors; ``param.grad`` tensors and ``b.input_grads`` are rewritten in place by every replay.  On the data-parallel path the
        bucketed NCCL all-reduces (head + fusion early, GNN + U-Net after the join) are captured INSIDE the graph (persistent flat buffers,
        ``tm_dp.FlatBucket``), where they overlap the backward as in the eager schedule; with
        ``TM_DP_GRAPH=0`` the graph holds the rank's compute only and one exchange is posted after each
        replay.  ``pool``: a ``torch.cuda.graph_pool_handle()`` shared by graphs that are replayed one
        after the other (several prepared designs of one rank share their activation memory).
        ``param_grads=False``: a frozen step (see ``run``); the replay leaves every ``.grad`` alone and posts nothing.
        Call ``close()`` before ``torch.distributed.destroy_process_group()``."""
        if not param_grads and not input_grads:
            raise ValueError("DesignStep.capture: param_grads=False computes input gradients only; pass input_grads=True")
        opts = dict(input_grads=input_grads, pred_grad=pred_grad, param_grads=param_grads)

        def rebind():
            grads = [(p, p.grad) for p in list(self.model.parameters()) + list(self.cnn.parameters())
                     if p.grad is not None] if param_grads else []
            igrads = b.input_grads if input_grads else None

            def after_replay():
                for p, gr in grads:                      # several captured steps may coexist: re-point .grad
                    p.grad = gr
                if igrads is not None:
                    b.input_grads = igrads
            return after_replay

        def fn():
            return self.run(b, **opts)
        if self.world <= 1 or not param_grads or os.environ.get("TM_DP_GRAPH", "1") != "0":
            return self._capture_local(fn, warmup, pool, rebind)
        world, self.world = self.world, 1                  # no collectives inside the captured region
        try:
            replay_local = self._capture_local(fn, warmup, pool, rebind)
        finally:
            self.world = world
        params = [p for p in list(self.model.parameters()) + list(self.cnn.parameters())]

        def replay():
            out = replay_local()
            self._post_allreduce("all", [p for p in params if p.grad is not None])
            self._wait_allreduce()
            return out
        replay.graph = replay_local.graph
        return replay

    def capture_evaluate(self, b, warmup=2, pool=None):
        """Capture ``evaluate(b)`` into one CUDA graph.  Returns ``replay() -> (pred, metrics)``: the same tensors on every
        replay, rewritten in place; refresh the batch's values (features, image, labels) in place in between.  The
        metric rows follow the endpoint levels the batch had when this was called (``DesignBatch.eval_segments``), so a
        dynamic batch, whose endpoints change between replays, is refused.  ``pool``: as in ``capture``."""
        if getattr(b, "dynamic", False):
            raise ValueError("DesignStep.capture_evaluate: a dynamic batch changes its endpoints between replays; "
                             "evaluate a fixed endpoint set")
        b.eval_segments()                                  # host work: before the capture
        return self._capture_local(lambda: self.evaluate(b), warmup, pool)

    def _capture_local(self, fn, warmup=2, pool=None, rebind=None):
        """Capture ``fn()`` (warmed up ``warmup`` times on a side stream) into one CUDA graph; returns ``replay()``, which
        replays it and returns what ``fn`` returned at capture.  ``rebind``: called once after the capture, it returns a
        function that runs after every replay (re-pointing state the capture left, such as ``.grad``)."""
        cur = torch.cuda.current_stream()
        s = torch.cuda.Stream(priority=int(os.environ.get("TM_MAIN_PRIORITY", "0")))   # (a higher priority for the netlist branch was measured: no effect)
        s.wait_stream(cur)
        with torch.cuda.stream(s):
            for _ in range(warmup):
                fn()
        cur.wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, pool=pool):
            out = fn()
        self._graphs.append(g)
        after_replay = rebind() if rebind is not None else None

        def replay():
            g.replay()
            if after_replay is not None:
                after_replay()
            return out
        replay.graph = g
        return replay

    def prepare(self, host, device, graph=None, pool=None, input_grads=False, param_grads=True, evaluate=False):
        """A design made resident for repeated steps: uploads everything once, builds the structure
        that depends only on the netlist and the endpoint batch (level schedule, CSRs, mask runs / CSC)
        and captures the step as a CUDA graph.  Returns a ``PreparedDesign``; its ``step(host)``
        refreshes the per-step VALUES (features, image, labels) from pinned host memory and replays.
        The structure (edges, endpoints, masks) must be the one given here.  ``input_grads``: every replay also
        rewrites ``batch.input_grads`` (see ``run``); ``param_grads=False``: a frozen step (see ``run``).
        ``evaluate=True``: the captured step is ``evaluate`` (``capture_evaluate``) and ``step(host)`` returns ``(pred,
        metrics)``; it takes neither ``input_grads`` nor ``param_grads=False`` (ValueError)."""
        return PreparedDesign(self, host, device, graph, pool, input_grads, param_grads, evaluate)

    def prepare_many(self, hosts, device, pool=None, input_grads=False, param_grads=True, evaluate=False):
        """K designs made resident for repeated steps over all of them (``DesignBatch.concat``), captured as ONE CUDA
        graph.  Returns a ``PreparedDesigns``; its ``step(hosts)`` refreshes the per-step VALUES of all K from pinned
        host memory and replays.  The structures must be the ones given here.  ``input_grads``, ``param_grads``,
        ``evaluate``: as in ``prepare``."""
        return PreparedDesigns(self, hosts, device, pool, input_grads, param_grads, evaluate)

    @staticmethod
    def _assign(pairs):
        for p, g in pairs:
            p.grad = g.reshape(p.shape)

    # ---------------------------------------------------------------- data parallel
    def _post_allreduce(self, name, params):
        if self.world <= 1:
            return
        bucket = self._buckets.get(name)
        if bucket is None:
            bucket = self._buckets[name] = tm_dp.FlatBucket(params, self.world, self.pg)
        bucket.post(self.comm_stream)

    def _wait_allreduce(self):
        if self.world > 1 and self.comm_stream is not None:
            torch.cuda.current_stream().wait_stream(self.comm_stream)

    def close(self):
        """Release the captured graphs (they hold NCCL kernels of this step's communicator): call before
        ``torch.distributed.destroy_process_group()``."""
        torch.cuda.synchronize()
        for g in self._graphs:
            g.reset()
        self._graphs = []
        torch.cuda.synchronize()

    def adam_step(self, state, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """Fused Adam over every parameter that has a gradient (train.py:431-435,555): ONE launch for all ~70
        tensors (``tm_adam_multi``).  The pointer / chunk tables live on the device and are rebuilt only when a
        ``.grad`` tensor moved (never under CUDA-graph replay, where gradients are rewritten in place)."""
        import numpy as np
        state["step"] = state.get("step", 0) + 1
        ps = [p for p in list(self.model.parameters()) + list(self.cnn.parameters()) if p.grad is not None]
        if not ps:
            return
        for p in ps:
            if id(p) not in state:
                state[id(p)] = (torch.zeros_like(p), torch.zeros_like(p))
            if not p.grad.is_contiguous():
                p.grad = p.grad.contiguous()
        key = tuple((p.data_ptr(), p.grad.data_ptr()) for p in ps)
        tab = state.get("_table")
        if tab is None or tab[0] != key:
            chunk = int(tm_lib.lib().tm_adam_chunk())
            rows = np.zeros((len(ps), 5), dtype=np.int64)
            ct, co = [], []
            for i, p in enumerate(ps):
                m, v = state[id(p)]
                rows[i] = (p.data_ptr(), p.grad.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel())
                for off in range(0, p.numel(), chunk):
                    ct.append(i)
                    co.append(off)
            dev = ps[0].device
            tab = state["_table"] = (key, torch.from_numpy(rows).to(dev), torch.tensor(ct, dtype=torch.int32, device=dev),
                                     torch.tensor(co, dtype=torch.int32, device=dev))
        call("tm_adam_multi", int(tab[2].numel()), tab[1], tab[2], tab[3], lr, betas[0], betas[1], eps, weight_decay,
             state["step"], 1.0, stream())


class IncrementalEvaluation:
    """Re-prediction of one batch after edits of its pin features, re-propagating only the edited pins' forward cone
    (``DesignStep.incremental(batch)``)::

        inc = step.incremental(batch)        # one full forward; keeps H, S and the head's image-side columns
        batch.cell_feat[pins] = new_rows     # edit cell_feat and / or net_feat rows in place
        pred = inc.update(pins)              # S rows of `pins`, cone build, cone propagation, head netlist side
        replay = inc.capture_update(pins)    # one CUDA graph for a fixed pin set: edit rows in place, replay() -> pred
        inc.refresh()                        # full recompute, after a parameter or image change
        inc.cone_size()                      # pins re-propagated by the last update (one device read)
        g = inc.input_grads(seed)            # d(seed . pred)/d features through the seeded endpoints' fan-in cone

    Predictions: ``pred`` (T,) and ``H`` (n, 128) are rewritten in place.  After any sequence of updates they are the
    same bits as ``step.forward(batch)`` and ``tm_ops.gnn_forward`` on the persistent back end over the edited
    features; against ``evaluate`` / ``run``, which propagate with the per-level kernels, they agree to fp32 class, as
    ``forward`` does.  The baseline and every update run the persistent forward, whatever ``tm_gnn_set_impl`` /
    ``TM_GNN_IMPL`` say.  The head's netlist side (endpoint gather + ``mlp_fuse`` over all T endpoints) reruns in
    full: the same launches as ``forward``'s head.

    The image branch runs once, in the constructor and in ``refresh()``; neither updates batch-norm running
    statistics.  Nothing touches a ``.grad``, a parameter or a buffer, and no collective runs.  The state holds the
    result of the weights and the image as they were at construction (or at the last ``refresh()``): call
    ``refresh()`` after changing either -- this is documented, not detected (an in-place optimiser step such as
    ``DesignStep.adam_step`` does not bump a tensor's version counter).

    Pins: a host sequence (list, ndarray or CPU tensor) of pin ids of the batch's netlist; for a joined batch
    (``DesignBatch.concat``) joined ids, design k owning ``pin_off_h[k]:pin_off_h[k + 1]``.  Duplicates are dropped;
    pins outside the schedule are accepted and change nothing; an empty list launches nothing; ids out of range or not
    integers raise ``ValueError``.  A dynamic batch raises ``ValueError``.  Memory: H and S (2 x n x 512 bytes, about
    340 MB for a 331 819-pin design) plus cone buffers the size of the schedule.

    ``what_if_rows=R`` > 0 makes ``H`` / ``S`` the first n rows of (n + R + 1)-row buffers, whose rows n.. hold the
    cone pins of ``what_if`` candidates (see ``WhatIf``): R x 1 KB more.  ``generation`` counts the changes of the
    base state (``update``, a replayed ``capture_update``, ``refresh``, ``WhatIf.commit``)."""

    def __init__(self, step, b, what_if_rows=0):
        if getattr(b, "dynamic", False):
            raise ValueError("DesignStep.incremental: a dynamic batch changes its endpoints between steps; "
                             "incremental evaluation needs a fixed endpoint set")
        if isinstance(what_if_rows, bool) or not isinstance(what_if_rows, (int, np.integer)) or what_if_rows < 0:
            raise ValueError(f"DesignStep.incremental: what_if_rows must be a non-negative integer, got {what_if_rows!r}")
        self.step, self.b = step, b
        sched = self.sched = b.graph.schedule()
        dev = b.image.device
        self.n = sched.n
        self.R = int(what_if_rows)
        if self.n + self.R + 1 >= 2 ** 31:
            raise ValueError(f"DesignStep.incremental: what_if_rows={self.R} exceeds the int32 row range")
        self._level = sched.level.cpu().numpy()          # host copy: splits edited pins into cell / net class
        T = int(b.endpoints.numel())
        if self.R:
            # rows n .. n+R-1: what-if candidates' virtual rows; row n+R: the sink of rows that are not admitted
            self.S_ext = torch.empty(self.n + self.R + 1, D, dtype=torch.float32, device=dev)
            self.H_ext = torch.zeros(self.n + self.R + 1, D, dtype=torch.float32, device=dev)
            self.S, self.H = self.S_ext[:self.n], self.H_ext[:self.n]
        else:
            self.S = torch.empty(self.n, D, dtype=torch.float32, device=dev)
            self.H = torch.zeros(self.n, D, dtype=torch.float32, device=dev)
        self.generation = 0
        self._overlay = None                              # the WhatIf whose candidates the rows n.. hold
        self._max_in_degree = None
        self.X = torch.empty(T, D + D + step.model.global_dim, dtype=torch.float32, device=dev)
        f0, f2 = step.model.mlp_fuse.layers[0], step.model.mlp_fuse.layers[2]
        self._pred2 = torch.empty(T, f2.weight.shape[0], dtype=torch.float32, device=dev)
        # the head's hidden rows live as long as inc: captured updates and gradients read and write this one buffer
        self._hf = torch.empty(T, f0.weight.shape[0], dtype=torch.float32, device=dev)
        self.pred = self._pred2.squeeze(-1)
        self.cone = ForwardCone(b.graph)
        self._last = None                                 # None: full pass; 0: empty update; "cone": the cone's count
        self._grad = None                                 # input_grads' cone, scratch and results (first call)
        self.refresh()

    def _params(self):
        return [p.detach() for p in self.step.gnn_params]

    def refresh(self):
        """Full recompute of the image side, S, H and pred (in place), from the current parameters, image and
        features.  Returns ``pred``."""
        st, b, sched = self.step, self.b, self.sched
        gp = self._params()
        fmap, _ = st._image_forward(b.image, need_bwd=False, update_stats=False)
        st._check_feature_map(fmap, b)
        self._hs = st._head_image_side(b, fmap.reshape(-1), self.X)
        tm_ops.gnn_self_terms(self.S, b.cell_feat, b.net_feat, gp, sched.cell_class, sched.net_class)
        self.H.zero_()
        tm_ops.gnn_forward_cone(sched, self.H, self.S, gp)
        st._head_netlist_side(self.H, b, self._hs, out=self._pred2, hf_out=self._hf)
        self._last = None
        self.generation += 1
        return self.pred

    def _distinct(self, pins):
        """-> int64 ndarray of the distinct pin ids (sorted), validated; empty for an empty sequence."""
        if torch.is_tensor(pins):
            if pins.device.type != "cpu":
                raise ValueError("IncrementalEvaluation: pins must be a host sequence (list, ndarray or CPU tensor)")
            pins = pins.numpy()
        arr = np.asarray(pins)
        if arr.size == 0:
            return np.zeros(0, np.int64)
        if not np.issubdtype(arr.dtype, np.integer):
            raise ValueError(f"IncrementalEvaluation: pin ids must be integers, got {arr.dtype}")
        arr = np.unique(arr.reshape(-1).astype(np.int64))
        if arr[0] < 0 or arr[-1] >= self.n:
            raise ValueError(f"IncrementalEvaluation: pin ids must lie in [0, {self.n}), got {arr[0]} .. {arr[-1]}")
        return arr

    def _pins(self, pins):
        """-> (device int32 [cell-class pins, net-class pins], n cell, n net) of the distinct scheduled pins, or None."""
        arr = self._distinct(pins)
        if arr.size == 0:
            return None
        lv = self._level[arr]
        cell, net = arr[(lv >= 0) & (lv % 2 == 0)], arr[(lv >= 0) & (lv % 2 == 1)]
        if cell.size + net.size == 0:
            return None
        idx = torch.from_numpy(np.concatenate([cell, net]).astype(np.int32)).to(self.H.device)
        return idx, int(cell.size), int(net.size)

    def _launch(self, sel):
        idx, nc, nn_ = sel
        gp = self._params()
        tm_ops.gnn_self_terms(self.S, self.b.cell_feat, self.b.net_feat, gp, idx[:nc], idx[nc:])
        self.cone.build(idx)
        tm_ops.gnn_forward_cone(self.cone, self.H, self.S, gp)
        self.step._head_netlist_side(self.H, self.b, self._hs, out=self._pred2, hf_out=self._hf)
        return self.pred

    def update(self, pins):
        """Re-predict after the feature rows of ``pins`` were edited in place.  Returns ``pred`` (rewritten in place)."""
        sel = self._pins(pins)
        self.generation += 1
        if sel is None:
            self._last = 0
            return self.pred
        self._launch(sel)
        self._last = "cone"
        return self.pred

    def capture_update(self, pins, pool=None):
        """``update(pins)`` captured as one CUDA graph for this fixed pin set (run once eagerly first).  Returns
        ``replay() -> pred``: edit the pins' feature rows in place, then replay.  Several captures coexist (they share
        the cone buffers and are replayed one after the other on the stream)."""
        sel = self._pins(pins)
        if sel is None:
            def replay_empty():
                self._last = 0
                self.generation += 1
                return self.pred
            return replay_empty
        inner = self.step._capture_local(lambda: self._launch(sel), warmup=1, pool=pool)
        self.generation += 1                             # the warm-up ran an update

        def replay():
            inner()
            self._last = "cone"
            self.generation += 1
            return self.pred
        replay.graph = inner.graph
        replay.pins = sel[0]            # the graph reads this device pin list: it lives as long as the replay
        return replay

    def cone_size(self):
        """Pins re-propagated by the last update: the schedule's size after a full pass, 0 after an empty update, else
        the cone's pin count (one device read)."""
        if self._last is None:
            return self.sched.n_sched
        if self._last == 0:
            return 0
        if isinstance(self._last, tuple):                # ("what_if", wi, k): a committed candidate
            return int(self._last[1].cone_sizes()[self._last[2]])
        return self.cone.size()

    # ---------------------------------------------------------------- input gradients
    def _check_seed(self, seed, what):
        T, dev = int(self.b.endpoints.numel()), self.b.endpoints.device
        if (not torch.is_tensor(seed) or seed.shape != (T,) or seed.dtype != torch.float32 or not seed.is_contiguous()
                or seed.device != dev):
            got = (f"{seed.dtype} {tuple(seed.shape)} on {seed.device}" if torch.is_tensor(seed) else type(seed).__name__)
            raise ValueError(f"IncrementalEvaluation.{what}: seed must be a contiguous float32 ({T},) tensor on {dev}, "
                             f"got {got}")

    def _grad_state(self):
        if self._grad is None:
            b, dev = self.b, self.H.device
            self._grad = dict(cone=FaninCone(b.graph), G=torch.empty(self.n, D, dtype=torch.float32, device=dev),
                              scratch=tm_ops.gnn_cone_scratch(self.sched, dev),
                              out={"cell_feat": torch.empty(b.cell_feat.shape, dtype=torch.float32, device=dev),
                                   "net_feat": torch.empty(b.net_feat.shape, dtype=torch.float32, device=dev)})
        return self._grad

    def _grad_launch(self, seed, mark=None):
        gs, b, st = self._grad_state(), self.b, self.step
        T, width = int(b.endpoints.numel()), self.X.shape[1]
        cone, G, out = gs["cone"], gs["G"], gs["out"]
        cone.build(b.endpoints, seed)
        if mark:
            mark("cone")
        f0, f2 = st.model.mlp_fuse.layers[0], st.model.mlp_fuse.layers[2]
        dX = tm_ops.mlp2_backward(self.X, width, None, T, f0.weight.detach(), f2.weight.detach(), self._hf,
                                  seed.reshape(T, 1), 1, need_dx=True, need_wgrad=False)[4]
        if mark:
            mark("head")
        # all of G is zeroed (one memset) rather than the cone's rows: the cone's size is known only on the device
        G.zero_()
        call("tm_scatter_add_cols", T, D, dX, width, 0, b.endpoints, G, D, stream())
        out["cell_feat"].zero_()
        out["net_feat"].zero_()
        if mark:
            mark("zero_scatter")
        tm_ops.gnn_backward_cone(cone, self.H, G, self._params(), b.cell_feat, b.net_feat, out["cell_feat"],
                                 out["net_feat"], gs["scratch"], mark=mark)
        return out

    def input_grads(self, seed):
        """The gradient of ``sum_t seed[t] * pred[t]`` with respect to the batch's ``cell_feat`` and ``net_feat`` at the
        current state (after every ``update``, replayed ``capture_update`` and ``WhatIf.commit``), backpropagated
        through only the fan-in cone of the endpoints whose seed is non-zero.  ``seed``: contiguous float32 (T,) on the
        batch's device, dObjective/dpred, taken as given as ``run(..., pred_grad=seed)`` takes it.  Returns the dict
        {"cell_feat", "net_feat"}, shaped like the features and rewritten by every call.  Rows outside the cone are
        exactly zero, and so are the rows the propagation never reads (net-class pins in "cell_feat", cell-class pins in
        "net_feat", unscheduled pins), as in ``batch.input_grads``.

        There is no image gradient: the image branch is frozen inside this object (use the frozen step,
        ``step.run(batch, input_grads=True, pred_grad=seed, param_grads=False)``, for it).  Device work only, no host
        synchronisation: the head's data gradient over the T endpoints (``mlp_fuse`` from X and its hidden rows), the
        cone build (``tm_fanin_cone``), A / LSE / HID of the cone's cell pins recomputed from ``H``, the persistent
        backward sweep over the cone, and the self-MLP data gradients of the cone's pins.  The rows are the same bits
        as the persistent full backward's (``tm_ops.gnn_backward(..., need_dx=True, need_wgrad=False)`` after
        ``gnn_forward`` on the persistent back end).  Nothing the committed state owns is written (``H``, ``S``,
        ``pred``, ``X``, the batch, what-if rows, parameters, buffers, ``.grad``), no collective runs and
        ``generation`` is unchanged.  Needs the tf32x3 arithmetic (``TM_MATH``), whose self-MLP kernels take a device
        row count.  Memory, on the first call: G (n x 512 bytes), four buffers per cell row (2.5 KB; the fc_cell_self
        hidden rows reuse one of them), the cone's buffers (the size of the schedule) and the two results."""
        self._check_seed(seed, "input_grads")
        return self._grad_launch(seed)

    def capture_input_grads(self, seed, pool=None):
        """``input_grads(seed)`` captured as one CUDA graph (run once eagerly first), with ``seed`` a static input.
        Returns ``replay() -> {"cell_feat", "net_feat"}``: edit ``seed`` in place -- other endpoints may be seeded,
        the cone is rebuilt on the device -- and the features / updates as usual, then replay."""
        self._check_seed(seed, "capture_input_grads")
        self._grad_state()              # allocated outside the graph's pool
        inner = self.step._capture_local(lambda: self._grad_launch(seed), warmup=1, pool=pool)

        def replay():
            inner()
            return self._grad["out"]
        replay.graph = inner.graph
        replay.seed = seed              # the graph reads this tensor: it lives as long as the replay
        return replay

    def grad_cone_size(self):
        """Pins of the last ``input_grads`` cone (one device read, diagnostics); 0 before the first call."""
        return self._grad["cone"].size() if self._grad is not None else 0

    def what_if(self, pin_sets, endpoints=None):
        """A ``WhatIf`` over the candidate edits ``pin_sets`` (a sequence of K pin sequences, validated as ``update``
        validates its pins).  ``endpoints``: a host sequence of endpoint positions (indices into ``pred``) to predict
        only those, propagating each candidate through only the pins that reach them; None predicts all T.  Needs
        ``what_if_rows`` > 0 at construction."""
        return WhatIf(self, pin_sets, endpoints)

    def max_in_degree(self):
        """The largest in-edge count of a scheduled pin (one device read, cached)."""
        if self._max_in_degree is None:
            fp = self.sched.f_ptr
            self._max_in_degree = int((fp[1:] - fp[:-1]).max()) if self.sched.n_sched else 0
        return self._max_in_degree


class WhatIf:
    """Score K alternative feature edits of one design in one call, without changing it
    (``IncrementalEvaluation.what_if(pin_sets)``)::

        inc = step.incremental(batch, what_if_rows=R)
        wi = inc.what_if(pin_sets)           # K host pin lists (joined ids for a joined batch)
        wi.cell_feat, wi.net_feat            # (P, 36) / (P, 2) candidate rows, from the batch's rows at creation
        wi.rows(k)                           # (pins, cell_feat, net_feat) of candidate k: views into the two above
        pred = wi.run()                      # (K, T): row k = the predictions with candidate k's rows alone
        replay = wi.capture()                # one CUDA graph: edit wi.cell_feat / net_feat in place, replay() -> (K, T)
        wi.commit(k)                         # apply candidate k to the batch and the incremental state
        wi.fitted(), wi.cone_sizes()         # (K,) admitted / cone pins (one device read each)

    Row k of ``run()`` is the same bits as ``step.forward(batch)`` with candidate k's rows written into the batch (and
    no other candidate's), i.e. as ``inc.pred`` after writing them and ``inc.update(pins)``.  Each candidate's cone
    pins propagate in private virtual rows n.. of ``inc``'s extended H / S (``tm_forward_cones``): one cone build of
    three launches, the edited pins' self terms, ONE persistent propagation over the joined cone levels, and the head
    over K x T rows, whose image-side columns are read from ``inc`` at run time.  Nothing the committed state owns is
    written: ``inc.H``, ``inc.S``, ``inc.pred``, the batch's features, parameters, buffers and ``.grad``.  So a
    ``WhatIf`` stays valid across ``inc.update`` / ``refresh`` / ``commit`` and always predicts against the current base.

    Pin sets: duplicates are dropped, pins outside the schedule are accepted and change nothing, an empty set predicts
    the base (cone 0), bad ids raise ``ValueError``; a pin may be in several sets, each with its own rows.  Capacity:
    candidates are admitted in index order while their cone pins fit in ``what_if_rows`` and their cone in-edges in
    ``what_if_rows`` x the schedule's largest in-degree; from the first that does not fit on, a candidate's row of the
    result is NaN and ``fitted()`` False.  Memory beyond ``inc``'s rows: two n/8-byte bitmaps per candidate, the joined
    schedule's arrays (sized by ``what_if_rows``), and the (K x T, 288) head matrix.

    ``commit(k)`` propagates nothing: it copies candidate k's virtual H / S rows back to their pins and its feature rows
    into the batch, then reruns the head over the committed H (``inc.pred`` gets candidate k's predictions, the same
    bits, and ``inc.X`` / the head's hidden rows follow) -- the state ``inc.update`` leaves.  It raises ``ValueError``
    when the base changed since this object's last run / replay, when another ``WhatIf`` of ``inc`` ran since, or when
    candidate k was not admitted.

    ``inc.what_if(pin_sets, endpoints=E)`` predicts only the endpoint positions E (indices into ``inc.pred``, joined
    positions for a joined batch; validated as pins are, against [0, T), and kept sorted in ``endpoints``).  Only pins
    from which an endpoint of E is reachable -- E's fan-in cone R(E), built once here (``within_size()``) -- can change
    an H row E reads, so each candidate propagates through its forward cone intersected with R(E)
    (``tm_forward_cones_within``), and the head runs over K x T_E rows.  ``run()`` / ``capture()`` return (K, T_E):
    row k is the same bits as ``step.forward`` with candidate k's rows alone at ``endpoints``, and as the unrestricted
    ``run()[k, endpoints]``.  A candidate's pins outside R(E) change nothing (an all-outside candidate has cone 0 and
    predicts the base), and admission counts restricted cones, so many more candidates fit in ``what_if_rows``.  Memory
    beyond the unrestricted form's: R(E)'s sub-schedule (the size of the schedule) and its n/8-byte bitmap.
    ``commit(k)`` of a restricted ``WhatIf`` has the same preconditions and errors, but the rest of candidate k's cone
    was never computed: it writes candidate k's feature rows into the batch and runs ``inc.update`` over its pins, so it
    propagates, and leaves exactly the state ``update`` leaves (``H``, ``S``, ``pred``, the batch, ``generation``,
    ``cone_size()``)."""

    def __init__(self, inc, pin_sets, endpoints=None):
        if inc.R == 0:
            raise ValueError("IncrementalEvaluation.what_if: built with what_if_rows=0; pass what_if_rows > 0 to "
                             "DesignStep.incremental")
        if torch.is_tensor(pin_sets) or isinstance(pin_sets, (str, bytes)):
            raise ValueError("IncrementalEvaluation.what_if: pin_sets must be a sequence of pin sequences")
        sets = [inc._distinct(p) for p in pin_sets]
        if not sets:
            raise ValueError("IncrementalEvaluation.what_if: no candidate")
        self.inc, b = inc, inc.b
        dev = inc.H.device
        K, T_all = len(sets), int(b.endpoints.numel())
        self.endpoints = None if endpoints is None else self._positions(endpoints, T_all)
        T = T_all if self.endpoints is None else int(self.endpoints.size)
        self.K, self.T = K, T
        self._off = np.concatenate([[0], np.cumsum([s.size for s in sets])]).astype(np.int64)
        self._pins = np.concatenate(sets).astype(np.int64)
        P = int(self._off[-1])
        idx = torch.from_numpy(self._pins).to(dev)
        self._pin_idx = idx
        self.cell_feat = b.cell_feat.index_select(0, idx).contiguous()
        self.net_feat = b.net_feat.index_select(0, idx).contiguous()
        # seeds: each candidate's scheduled pins (candidate by candidate); self-term slots: cell class first
        lv = inc._level[self._pins] if P else np.zeros(0, np.int32)
        loc = np.nonzero(lv >= 0)[0]
        is_cell = lv[loc] % 2 == 0
        cand = np.searchsorted(self._off, loc, side="right") - 1
        seed_ptr = np.concatenate([[0], np.cumsum(np.bincount(cand, minlength=K))]).astype(np.int32)
        slot = np.empty(loc.size, np.int64)
        nc = int(is_cell.sum())
        slot[is_cell] = np.arange(nc)
        slot[~is_cell] = nc + np.arange(loc.size - nc)
        i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)    # noqa: E731
        self._seed_ptr, self._seeds, self._seed_slot = i32(seed_ptr), i32(self._pins[loc]), i32(slot)
        self._x_cell, self._x_net = i32(loc[is_cell]), i32(loc[~is_cell])
        self._nc = nc
        edge_cap = inc.R * max(inc.max_in_degree(), 1)
        if self.endpoints is None:
            self._fanin = None
            self.cones = ForwardCones(b.graph, K, inc.R, edge_cap, b.endpoints, loc.size)
            img = np.arange(T)
        else:
            # R(E): built once, E and the structure are fixed for this object's life
            ep = b.endpoints.index_select(0, torch.from_numpy(self.endpoints).to(dev)).contiguous()
            self._fanin = FaninCone(b.graph, keep_bits=True)
            self._fanin.build(ep, torch.ones(T, dtype=torch.float32, device=dev))
            self.cones = ForwardCones(b.graph, K, inc.R, edge_cap, ep, loc.size, within=self._fanin)
            img = self.endpoints
        self._img_rows = i32(np.tile(img, K))
        width = inc.X.shape[1]
        self._Xw = torch.empty(K * T, width, dtype=torch.float32, device=dev)
        self._pred2 = torch.empty(K * T, inc._pred2.shape[1], dtype=torch.float32, device=dev)
        self.pred = self._pred2.view(K, T)
        self._gen = None                                  # inc.generation at the last run / replay

    @staticmethod
    def _positions(endpoints, T):
        """-> int64 ndarray of the distinct endpoint positions (sorted), validated against [0, T)."""
        if torch.is_tensor(endpoints):
            if endpoints.device.type != "cpu":
                raise ValueError("IncrementalEvaluation.what_if: endpoints must be a host sequence (list, ndarray or "
                                 "CPU tensor)")
            endpoints = endpoints.numpy()
        arr = np.asarray(endpoints)
        if arr.size == 0:
            raise ValueError("IncrementalEvaluation.what_if: no endpoint")
        if not np.issubdtype(arr.dtype, np.integer):
            raise ValueError(f"IncrementalEvaluation.what_if: endpoint positions must be integers, got {arr.dtype}")
        arr = np.unique(arr.reshape(-1).astype(np.int64))
        if arr[0] < 0 or arr[-1] >= T:
            raise ValueError(f"IncrementalEvaluation.what_if: endpoint positions must lie in [0, {T}), got "
                             f"{arr[0]} .. {arr[-1]}")
        return arr

    def rows(self, k):
        """(pins int64 ndarray, cell_feat rows, net_feat rows) of candidate k: views into ``cell_feat`` / ``net_feat``."""
        if not 0 <= k < self.K:
            raise ValueError(f"WhatIf.rows: candidate {k} out of range [0, {self.K})")
        s, e = int(self._off[k]), int(self._off[k + 1])
        return self._pins[s:e], self.cell_feat[s:e], self.net_feat[s:e]

    def _launch(self):
        inc, c, st = self.inc, self.cones, self.inc.step
        gp = inc._params()
        c.build(self._seed_ptr, self._seeds, self._seed_slot, inc.S_ext)
        nc = self._nc
        tm_ops.gnn_self_terms(inc.S_ext, self.cell_feat, self.net_feat, gp, self._x_cell, self._x_net,
                              cell_out=c.seed_rows[:nc], net_out=c.seed_rows[nc:])
        tm_ops.gnn_forward_cone(c, inc.H_ext, inc.S_ext, gp)
        KT, Xw = self.K * self.T, self._Xw
        width = Xw.shape[1]
        call("tm_gather_cols", KT, D, inc.H_ext, D, c.head_rows, Xw, width, 0, stream())
        call("tm_gather_cols", KT, width - D, inc.X[:, D:], width, self._img_rows, Xw, width, D, stream())
        f0, f2 = st.model.mlp_fuse.layers[0], st.model.mlp_fuse.layers[2]
        tm_ops.mlp2_forward(Xw, width, None, KT, f0.weight.detach(), f0.bias.detach(), f2.weight.detach(),
                            f2.bias.detach(), self._pred2, self._pred2.shape[1])
        call("tm_what_if_mask", self.K, self.T, c.fitted, self._pred2, stream())
        return self.pred

    def _ran(self):
        self._gen = self.inc.generation
        self.inc._overlay = self

    def run(self):
        """Every candidate's predictions against the current base: (K, T) device tensor, rewritten by every run /
        replay."""
        self._launch()
        self._ran()
        return self.pred

    def capture(self, pool=None):
        """``run()`` captured as one CUDA graph (run once eagerly first).  Returns ``replay() -> (K, T)``: edit
        ``cell_feat`` / ``net_feat`` in place, then replay."""
        inner = self.inc.step._capture_local(self._launch, warmup=1, pool=pool)
        self._ran()

        def replay():
            inner()
            self._ran()
            return self.pred
        replay.graph = inner.graph
        return replay

    def commit(self, k):
        """Apply candidate k: the batch's feature rows, ``inc.H``, ``inc.S``, ``inc.pred`` and the head's inputs as
        ``inc.update`` leaves them, without a propagation.  With ``endpoints`` the run computed only the part of the
        cone inside R(E): candidate k's feature rows are written into the batch and ``inc.update(pins)`` propagates
        them, so the state is exactly the one ``update`` leaves."""
        inc = self.inc
        if self._gen is None or self._gen != inc.generation or inc._overlay is not self:
            raise ValueError("WhatIf.commit: the base changed (or another what-if ran) since this object's last run / "
                             "replay; run it again first")
        if not isinstance(k, (int, np.integer)) or not 0 <= k < self.K:
            raise ValueError(f"WhatIf.commit: candidate {k!r} out of range [0, {self.K})")
        c = self.cones
        if not bool(c.fitted[k].item()):
            raise ValueError(f"WhatIf.commit: candidate {k} was not admitted (what_if_rows too small)")
        s, e = int(self._off[k]), int(self._off[k + 1])
        if self._fanin is not None:                      # restricted: only the part of the cone inside R(E) ran
            if e > s:
                inc.b.cell_feat.index_copy_(0, self._pin_idx[s:e], self.cell_feat[s:e])
                inc.b.net_feat.index_copy_(0, self._pin_idx[s:e], self.net_feat[s:e])
            inc.update(self._pins[s:e])
            return
        call("tm_what_if_commit", inc.n, int(k), c.fitted, c.sizes, c.row_base, c.vpin, inc.H_ext, inc.S_ext, stream())
        if e > s:
            inc.b.cell_feat.index_copy_(0, self._pin_idx[s:e], self.cell_feat[s:e])
            inc.b.net_feat.index_copy_(0, self._pin_idx[s:e], self.net_feat[s:e])
        # the head over the committed H: candidate k's predictions (the same bits) and the head's X / hidden rows
        inc.step._head_netlist_side(inc.H, inc.b, inc._hs, out=inc._pred2, hf_out=inc._hf)
        inc.generation += 1
        inc._last = ("what_if", self, int(k))

    def fitted(self):
        """(K,) bool host array: the candidates admitted by the last run / replay (one device read)."""
        return self.cones.fitted.cpu().numpy().astype(bool)

    def cone_sizes(self):
        """(K,) int host array: each candidate's cone pins in the last run / replay (one device read); with
        ``endpoints``, the pins of its cone inside R(E)."""
        return self.cones.sizes.cpu().numpy().astype(np.int64)

    def within_size(self):
        """|R(E)|, the pins of the endpoints' fan-in cone (one device read, diagnostics only); the schedule's pin count
        without ``endpoints``."""
        return self._fanin.size() if self._fanin is not None else self.inc.sched.n_sched
