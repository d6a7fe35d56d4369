"""Batch-format loader (SURVEY.md 8f N3): the reference's per-design 7-tuple, without DGL.

``generate_data.py:50-54`` writes, per design, ``th.save((graph, topo_levels, path_masks, path2level,
path2endpoint, critical_paths, cnn_inputs), '<design>.pkl')`` and ``train.py:335-388``
(``load_single_design``) turns it into what the training loop iterates.  This module reads the same
tuple -- ``graph`` may be a ``TimingGraph`` (our DGL-free container, picklable) or anything with DGL's
heterograph surface (``tm_graph.as_timing_graph``) -- and offers two consumers:

* ``load_single_design(...)``: the reference function, same arguments, same seven return values
  (``train.py:335-388``: ``ndata['h']`` / ``edata['a']`` zeros, ``feat_reduce`` trimming, min-max
  ``norm``, the 1/5 validation split file, critical-path oversampling, ``PathDataset``), so a
  ``train.py``-shaped loop runs on it unchanged;
* ``load_design(...) -> LoadedDesign``: the device-resident form the fused step consumes -- level
  schedule from ``topo_levels``, path masks as CSR, ``path -> (level, endpoint)`` as int32 tensors --
  whose ``loader(batch_size)`` yields one ``DesignBatch`` per shuffled endpoint batch, ordered exactly
  like the reference loop orders its predictions (levels ascending, inside a level the DataLoader's
  order: ``train.py:470-511``).  Building a batch is O(batch) host work and a few gathers on the device.

``design_tuple_from_synth`` / ``save_design`` write synthetic designs (``tm_synth``) in this format with
the reference's raw feature widths (``cell_feat`` 34 one-hot + 8, ``net_feat`` 3: ``dataset.py:88-99``), so
that ``feat_reduce = [6, 1]`` (``options.py:41``) trims them to the 36 / 2 columns the model is built for.
"""
import os
import pickle
import random

import numpy as np
import torch

from tm_graph import MaskCSR, TimingGraph, as_timing_graph

NUM_CTYPES = 34                  # len(ctype2id) of the ASAP7 library the reference was trained on (options.py:11)


class PathDataset(torch.utils.data.Dataset):
    """List of path ids (MyDataloader.py:62-73)."""

    def __init__(self, paths):
        self.paths = list(paths)

    def __len__(self):
        return len(self.paths)

    def __getitem__(self, i):
        return self.paths[i]


def min_max_norm(feature, start_idx):
    """train.py:308-318: columns ``start_idx..`` scaled to [0, 1] by their own min / max (NaN for a
    constant column, as in the reference: 0/0)."""
    feature = feature.clone()
    for i in range(start_idx, feature.shape[1]):
        col = feature[:, i]
        lo, hi = torch.min(col), torch.max(col)
        feature[:, i:i + 1] = ((col - lo) / (hi - lo)).reshape(-1, 1)
    return feature


def split_dataset(paths, critical_paths, rng=random):
    """train.py:294-304: one fifth of the critical and of the non-critical paths validate, the rest test."""
    non_critical = list(set(paths) - set(critical_paths))
    critical = list(critical_paths)
    rng.shuffle(critical)
    val, test = critical[:len(critical) // 5], critical[len(critical) // 5:]
    rng.shuffle(non_critical)
    val = val + non_critical[:len(non_critical) // 5]
    test = test + non_critical[len(non_critical) // 5:]
    return val, test


# --------------------------------------------------------------------------------------------
# writing (synthetic fixtures)
# --------------------------------------------------------------------------------------------
def design_tuple_from_synth(d, unet=True, seed=0, critical_frac=0.2):
    """SynthDesign -> the reference's 7-tuple with raw feature widths (42 / 3 columns)."""
    rng = np.random.default_rng(seed)
    n, P = d.n, len(d.endpoints)
    g = TimingGraph(n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis)
    cf = np.concatenate([d.cell_feat, rng.random((n, 6), dtype=np.float32)], 1)            # + the 6 trimmed columns
    nf = np.concatenate([d.net_feat, rng.random((n, 1), dtype=np.float32)], 1)
    g.ndata["cell_feat"], g.ndata["net_feat"] = torch.from_numpy(cf), torch.from_numpy(nf)
    end = np.zeros((n, 1), np.int64)
    end[d.endpoints] = 1
    start = np.zeros((n, 1), np.int64)
    start[d.pis] = 1
    arr = np.zeros((n, 1), np.float32)
    arr[d.endpoints, 0] = d.arrival_time
    critical = np.sort(rng.choice(P, max(1, int(critical_frac * P)), replace=False))
    req = arr + 0.25
    req[d.endpoints[critical], 0] = arr[d.endpoints[critical], 0] - 0.1                      # negative slack
    label = np.zeros((n, 1), np.int64)
    label[d.endpoints[critical]] = 1                                                          # dataset.py:118-122
    for k, v in (("start", start), ("end", end), ("label", label), ("arrival_time", arr), ("required_time", req)):
        g.ndata[k] = torch.from_numpy(v)
    rows = np.repeat(np.arange(P), np.diff(d.mask_indptr))
    masks = torch.sparse_coo_tensor(np.stack([rows, d.mask_cols.astype(np.int64)]), torch.ones(len(rows), dtype=torch.int64),
                                    (P, d.map_size * d.map_size))
    ep_level = d.level[d.endpoints]
    path2level = {int(p): int(ep_level[p]) for p in range(P)}
    path2endpoint = {int(p): int(d.endpoints[p]) for p in range(P)}
    image = d.image if unet else rng.random((2, 4 * d.map_size, 4 * d.map_size), dtype=np.float32)
    return g, d.topo_levels(), masks, path2level, path2endpoint, [int(c) for c in critical], image


def save_design(path, tup):
    torch.save(tup, path)


def read_design(tuple_or_path):
    if isinstance(tuple_or_path, (str, os.PathLike)):
        return torch.load(tuple_or_path, weights_only=False)          # D10: the tuple holds Python objects
    return tuple_or_path


# --------------------------------------------------------------------------------------------
# the reference function (train.py:335-388)
# --------------------------------------------------------------------------------------------
def load_single_design(usage, data_path, design, init_feat_dim, os_rate, feat_reduce, if_norm, num_ctypes=NUM_CTYPES):
    graph, topo_levels, path_masks, path2level, path2endpoint, critical_paths, cnn_inputs = \
        read_design(os.path.join(data_path, f"{design}.pkl"))
    graph = as_timing_graph(graph)
    graph.ndata["h"] = torch.zeros((graph.number_of_nodes(), init_feat_dim), dtype=torch.float)
    graph.edges["cell"].data["a"] = torch.zeros((graph.number_of_edges(etype="cell"), 1), dtype=torch.float)
    if feat_reduce is not None:
        if feat_reduce[1] != 0:
            graph.ndata["net_feat"] = graph.ndata["net_feat"][:, :-feat_reduce[1]]
        if feat_reduce[0] != 0:
            graph.ndata["cell_feat"] = graph.ndata["cell_feat"][:, :-feat_reduce[0]]
    if if_norm:
        graph.ndata["cell_feat"] = min_max_norm(graph.ndata["cell_feat"], num_ctypes)
        graph.ndata["net_feat"] = min_max_norm(graph.ndata["net_feat"], num_ctypes)
    if isinstance(cnn_inputs, np.ndarray):
        cnn_inputs = torch.from_numpy(cnn_inputs).float()
    end = graph.ndata["end"]
    paths = list(range(int((end.squeeze() == 1).sum())))
    critical_paths = list(critical_paths)
    num_pos = len(critical_paths)
    ratio = (len(paths) - num_pos) / num_pos - 1 if num_pos else 0.0
    if usage == "test":
        split_file = os.path.join(data_path, f"{design}_split.pkl")
        if os.path.exists(split_file):
            with open(split_file, "rb") as f:
                val_paths, _ = pickle.load(f)
        else:
            val_paths, test_paths = split_dataset(paths, critical_paths)
            with open(split_file, "wb") as f:
                pickle.dump((val_paths, test_paths), f)
        paths = val_paths
    if usage == "train" and os_rate != 0 and ratio > 1:
        for _ in range(os_rate):
            paths.extend(critical_paths)
    return PathDataset(paths), graph, path2level, path2endpoint, topo_levels, cnn_inputs, path_masks


# --------------------------------------------------------------------------------------------
# device-resident form for the fused step
# --------------------------------------------------------------------------------------------
class LoadedDesign:
    """One design, resident on ``device``: graph + level schedule, mask CSR, path tables, image, labels."""

    def __init__(self, tuple_or_path, device, usage="train", os_rate=1, feat_reduce=(6, 1), norm=False,
                 num_ctypes=NUM_CTYPES, data_path=None, design=None):
        if data_path is not None:
            tuple_or_path = os.path.join(data_path, f"{design}.pkl")
        (self.paths_ds, graph, path2level, path2endpoint, topo_levels, image, path_masks) = _prepared(
            tuple_or_path, usage, os_rate, feat_reduce, norm, num_ctypes)
        self.device = torch.device(device)
        self.paths = list(self.paths_ds.paths)                     # with the oversampled critical paths (train.py:377-380)
        graph.set_topo_levels(topo_levels)
        self.graph = graph.to(self.device)
        self.num_levels = len(topo_levels)
        P = path_masks.shape[0]
        self.mask_csr = MaskCSR.from_sparse_coo(path_masks).to(self.device)
        lv = torch.full((P,), -1, dtype=torch.int32)
        ep = torch.full((P,), -1, dtype=torch.int32)
        for p, l in path2level.items():
            lv[int(p)] = int(l)
        for p, e in path2endpoint.items():
            ep[int(p)] = int(e)
        self.path_level, self.path_endpoint = lv, ep                # host tables: batching is host-side index work
        self.path_level_d, self.path_endpoint_d = lv.to(self.device), ep.to(self.device)
        self.image = image.float().to(self.device)
        self.arrival = self.graph.ndata["arrival_time"].reshape(-1)
        self.required = self.graph.ndata["required_time"].reshape(-1) if "required_time" in self.graph.ndata else None
        self.label = self.graph.ndata["label"].reshape(-1) if "label" in self.graph.ndata else None

    def order_batch(self, path_ids):
        """The reference's prediction order for one DataLoader batch (train.py:477-511): levels ascending, inside
        a level the batch's own order (a stable sort by level)."""
        ids = torch.as_tensor(path_ids, dtype=torch.int64)
        return ids[torch.sort(self.path_level[ids].long(), stable=True).indices]

    def batch_tensors(self, path_ids):
        """(endpoints int32, endpoint_level fp32, arrival_time fp32, rows int32) on the device, in prediction order."""
        ids = self.order_batch(path_ids).to(self.device, non_blocking=True)
        ep = self.path_endpoint_d[ids]
        return ep, self.path_level_d[ids].float(), self.arrival[ep.long()], ids.to(torch.int32)

    def batch(self, path_ids, dynamic=False):
        """-> ``tm_engine.DesignBatch`` for these paths."""
        import tm_engine
        ep, lv, arr, rows = self.batch_tensors(path_ids)
        return tm_engine.DesignBatch(self.graph, self.mask_csr, ep, lv, arr.clone(), self.image, rows=rows, dynamic=dynamic)

    def prepare(self, step, batch_size=1350):
        """One CUDA-graph capture for the whole design: returns ``run(path_ids) -> (loss, pred)`` that refreshes the
        endpoint batch in place (O(batch) host work: a stable sort of ``batch_size`` levels and four small copies) and
        replays the captured step, which re-selects the mask rows on the device.  ``len(path_ids)`` must equal
        ``batch_size`` (the reference drops the last partial batch when a design has more paths than that)."""
        first = [self.paths[i % len(self.paths)] for i in range(batch_size)]
        b = self.batch(first, dynamic=True)
        replay = step.capture(b)

        def run(path_ids):
            assert len(path_ids) == batch_size, "a prepared design replays fixed-size batches"
            b.set_endpoints(*self.batch_tensors(path_ids))
            return replay()
        run.batch = b
        return run

    def eval_batch(self, paths=None):
        """-> (``tm_engine.DesignBatch``, path ids in prediction order) for ``DesignStep.evaluate``: ``paths`` (default:
        the design's paths without the oversampled critical duplicates -- for ``usage="test"`` the validation split), with
        the endpoints' required times and critical labels when the design has them."""
        ids = self.order_batch(list(dict.fromkeys(self.paths)) if paths is None else paths)
        b = self.batch(ids)
        ep = b.endpoints.long()
        if self.required is not None:
            b.required = self.required[ep].contiguous()
        if self.label is not None:
            b.label = self.label[ep].to(torch.int64).contiguous()
        return b, ids

    def prepare_evaluate(self, step, paths=None):
        """One CUDA-graph capture of ``step.evaluate`` over a fixed set of paths (validate(), train.py:137-291, or one
        test design, test.py:124-318): returns ``run() -> (pred, metrics)`` that replays it; ``run.batch`` is the batch
        and ``run.paths`` the path ids in prediction order.  Refresh values in place (``run.batch.cell_feat`` ...,
        ``arrival_time``) between replays if they change; the paths and their levels are fixed."""
        b, ids = self.eval_batch(paths)
        run = step.capture_evaluate(b)
        run.batch, run.paths = b, ids
        return run

    def loader(self, batch_size=1350, shuffle=True, generator=None):
        """Batches like ``DataLoader(PathDataset(paths), batch_size, shuffle=True, drop_last=len(paths) > batch_size)``
        (train.py:468-472; the reference decides ``drop_last`` on ``len(path2level)``)."""
        n = len(self.paths)
        order = torch.randperm(n, generator=generator) if shuffle else torch.arange(n)
        ids = torch.as_tensor(self.paths, dtype=torch.int64)[order]
        drop_last = int((self.path_level >= 0).sum()) > batch_size
        stop = (n // batch_size) * batch_size if drop_last else n
        for i in range(0, stop, batch_size):
            yield self.batch(ids[i:i + batch_size])


def prepare_many(designs, step, batch_size=1350):
    """``LoadedDesign.prepare`` for K designs stepped together (``tm_engine.DesignBatch.concat``): ONE CUDA-graph
    capture, and ``run(list of K path-id lists) -> (loss, pred)`` refreshes every design's endpoint batch in place and
    replays the captured step, which re-selects every design's mask rows on the device.  Each list must hold
    ``batch_size`` path ids."""
    import tm_engine
    designs = list(designs)
    parts = [d.batch([d.paths[i % len(d.paths)] for i in range(batch_size)], dynamic=True) for d in designs]
    b = tm_engine.DesignBatch.concat(parts)
    replay = step.capture(b)

    def run(path_id_lists):
        assert len(path_id_lists) == len(designs), "one path-id list per prepared design"
        for k, (d, ids) in enumerate(zip(designs, path_id_lists)):
            assert len(ids) == batch_size, "a prepared design replays fixed-size batches"
            b.set_endpoints(*d.batch_tensors(ids), design=k)
        return replay()
    run.batch = b
    return run


def prepare_evaluate_many(designs, step, paths=None):
    """``LoadedDesign.prepare_evaluate`` for K designs in ONE CUDA graph (``tm_engine.DesignBatch.concat``): a whole test
    set per replay.  ``paths``: None (every design's default) or one path-id list per design.  Returns ``run() -> (pred,
    metrics)``; ``metrics.design[k]`` / ``metrics.level[k]`` are design k's rows, ``run.paths[k]`` its path ids in
    prediction order (its predictions are ``pred[run.batch.ep_off_h[k]:run.batch.ep_off_h[k + 1]]``)."""
    import tm_engine
    designs = list(designs)
    if paths is None:
        paths = [None] * len(designs)
    if len(paths) != len(designs):
        raise ValueError(f"prepare_evaluate_many: {len(paths)} path lists for {len(designs)} designs")
    parts = [d.eval_batch(p) for d, p in zip(designs, paths)]
    b = tm_engine.DesignBatch.concat([x[0] for x in parts])
    run = step.capture_evaluate(b)
    run.batch, run.paths = b, [x[1] for x in parts]
    return run


def _prepared(tuple_or_path, usage, os_rate, feat_reduce, norm, num_ctypes):
    if isinstance(tuple_or_path, (str, os.PathLike)):
        data_path, fname = os.path.split(str(tuple_or_path))
        return load_single_design(usage, data_path, fname[:-4], 128, os_rate, list(feat_reduce) if feat_reduce else None,
                                  norm, num_ctypes)
    # an in-memory tuple: same treatment without touching the file system
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        save_design(os.path.join(tmp, "d.pkl"), tuple_or_path)
        return load_single_design("train" if usage == "train" else usage, tmp, "d", 128, os_rate,
                                  list(feat_reduce) if feat_reduce else None, norm, num_ctypes)


def load_design(tuple_or_path, device="cuda", **kw):
    return LoadedDesign(tuple_or_path, device, **kw)
