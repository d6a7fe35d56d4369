"""Device-resident graph batch: a DGL-heterograph-shaped container plus its level schedule.

``TimingGraph`` exposes exactly the surface of the DGL graph that the reference touches
(SURVEY.md 8b): ``ndata``, ``nodes['pin'].data``, ``edges[etype].data``, ``number_of_nodes``,
``number_of_edges(etype=)``, ``edges(etype=)``, ``to(device)`` -- the batch format produced by
``src/dataset.py:274-287`` -- so ``src/train.py`` / ``src/test.py`` style loops can hand it to
``PathModel`` unchanged.  A real ``dgl.DGLGraph`` is accepted too (``as_timing_graph``).

``Schedule`` is what replaces DGL's per-``pull`` graph slicing: in/out CSRs of both edge types,
pin -> level, pins ordered by (level, id), level offsets -- built ONCE per graph on the GPU by
``libtm_b200`` (``tm_csr_build``, ``tm_levelize``, ``tm_level_order``, ``tm_schedule_aux``).
"""
import ctypes

import numpy as np
import torch

import tm_lib


class _View:
    def __init__(self, data):
        self.data = data


class TimingGraph:
    def __init__(self, num_nodes, net_edges, cell_edges, pis=None):
        """``net_edges`` / ``cell_edges``: ``(src, dst)`` int64 tensors or arrays
        (driver pin -> sink pin; cell input pin -> cell output pin, dataset.py:274-278)."""
        self._n = int(num_nodes)
        self._edges = {"net": tuple(torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x,
                                                    dtype=torch.int64) for x in net_edges),
                       "cell": tuple(torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x,
                                                     dtype=torch.int64) for x in cell_edges)}
        self.pis = None if pis is None else torch.as_tensor(np.asarray(pis) if not torch.is_tensor(pis) else pis,
                                                            dtype=torch.int64)
        self.ndata = {}
        self.nodes = {"pin": _View(self.ndata)}
        self.edges_data = {"net": {}, "cell": {}}
        self._topo_levels = None
        self._levels = None                        # (device int32 level per pin, number of levels): see ConeGraph
        self._schedule = None

    # ---- pickling (the reference stores the graph inside its per-design tuple, generate_data.py:50-54) ----
    def __getstate__(self):
        st = dict(self.__dict__)
        st["_schedule"] = None                     # device-side, rebuilt on first use
        st.pop("nodes", None)
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        self.nodes = {"pin": _View(self.ndata)}

    # ---- DGL surface -------------------------------------------------------------------------
    class _EdgeAccessor:
        def __init__(self, g):
            self._g = g

        def __getitem__(self, etype):
            return _View(self._g.edges_data[etype])

        def __call__(self, etype=None):
            return self._g._edges[etype]

    @property
    def edges(self):
        return TimingGraph._EdgeAccessor(self)

    def number_of_nodes(self):
        return self._n

    num_nodes = number_of_nodes

    def number_of_edges(self, etype=None):
        if etype is None:
            return sum(int(e[0].numel()) for e in self._edges.values())
        return int(self._edges[etype][0].numel())

    def to(self, device):
        """Moves edges and every ndata/edata tensor (``graph.to(device)``, train.py:467); in place."""
        device = torch.device(device)
        self._edges = {k: tuple(t.to(device, non_blocking=True) for t in v) for k, v in self._edges.items()}
        if self.pis is not None:
            self.pis = self.pis.to(device, non_blocking=True)
        for k in list(self.ndata):
            self.ndata[k] = self.ndata[k].to(device, non_blocking=True)
        for et in self.edges_data:
            for k in list(self.edges_data[et]):
                self.edges_data[et][k] = self.edges_data[et][k].to(device, non_blocking=True)
        if self._schedule is not None and self._schedule.device != device:
            self._schedule = None
        return self

    @property
    def device(self):
        return self._edges["net"][0].device

    # ---- schedule ----------------------------------------------------------------------------
    def set_topo_levels(self, topo_levels):
        """Use caller-provided levels (the reference's ``topo_levels``: a list of
        ``(nodes, targets, path_ids)`` tuples or of plain node lists) instead of recomputing them."""
        self._topo_levels = [lv[0] if isinstance(lv, (tuple, list)) and len(lv) and
                             isinstance(lv[0], (list, tuple, np.ndarray, torch.Tensor)) else lv
                             for lv in topo_levels]
        self._schedule = None

    def schedule(self):
        if self._schedule is None:
            self._schedule = Schedule.build(self)
        return self._schedule


def as_timing_graph(g):
    """Accept a TimingGraph or anything with DGL's heterograph surface."""
    if isinstance(g, TimingGraph):
        return g
    cached = getattr(g, "_tm_timing_graph", None)
    if cached is not None:
        return cached
    net = g.edges(etype="net")
    cell = g.edges(etype="cell")
    tg = TimingGraph(g.number_of_nodes(), (net[0], net[1]), (cell[0], cell[1]))
    tg.ndata = g.ndata                      # share the frame: features / 'h' live with the caller
    tg.nodes = {"pin": _View(tg.ndata)}
    try:
        g._tm_timing_graph = tg
    except Exception:
        pass
    return tg


def build_csr(n, key, val):
    """-> (indptr int32 [n+1], indices int32 [e]) on ``key.device`` via tm_csr_build."""
    tm_lib.require_cuda(key, "edge list")
    e = int(key.numel())
    dev = key.device
    indptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
    indices = torch.empty(max(e, 1), dtype=torch.int32, device=dev)
    nb = tm_lib.ws_bytes("tm_csr_build_ws", n, e)
    ws = tm_lib.workspace(nb, dev)
    tm_lib.call("tm_csr_build", n, e, key.contiguous(), val.contiguous(), indptr, indices, ws, nb,
                tm_lib.stream())
    return indptr, indices[:e]


class Schedule:
    """Level schedule + CSRs of one graph, all int32 tensors on the device."""

    @staticmethod
    def build(g):
        dev = g.device
        if dev.type != "cuda":
            raise RuntimeError("TimingGraph must be moved to a CUDA device first (graph.to('cuda')): "
                               "there is no CPU path")
        s = Schedule()
        s.device = dev
        n = s.n = g.number_of_nodes()
        ns, nd = g._edges["net"]
        cs, cd = g._edges["cell"]
        s.net_iptr, s.net_isrc = build_csr(n, nd, ns)
        s.cell_iptr, s.cell_isrc = build_csr(n, cd, cs)
        s.net_optr, s.net_odst = build_csr(n, ns, nd)
        s.cell_optr, s.cell_odst = build_csr(n, cs, cd)
        st = tm_lib.stream()
        s.level = torch.empty(n, dtype=torch.int32, device=dev)
        if getattr(g, "_levels", None) is not None:
            s.level.copy_(g._levels[0])
            L = int(g._levels[1])
        elif g._topo_levels is not None:
            lv = np.full(n, -1, np.int32)
            for lid, nodes in enumerate(g._topo_levels):
                lv[np.asarray(nodes, dtype=np.int64)] = lid
            s.level.copy_(torch.from_numpy(lv))
            L = len(g._topo_levels)
        else:
            src_all, dst_all = torch.cat([ns, cs]), torch.cat([nd, cd])
            optr, odst = build_csr(n, src_all, dst_all)
            if g.pis is not None:
                pis = g.pis.to(dev)
            else:                                   # pins without any in-edge start the sweep
                indeg = (s.net_iptr[1:] - s.net_iptr[:-1]) + (s.cell_iptr[1:] - s.cell_iptr[:-1])
                pis = torch.nonzero(indeg == 0).squeeze(1)
            nl = torch.zeros(1, dtype=torch.int32, device=dev)
            nb = tm_lib.ws_bytes("tm_levelize_ws", n)
            ws = tm_lib.workspace(nb, dev)
            tm_lib.call("tm_levelize", n, optr, odst, pis.contiguous(), int(pis.numel()), s.level, nl, ws, nb, st)
            L = int(nl.item())
        if L <= 0:
            raise RuntimeError("empty level schedule (no primary inputs?)")
        s.num_levels = L
        s.order = torch.empty(n, dtype=torch.int32, device=dev)
        level_ptr = torch.empty(L + 1, dtype=torch.int32, device=dev)
        nb = tm_lib.ws_bytes("tm_level_order_ws", n, L)
        ws = tm_lib.workspace(nb, dev)
        tm_lib.call("tm_level_order", n, L, s.level, s.order, level_ptr, ws, nb, st)
        s.crow = torch.empty(n, dtype=torch.int32, device=dev)
        cell_base = torch.empty(L + 1, dtype=torch.int32, device=dev)
        viol = torch.zeros(1, dtype=torch.int32, device=dev)
        tm_lib.call("tm_schedule_aux", n, L, s.level, s.order, level_ptr, s.net_iptr, s.net_isrc,
                    s.cell_iptr, s.cell_isrc, s.crow, cell_base, viol, st)
        host = torch.cat([level_ptr, cell_base, viol]).cpu().numpy()          # the one sync
        s.level_ptr = level_ptr
        s.cell_base = cell_base
        s.h_level_ptr = np.ascontiguousarray(host[:L + 1], dtype=np.int32)
        s.h_cell_base = np.ascontiguousarray(host[L + 1:2 * L + 2], dtype=np.int32)
        s.n_sched = int(s.h_level_ptr[L])
        s.n_cell_rows = int(s.h_cell_base[L])
        if int(host[-1]) != 0:
            raise RuntimeError(f"level schedule is not topological: {int(host[-1])} in-edges come from "
                               "the same or a later level")
        s.order = s.order[:s.n_sched]
        # pins grouped by which hoisted self-term MLP feeds them (even levels: fc_cell_self,
        # odd levels: fc_net_self; model.py:104,141,151)
        lv_sorted = s.level[s.order.long()]
        s.cell_class = s.order[(lv_sorted % 2) == 0].contiguous()
        s.net_class = s.order[(lv_sorted % 2) == 1].contiguous()
        s.struct = tm_lib.tm_schedule(
            n=n, num_levels=L, n_cell_rows=s.n_cell_rows,
            h_level_ptr=s.h_level_ptr.ctypes.data_as(ctypes.c_void_p).value,
            order=s.order.data_ptr(), level=s.level.data_ptr(), crow=s.crow.data_ptr(),
            net_iptr=s.net_iptr.data_ptr(), net_isrc=s.net_isrc.data_ptr(),
            cell_iptr=s.cell_iptr.data_ptr(), cell_isrc=s.cell_isrc.data_ptr(),
            net_optr=s.net_optr.data_ptr(), net_odst=s.net_odst.data_ptr(),
            cell_optr=s.cell_optr.data_ptr(), cell_odst=s.cell_odst.data_ptr(),
            level_ptr=s.level_ptr.data_ptr(), cell_base=s.cell_base.data_ptr())
        # level-ordered edge lists: what the propagation kernels actually walk
        e_net, e_cell = int(s.net_isrc.numel()), int(s.cell_isrc.numel())
        ns1 = s.n_sched + 1
        s.f_ptr = torch.empty(ns1, dtype=torch.int32, device=dev)
        s.f_src = torch.empty(max(e_net + e_cell, 1), dtype=torch.int32, device=dev)
        s.bn_ptr = torch.empty(ns1, dtype=torch.int32, device=dev)
        s.bn_dst = torch.empty(max(e_net, 1), dtype=torch.int32, device=dev)
        s.bn_w = torch.empty(max(e_net, 1), dtype=torch.float32, device=dev)
        s.bc_ptr = torch.empty(ns1, dtype=torch.int32, device=dev)
        s.bc_row = torch.empty(max(e_cell, 1), dtype=torch.int32, device=dev)
        nb = tm_lib.ws_bytes("tm_schedule_edges_ws", s.n_sched)
        ws = tm_lib.workspace(nb, dev)
        tm_lib.call("tm_schedule_edges", s.struct, s.n_sched, s.f_ptr, s.f_src, s.bn_ptr, s.bn_dst, s.bn_w,
                    s.bc_ptr, s.bc_row, ws, nb, st)
        for k in ("f_ptr", "f_src", "bn_ptr", "bn_dst", "bn_w", "bc_ptr", "bc_row"):
            setattr(s.struct, k, getattr(s, k).data_ptr())
        return s

    def level_nodes(self, lid):
        return self.order[int(self.h_level_ptr[lid]):int(self.h_level_ptr[lid + 1])]

    def algorithmic_bytes_fwd(self, D=128):
        """SURVEY.md 8d: bytes the forward propagation must move (fp32, int32 indices)."""
        e = int(self.net_isrc.numel() + self.cell_isrc.numel())
        n = self.n_sched
        return 4 * D * e + 4 * D * n + 4 * D * n + 4 * e + 4 * (2 * n + self.num_levels)

    def algorithmic_bytes_bwd(self, D=128):
        e = int(self.net_isrc.numel() + self.cell_isrc.numel())
        return 4 * D * (2 * e + 4 * self.n_sched)


class BackwardCone:
    """The pins that can receive a gradient from one endpoint batch: everything from which an endpoint is reachable
    along net / cell edges.  Every other pin's dLoss/dz row is exactly zero, so the weight-gradient contractions of
    the backward pass (three per hoisted MLP, two for ``fc_cell_neigh``) only need the cone's rows -- 44 % of the pins
    for 1 350 endpoints of the config-2 design.  Built once per (graph, endpoint batch): ~100 scatter passes over the
    edge list on the device, one host read of the three list lengths.

    ``cell_pins`` / ``net_pins``: the cone's members of ``Schedule.cell_class`` / ``net_class`` (pin ids, schedule
    order); ``cell_pos``: their positions inside ``cell_class`` (rows of the saved hidden activations);
    ``crows``: the cone's rows of the per-cell-level buffers A / LSE / HID / GZC / GHID."""

    def __init__(self, graph, sched, endpoints):
        n = graph.number_of_nodes()
        act = _reaches_endpoint(graph, endpoints)
        cur = int(act.sum())
        self.active = act.bool()
        cc, nc = sched.cell_class.long(), sched.net_class.long()
        mc, mn = self.active[cc], self.active[nc]
        self.cell_pos = torch.nonzero(mc).flatten().int().contiguous()
        self.cell_pins = sched.cell_class[mc].contiguous()
        self.net_pins = sched.net_class[mn].contiguous()
        self.net_pos = torch.nonzero(mn).flatten().int().contiguous()
        cr = sched.crow[self.active]
        self.crows = torch.sort(cr[cr >= 0]).values.int().contiguous()
        self.n_active = cur
        self.fraction = cur / max(n, 1)


class ForwardCone:
    """The forward cone of a set of seed pins as a device-side sub-schedule of ``graph.schedule()``: every scheduled pin
    reachable from a scheduled seed along the in-edges the propagation reads, the seeds included -- the pins whose H
    row can change when the seeds' self terms change.  ``build(seeds)`` enqueues ``tm_forward_cone`` (no host
    synchronisation, so it can be captured) and returns ``.struct``, a ``tm_schedule`` that ``tm_gnn_forward_cone``
    propagates over.  The buffers are allocated once, sized by the parent schedule, and rewritten by every build.

    The struct has no host level offsets (``h_level_ptr`` NULL), so ``tm_gnn_forward`` / ``tm_gnn_backward`` refuse
    it; it has no cell rows (``n_cell_rows`` 0, ``cell_base`` all zero) and no backward edge lists."""

    def __init__(self, graph):
        s = self.sched = graph.schedule()
        dev = s.device
        i32 = lambda k: torch.empty(max(int(k), 1), dtype=torch.int32, device=dev)      # noqa: E731
        self.order = i32(s.n_sched)
        self.level_ptr = i32(s.num_levels + 1)
        self.f_ptr = i32(s.n_sched + 1)
        self.f_src = i32(s.f_src.numel())
        self.count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.cell_base = torch.zeros(s.num_levels + 1, dtype=torch.int32, device=dev)
        self.nb = tm_lib.ws_bytes("tm_forward_cone_ws", s.n)
        self.ws = tm_lib.workspace(self.nb, dev)
        p = s.struct
        self.struct = tm_lib.tm_schedule(
            n=s.n, num_levels=s.num_levels, n_cell_rows=0, h_level_ptr=None,
            order=self.order.data_ptr(), level=p.level, crow=None,
            net_iptr=p.net_iptr, net_isrc=p.net_isrc, cell_iptr=p.cell_iptr, cell_isrc=p.cell_isrc,
            net_optr=p.net_optr, net_odst=p.net_odst, cell_optr=p.cell_optr, cell_odst=p.cell_odst,
            f_ptr=self.f_ptr.data_ptr(), f_src=self.f_src.data_ptr(),
            level_ptr=self.level_ptr.data_ptr(), cell_base=self.cell_base.data_ptr())

    def build(self, seeds):
        """Enqueue the cone of ``seeds`` (int32 pin ids on the device; duplicates and pins outside the schedule are
        allowed) on the current stream.  Returns ``.struct``."""
        if not (torch.is_tensor(seeds) and seeds.dtype == torch.int32 and seeds.device == self.sched.device):
            raise ValueError(f"ForwardCone.build: seeds must be an int32 tensor on {self.sched.device}")
        seeds = seeds.contiguous()
        tm_lib.call("tm_forward_cone", self.sched.struct, int(seeds.numel()), seeds, self.order, self.level_ptr,
                    self.f_ptr, self.f_src, self.count, self.ws, self.nb, tm_lib.stream())
        return self.struct

    def size(self):
        """Pins in the last built cone (one device read: diagnostics only)."""
        return int(self.count.item())


class FaninCone:
    """The fan-in cone of the endpoints a backward pass is seeded on, as a device-side sub-schedule of
    ``graph.schedule()``: every scheduled pin from which an endpoint with a non-zero seed is reachable along the out-edges
    the backward reads, those endpoints included -- the pins whose gradient can be non-zero.  ``build(endpoints, seed)``
    enqueues ``tm_fanin_cone``, which reads both on the device (no host synchronisation, so it can be captured with the
    seed as a static input), and returns ``.struct``: the sub-schedule ``tm_gnn_save_cone`` / ``tm_gnn_backward_cone``
    run over, laid out at the end of the buffers (see the header), with the backward edge lists filtered to the cone and
    cone cell rows.  ``cell_pins`` / ``net_pins`` list the cone's pins on even / odd levels (the rows of the two
    self-term MLPs), ``counts`` (device int32 [3]) the cone's pins and the two lists' lengths.  The buffers are
    allocated once, sized by the parent schedule, and rewritten by every build.

    ``keep_bits=True`` keeps the cone's membership bitmap in ``bits`` (device int32 [ceil(n / 32)], bit v of word
    v // 32 for pin v; ``tm_fanin_cone_bits``): the restriction ``ForwardCones(..., within=cone)`` reads it.

    Not ``BackwardCone``: that one is built on the host for the weight-gradient contractions of a training step."""

    def __init__(self, graph, keep_bits=False):
        s = self.sched = graph.schedule()
        dev = s.device
        i32 = lambda k: torch.empty(max(int(k), 1), dtype=torch.int32, device=dev)      # noqa: E731
        self.bits = i32((s.n + 31) // 32) if keep_bits else None
        self.order = i32(s.n_sched)
        self.level_ptr = i32(s.num_levels + 1)
        self.cell_base = i32(s.num_levels + 1)
        self.f_ptr, self.f_src = i32(s.n_sched + 1), i32(s.f_src.numel())
        self.bn_ptr, self.bn_dst = i32(s.n_sched + 1), i32(s.bn_dst.numel())
        self.bn_w = torch.empty(max(int(s.bn_w.numel()), 1), dtype=torch.float32, device=dev)
        self.bc_ptr, self.bc_row = i32(s.n_sched + 1), i32(s.bc_row.numel())
        self.n_cell_cap, self.n_net_cap = int(s.cell_class.numel()), int(s.net_class.numel())
        self.cell_pins, self.net_pins = i32(self.n_cell_cap), i32(self.n_net_cap)
        self.counts = torch.zeros(3, dtype=torch.int32, device=dev)
        self.nb = tm_lib.ws_bytes("tm_fanin_cone_ws", s.n, s.n_cell_rows)
        self.ws = tm_lib.workspace(self.nb, dev)
        p = s.struct
        self.struct = tm_lib.tm_schedule(
            n=s.n, num_levels=s.num_levels, n_cell_rows=s.n_cell_rows, h_level_ptr=None,
            order=self.order.data_ptr(), level=p.level, crow=None,
            net_iptr=p.net_iptr, net_isrc=p.net_isrc, cell_iptr=p.cell_iptr, cell_isrc=p.cell_isrc,
            net_optr=p.net_optr, net_odst=p.net_odst, cell_optr=p.cell_optr, cell_odst=p.cell_odst,
            f_ptr=self.f_ptr.data_ptr(), f_src=self.f_src.data_ptr(),
            bn_ptr=self.bn_ptr.data_ptr(), bn_dst=self.bn_dst.data_ptr(), bn_w=self.bn_w.data_ptr(),
            bc_ptr=self.bc_ptr.data_ptr(), bc_row=self.bc_row.data_ptr(),
            level_ptr=self.level_ptr.data_ptr(), cell_base=self.cell_base.data_ptr())

    def build(self, endpoints, seed):
        """Enqueue the cone of the ``endpoints`` (int32 pin ids on the device) whose ``seed`` (float32, as long) is
        non-zero, on the current stream.  Returns ``.struct``."""
        dev = self.sched.device
        if not (torch.is_tensor(endpoints) and endpoints.dtype == torch.int32 and endpoints.device == dev
                and torch.is_tensor(seed) and seed.dtype == torch.float32 and seed.device == dev
                and seed.shape == endpoints.shape and endpoints.is_contiguous() and seed.is_contiguous()):
            raise ValueError(f"FaninCone.build: endpoints (int32) and seed (float32) must be contiguous tensors of one "
                             f"shape on {dev}")
        args = (self.sched.struct, int(endpoints.numel()), endpoints, seed, self.order, self.level_ptr, self.cell_base,
                self.f_ptr, self.f_src, self.bn_ptr, self.bn_dst, self.bn_w, self.bc_ptr, self.bc_row, self.cell_pins,
                self.net_pins, self.counts)
        if self.bits is None:
            tm_lib.call("tm_fanin_cone", *args, self.ws, self.nb, tm_lib.stream())
        else:
            tm_lib.call("tm_fanin_cone_bits", *args, self.bits, self.ws, self.nb, tm_lib.stream())
        return self.struct

    def size(self):
        """Pins in the last built cone (one device read: diagnostics only)."""
        return int(self.counts[0].item())


class ForwardCones:
    """The forward cones of ``n_cand`` candidate edits of one design, joined into one device-side sub-schedule over
    private virtual rows (``tm_forward_cones``): candidate k's cone pins get the rows ``n + row_base[k] + rank`` of
    (n + rows + 1)-row H / S buffers, so K alternative edits propagate side by side in one ``tm_gnn_forward_cone``
    without touching the rows of the design's pins.  Row ``n + rows`` is a sink row.  Candidates are admitted in index
    order while their cone pins fit in ``rows`` and their cone in-edges in ``edge_cap``; ``fitted`` marks them.

    ``build(seed_ptr, seeds, seed_slot, S)`` enqueues the build (no host synchronisation, so it can be captured),
    copies every cone pin's S row to its virtual row and returns ``.struct``.  It also fills ``seed_rows`` (the
    virtual row of every seed, or the sink row), ``head_rows`` (K x T: each endpoint's row per candidate), ``vpin``,
    ``fitted``, ``sizes`` and ``row_base``.  The buffers are allocated once: the joined arrays sized by ``rows`` and
    ``edge_cap``, two n/8-byte bitmaps per candidate in the workspace.

    ``within``: a built ``FaninCone(graph, keep_bits=True)`` of endpoints E restricts every cone to E's fan-in cone
    R(E) (``tm_forward_cones_within``): candidate k's cone is its forward cone intersected with R(E), the sweeps walk
    R(E)'s sub-schedule instead of the whole schedule, and seeds outside R(E) are treated as seeds outside the schedule.
    Exact for the predictions of E: R(E) holds every in-edge source of its pins.  The fan-in cone must not be rebuilt
    for other endpoints while this object is in use."""

    def __init__(self, graph, n_cand, rows, edge_cap, endpoints, n_seeds, within=None):
        s = self.sched = graph.schedule()
        dev = s.device
        if within is not None and within.bits is None:
            raise ValueError("ForwardCones: the restriction needs a FaninCone built with keep_bits=True")
        self.within, self.n_seeds = within, int(n_seeds)
        i32 = lambda k: torch.empty(max(int(k), 1), dtype=torch.int32, device=dev)      # noqa: E731
        self.K, self.rows, self.edge_cap, self.T = int(n_cand), int(rows), int(edge_cap), int(endpoints.numel())
        self.endpoints = endpoints
        self.order = i32(rows)
        self.level_ptr = i32(s.num_levels + 1)
        self.f_ptr = i32(rows + 1)
        self.f_src = i32(edge_cap)
        self.count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.vpin = i32(rows)
        self.seed_rows = i32(n_seeds)
        self.head_rows = i32(self.K * self.T)
        self.fitted = torch.zeros(self.K, dtype=torch.int32, device=dev)
        self.sizes = torch.zeros(self.K, dtype=torch.int32, device=dev)
        self.row_base = torch.zeros(self.K, dtype=torch.int32, device=dev)
        self.cell_base = torch.zeros(s.num_levels + 1, dtype=torch.int32, device=dev)
        if within is None:
            self.nb = tm_lib.ws_bytes("tm_forward_cones_ws", s.n, self.K, s.num_levels)
        else:
            self.nb = tm_lib.ws_bytes("tm_forward_cones_within_ws", s.n, self.K, s.num_levels, self.n_seeds)
        self.ws = tm_lib.workspace(self.nb, dev)
        # only what tm_gnn_forward_cone reads: the joined order / level_ptr / f_ptr / f_src over n + rows + 1 rows
        self.struct = tm_lib.tm_schedule(
            n=s.n + rows + 1, num_levels=s.num_levels, n_cell_rows=0, h_level_ptr=None,
            order=self.order.data_ptr(), f_ptr=self.f_ptr.data_ptr(), f_src=self.f_src.data_ptr(),
            level_ptr=self.level_ptr.data_ptr(), cell_base=self.cell_base.data_ptr())

    def build(self, seed_ptr, seeds, seed_slot, S):
        """Enqueue the joined cones of the candidates' seeds (int32 device CSR ``seed_ptr`` (K+1) / ``seeds``; seed i's
        row goes to ``seed_rows[seed_slot[i]]``) on the current stream, with S the (n + rows + 1, 128) self terms.
        Returns ``.struct``."""
        out = (self.rows, self.edge_cap, self.T, self.endpoints, S, self.order, self.level_ptr, self.f_ptr, self.f_src,
               self.count, self.vpin, self.seed_rows, self.head_rows, self.fitted, self.sizes, self.row_base, self.ws,
               self.nb, tm_lib.stream())
        if self.within is None:
            tm_lib.call("tm_forward_cones", self.sched.struct, self.K, seed_ptr, seeds, seed_slot, *out)
        else:
            if int(seeds.numel()) > self.n_seeds:
                raise ValueError(f"ForwardCones.build: {int(seeds.numel())} seeds, sized for {self.n_seeds}")
            tm_lib.call("tm_forward_cones_within", self.within.struct, self.within.bits, self.K, seed_ptr, seeds,
                        seed_slot, int(seeds.numel()), *out)
        return self.struct


def _reaches_endpoint(graph, endpoints):
    """int32 (n,): 1 for every pin from which one of ``endpoints`` is reachable along net / cell edges (the endpoints
    included).  ~num_levels scatter passes over the edge list, on the device."""
    dev = endpoints.device
    n = graph.number_of_nodes()
    src = torch.cat([e[0] for e in graph._edges.values()]).to(dev).long()
    dst = torch.cat([e[1] for e in graph._edges.values()]).to(dev).long()
    act = torch.zeros(n, dtype=torch.int32, device=dev)
    act[endpoints.long()] = 1
    prev = -1
    while True:
        for _ in range(16):
            act.scatter_reduce_(0, src, act[dst], "amax", include_self=True)
        cur = int(act.sum())
        if cur == prev:
            return act
        prev = cur


class ConeGraph:
    """The sub-netlist that one endpoint batch can see: the pins from which an endpoint is reachable, renumbered in
    their original order, with every edge between them and their ORIGINAL levels.

    A pin outside this cone influences no prediction of the batch (its H row is never read on a path to an endpoint)
    and receives no gradient, and every in-edge of a cone pin comes from a cone pin -- so the propagation, the
    hoisted MLPs and every weight gradient computed on the sub-netlist give the same predictions, loss and parameter
    gradients as on the whole netlist, over ``fraction`` of the pins (44 % for 1 350 endpoints of the config-2
    design).  Built once per (graph, endpoint batch).

    ``graph``: the sub-netlist (a TimingGraph on the device, schedule cached); ``pins``: original id of sub pin i;
    ``endpoints``: the batch's endpoints as sub pin ids; ``cell_x_rows`` / ``net_x_rows``: rows of the caller's
    feature matrices for ``schedule().cell_class`` / ``net_class``."""

    def __init__(self, graph, endpoints):
        full = graph.schedule()
        act = _reaches_endpoint(graph, endpoints)
        keep = act.bool()
        self.active = keep
        new_id = torch.cumsum(act, 0, dtype=torch.int64) - 1
        pins = torch.nonzero(keep).flatten()
        edges = {}
        for et, (s, d) in graph._edges.items():
            s, d = s.to(endpoints.device).long(), d.to(endpoints.device).long()
            k = keep[d]
            edges[et] = (new_id[s[k]].contiguous(), new_id[d[k]].contiguous())
        sub = TimingGraph(int(pins.numel()), edges["net"], edges["cell"])
        sub._edges = edges                                        # already on the device
        sub._levels = (full.level[pins].contiguous(), full.num_levels)
        self.graph = sub
        self.pins = pins.int().contiguous()
        self.endpoints = new_id[endpoints.long()].int().contiguous()
        sch = sub.schedule()
        self.cell_x_rows = self.pins[sch.cell_class.long()].contiguous()
        self.net_x_rows = self.pins[sch.net_class.long()].contiguous()
        self.n_active = int(pins.numel())
        self.fraction = self.n_active / max(graph.number_of_nodes(), 1)


class MaskCSR:
    """Sparse path masks (``path_masks``, verilog_parser_asap7.py:1368): CSR over map*map columns."""

    def __init__(self, indptr, cols, width):
        self.indptr = torch.as_tensor(indptr, dtype=torch.int32)
        self.cols = torch.as_tensor(cols, dtype=torch.int32)
        self.width = int(width)
        self.num_rows = int(self.indptr.numel()) - 1
        self._max_row = None

    def max_row_len(self):
        """Longest row (one host read per design; bounds the buffers of every row selection)."""
        if self._max_row is None:
            self._max_row = int((self.indptr[1:] - self.indptr[:-1]).max().item()) if self.num_rows else 0
        return self._max_row

    @staticmethod
    def from_sparse_coo(t):
        """From the reference's ``torch.sparse_coo_tensor`` of int64 ones."""
        t = t.coalesce()
        rows, cols = t.indices()
        order = torch.argsort(rows * t.shape[1] + cols)
        indptr = torch.zeros(t.shape[0] + 1, dtype=torch.int64)
        indptr[1:] = torch.cumsum(torch.bincount(rows, minlength=t.shape[0]), 0)
        return MaskCSR(indptr.to(torch.int32), cols[order].to(torch.int32), t.shape[1])

    def to(self, device):
        self.indptr = self.indptr.to(device, non_blocking=True)
        self.cols = self.cols.to(device, non_blocking=True)
        return self

    def select(self, rows):
        """-> MaskRows for the given path ids (``th.index_select(path_masks, 0, paths)``, train.py:500)."""
        return MaskRows(self, rows)

    def select_all(self):
        """Every row, in order (one design's endpoints in one batch, test.py:176)."""
        dev = self.indptr.device
        return MaskRows(self, torch.arange(self.num_rows, dtype=torch.int32, device=dev), identity=True)


def rasterize_path_masks(n, src, dst, level, endpoints, pin_xy, map_size):
    """GPU replacement of the host preprocessing behind ``path_masks`` (critical-path back-trace,
    verilog_parser_asap7.py:1433-1450, + bounding-box rasterisation, :1302-1369).

    src, dst: every pin-graph edge in insertion order (net edges then cell edges for the synthetic
    generator; whatever order the caller's nx.DiGraph was filled in); level: (n,) longest-path levels;
    endpoints: (T,) pin ids; pin_xy: (n,2) integer bins.  All CUDA tensors.  Returns a ``MaskCSR``
    on the device whose row t is bit-identical to the reference's sparse mask row."""
    import tm_lib
    dev = level.device
    tm_lib.require_cuda(level, "level")
    i32 = lambda t: t.to(device=dev, dtype=torch.int32).contiguous()      # noqa: E731
    src, dst, level, endpoints, pin_xy = i32(src), i32(dst), i32(level), i32(endpoints), i32(pin_xy)
    T, E = int(endpoints.numel()), int(src.numel())
    nb = tm_lib.ws_bytes("tm_mask_ws_bytes", n, T, map_size)
    ws = tm_lib.workspace(nb, dev)
    counts = torch.empty(max(T, 1), dtype=torch.int32, device=dev)
    tm_lib.call("tm_mask_count", n, E, src, dst, level, T, endpoints, pin_xy, map_size, counts, ws, nb, tm_lib.stream())
    counts = counts[:T]
    if T and int(counts.min().item()) < 0:
        raise RuntimeError("rasterize_path_masks: a pin on a critical path has no predecessor one level below "
                           "(the reference's find_critical_path would not terminate)")
    indptr = torch.zeros(T + 1, dtype=torch.int32, device=dev)
    indptr[1:] = torch.cumsum(counts, 0)
    nnz = int(indptr[-1].item()) if T else 0
    cols = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    tm_lib.call("tm_mask_fill", n, T, map_size, indptr, cols, ws, nb, tm_lib.stream())
    return MaskCSR(indptr, cols[:nnz], map_size * map_size)


class MaskRows:
    """A row selection of a MaskCSR -- ``th.index_select(path_masks, 0, paths)`` (train.py:500) -- in the two forms
    the fusion kernels read: the run-length form of the selected rows (forward) and their column-major transpose
    (backward pull).  Both are built by ``tm_mask_select`` on the device with no host synchronisation into
    buffers sized by bounds the host already knows, so ``rebuild()`` can be replayed inside a CUDA graph after the
    caller refreshed ``rows`` in place (a new shuffled endpoint batch costs O(1) host work)."""

    def __init__(self, csr, rows, identity=False):
        self.csr = csr
        dev = csr.indptr.device
        self.rows = torch.as_tensor(rows, dtype=torch.int32).to(dev).contiguous()
        self.T = int(self.rows.numel())
        self.identity = bool(identity)        # rows == arange(num_rows)
        self._buf = None

    def _alloc(self):
        csr, dev = self.csr, self.csr.indptr.device
        tm_lib.require_cuda(csr.indptr, "path masks")
        cap = int(csr.cols.numel()) if self.identity else self.T * csr.max_row_len()
        cap = max(cap, 1)
        i32 = lambda n: torch.empty(n, dtype=torch.int32, device=dev)      # noqa: E731
        nb = tm_lib.ws_bytes("tm_mask_select_ws", self.T, csr.width)
        self._buf = dict(run_ptr=i32(self.T + 1), run_lo=i32(cap), run_hi=i32(cap), csc_ptr=i32(csr.width + 1),
                         csc_t=i32(cap), ws=tm_lib.workspace(nb, dev), nb=nb)

    def rebuild(self):
        """(Re)run the selection kernels for the current contents of ``rows`` on the current stream."""
        if self._buf is None:
            self._alloc()
        b, csr = self._buf, self.csr
        tm_lib.call("tm_mask_select", self.T, csr.width, csr.indptr, csr.cols, self.rows, b["run_ptr"], b["run_lo"],
                    b["run_hi"], b["csc_ptr"], b["csc_t"], b["ws"], b["nb"], tm_lib.stream())
        self._built = True

    def _ensure(self):
        if self._buf is None or not getattr(self, "_built", False):
            self.rebuild()
        return self._buf

    def runs(self):
        """(run_ptr int32[T+1], run_lo, run_hi): endpoint t owns runs run_ptr[t]..run_ptr[t+1], run r covers columns
        [run_lo[r], run_hi[r]).  Needs ascending columns inside a row (the CSR convention)."""
        b = self._ensure()
        return b["run_ptr"], b["run_lo"], b["run_hi"]

    def csc(self):
        """(csc_ptr int32[J+1], csc_t): positions t (0..T-1, ascending) whose mask contains column j."""
        b = self._ensure()
        return b["csc_ptr"], b["csc_t"]
