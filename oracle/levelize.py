"""Integer side of the oracle: level construction, CSR, critical-path masks.

Oracle / test infrastructure only (see oracle/__init__.py).  Plain-Python and
numpy restatements of

* ``Parser.cal_topo_level``      verilog_parser_asap7.py:1452-1517
* ``Parser.find_critical_path``  verilog_parser_asap7.py:1433-1450
* path-mask rasterisation        verilog_parser_asap7.py:1302-1369
* the in-edge CSR that DGL builds lazily inside ``pull``  (dataset.py:274-278,
  model.py:186-204)

Pinned against the reference's own ``cal_topo_level`` / ``find_critical_path``
source, executed from the original project on networkx graphs
(``oracle/make_golden.py`` -> ``tests/golden/levels_*.npz``,
``tests/test_oracle_pinning.py``).
"""
import numpy as np


# ---------------------------------------------------------------------------
# level construction
# ---------------------------------------------------------------------------
def topo_levels_frontier(n, src, dst, pis, pos=(), po2path=None):
    """Frontier restatement of cal_topo_level (verilog_parser_asap7.py:1468-1517).

    Forward sweep: frontier k+1 = set of successors of frontier k, starting at
    the PI set (:1469-1490).  Reverse sweep: every pin is kept only in the LAST
    frontier it appears in (:1494-1511).  Pins never reached are dropped
    (:1514-1515).  Returns ``(levels, removed)`` where ``levels`` is a list of
    ``(sorted nodes, sorted targets, path_ids)`` -- the reference's order inside
    a level is Python-set iteration order, i.e. undefined, so it is
    canonicalised to ascending here.
    """
    succ = [[] for _ in range(n)]
    for s, d in zip(np.asarray(src).tolist(), np.asarray(dst).tolist()):
        succ[s].append(d)
    pos = set(int(p) for p in pos)
    po2path = po2path or {}
    frontiers = [set(int(p) for p in pis)]
    reached = set(frontiers[0])
    cur = frontiers[0]
    while True:
        nxt = set()
        for nd in cur:
            nxt.update(succ[nd])
        if not nxt:
            break
        frontiers.append(nxt)
        reached |= nxt
        cur = nxt
    visited = set()
    out = []
    for fr in reversed(frontiers):
        keep = fr - visited
        visited |= keep
        tg = sorted(pos & keep)
        out.append((sorted(keep), tg, [po2path[t] for t in tg if t in po2path]))
    out.reverse()
    removed = sorted(set(range(n)) - reached)
    return out, removed


def node_levels(n, src, dst, pis):
    """node -> level (int32, -1 for dropped pins): numpy form of the same rule.

    ``level(v)`` = length of the longest walk from any PI to ``v`` over pins
    reachable from the PI set -- what the last-frontier rule of
    verilog_parser_asap7.py:1494-1511 yields on a DAG.  Computed as Kahn
    peeling restricted to the reachable sub-graph.
    """
    src = np.asarray(src, dtype=np.int64)
    dst = np.asarray(dst, dtype=np.int64)
    order = np.argsort(src, kind="stable")
    optr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(src, minlength=n), out=optr[1:])
    odst = dst[order]

    def out_edges(nodes):
        cnt = optr[nodes + 1] - optr[nodes]
        tot = int(cnt.sum())
        if tot == 0:
            return np.zeros(0, dtype=np.int64)
        base = np.repeat(optr[nodes], cnt)
        off = np.arange(tot) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        return odst[base + off]

    reach = np.zeros(n, dtype=bool)
    fr = np.unique(np.asarray(list(pis), dtype=np.int64))
    reach[fr] = True
    while fr.size:
        nb = np.unique(out_edges(fr))
        nb = nb[~reach[nb]]
        reach[nb] = True
        fr = nb
    keep = reach[src] & reach[dst]
    indeg = np.bincount(dst[keep], minlength=n)
    level = np.full(n, -1, dtype=np.int32)
    fr = np.nonzero(reach & (indeg == 0))[0]
    k = 0
    while fr.size:
        level[fr] = k
        nb = out_edges(fr)
        if nb.size:
            dec = np.bincount(nb, minlength=n)
            indeg -= dec
            cand = np.unique(nb)
            fr = cand[indeg[cand] == 0]
        else:
            fr = nb
        k += 1
    return level


def in_csr(n, src, dst):
    """In-edge CSR with source ids ascending inside every row.

    ``indptr`` int32 (n+1), ``indices`` int32 (E).  This is the gather structure
    DGL derives from the ``(src, dst)`` lists of one edge type
    (dataset.py:274-278) when ``pull`` asks for the in-edges of a pin
    (model.py:186,203).  Mailbox order only changes fp32 summation order, so the
    row order is canonicalised to ascending source id (duplicates kept).
    """
    src = np.asarray(src, dtype=np.int64)
    dst = np.asarray(dst, dtype=np.int64)
    order = np.lexsort((src, dst))
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(dst, minlength=n), out=indptr[1:])
    return indptr.astype(np.int32), src[order].astype(np.int32)


# ---------------------------------------------------------------------------
# critical-path trace and path masks
# ---------------------------------------------------------------------------
def find_critical_path(endpoint, level, preds):
    """verilog_parser_asap7.py:1433-1450 without the clock-name escape.

    ``preds[v]`` lists predecessors in edge-insertion order (what
    ``networkx.DiGraph.predecessors`` iterates).  Walk back from the endpoint,
    at each step taking the FIRST predecessor that sits exactly one level lower,
    until the level drops below 2.
    """
    cur, cur_level = int(endpoint), int(level[endpoint])
    path = [cur]
    while cur_level >= 2:
        for nd in preds[cur]:
            if level[nd] == cur_level - 1:
                path.append(nd)
                cur_level -= 1
                cur = nd
                break
        else:
            raise RuntimeError("no predecessor one level below (reference would spin forever)")
    return path


def path_mask_columns(path, pin_xy, map_size):
    """verilog_parser_asap7.py:1315-1333,1351: union of the bin bounding boxes of
    consecutive pins on the path; column index = x*map_size + y; deduplicated."""
    cols = set()
    for a, b in zip(path[:-1], path[1:]):
        (ax, ay), (bx, by) = pin_xy[a], pin_xy[b]
        x1, x2 = min(ax, bx), max(ax, bx)
        y1, y2 = min(ay, by), max(ay, by)
        for x in range(int(x1), int(x2) + 1):
            cols.update(range(x * map_size + int(y1), x * map_size + int(y2) + 1))
    return sorted(cols)


def path_masks_csr(endpoints, level, n, src, dst, pin_xy, map_size):
    """Mask CSR (indptr int32, cols int32 ascending) for a list of endpoints."""
    preds = [[] for _ in range(n)]
    for s, d in zip(np.asarray(src).tolist(), np.asarray(dst).tolist()):
        preds[d].append(s)
    indptr, cols = [0], []
    for e in endpoints:
        c = path_mask_columns(find_critical_path(e, level, preds), pin_xy, map_size)
        cols.extend(c)
        indptr.append(len(cols))
    return np.asarray(indptr, dtype=np.int32), np.asarray(cols, dtype=np.int32)
