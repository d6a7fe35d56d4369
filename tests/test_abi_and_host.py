"""CPU-side tests: the C ABI is loadable and complete, and the host logic around it."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG, ROOT
import tm_lib
import tm_synth


def test_library_exports_every_declared_symbol():
    sigs = tm_lib.parse_header()
    assert len(sigs) >= 40
    l = ctypes.CDLL(tm_lib.LIB_PATH)
    for name in sigs:
        assert hasattr(l, name), f"{name} declared in include/tm_b200.h but not exported"
    # and nothing is exported that the header does not declare
    out = subprocess.run(["nm", "-D", "--defined-only", tm_lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (tm_\w+)", out))
    assert exported == set(sigs), exported ^ set(sigs)


def test_library_loads_without_gpu_and_reports_errors():
    l = tm_lib.lib()
    assert l.tm_version() >= 100
    assert tm_lib.launch_count() >= 0
    assert tm_lib.ws_bytes("tm_csr_build_ws", 1000, 5000) > 8000
    assert tm_lib.ws_bytes("tm_gemm_tn_ws", 256, 128, 100000) > 256 * 128 * 4
    with pytest.raises(RuntimeError, match="bad sizes"):
        tm_lib.call("tm_csr_build", -1, 0, None, None, None, None, None, 0, None)


def test_schedule_struct_layout_matches_header():
    text = open(tm_lib.HEADER_PATH).read()
    body = re.search(r"typedef struct \{(.*?)\} tm_schedule;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"(\w+)\s*;", body)
    assert names == [f[0] for f in tm_lib.tm_schedule._fields_]
    assert ctypes.sizeof(tm_lib.tm_schedule) == 8 + 4 + 4 + 21 * 8


def test_cuda_sources_target_sm100a_only():
    mk = open(os.path.join(PKG, "csrc", "Makefile")).read()
    assert "arch=compute_100a,code=sm_100a" in mk and "-lineinfo" in mk
    for f in os.listdir(os.path.join(PKG, "csrc")):
        if f.endswith((".cu", ".cuh")):
            src = open(os.path.join(PKG, "csrc", f)).read()
            assert "triton" not in src.lower()


def _strip_c_comments(src):
    """Source text with // and /* */ comments blanked out; string and character literals are kept."""
    return re.sub(r'//[^\n]*|/\*.*?\*/|("(?:\\.|[^"\\])*"|\'(?:\\.|[^\'\\])*\')',
                  lambda m: m.group(1) or " ", src, flags=re.S)


def _asm_statements(src):
    """The concatenated string literals of every asm statement in comment-free source."""
    out = []
    for m in re.finditer(r"\basm\b(\s+volatile\b)?\s*\(", src):
        depth, i = 1, m.end()
        while depth:
            c = src[i]
            if c == '"':
                i = re.compile(r'"(?:\\.|[^"\\])*"').match(src, i).end()
                continue
            depth += (c == "(") - (c == ")")
            i += 1
        out.append("".join(re.findall(r'"((?:\\.|[^"\\])*)"', src[m.end():i])))
    return out


def test_sm100_primitives_are_defined_once():
    """mbarrier / tcgen05 / async-proxy PTX and the fp16 split live in tm_sm100.cuh and tm_split.cuh only."""
    csrc = os.path.join(PKG, "csrc")
    srcs = {f: _strip_c_comments(open(os.path.join(csrc, f)).read())
            for f in sorted(os.listdir(csrc)) if f.endswith((".cu", ".cuh"))}
    assert "tm_sm100.cuh" in srcs and "tm_split.cuh" in srcs
    forbidden = ("mbarrier.", "tcgen05.", "fence.proxy.async", "fence.mbarrier_init",
                 "cp.async.bulk.shared::cluster.global")
    n_asm = 0
    for f, src in srcs.items():
        for stmt in _asm_statements(src):
            n_asm += 1
            if f != "tm_sm100.cuh":
                assert not any(k in stmt for k in forbidden), f"{f}: {stmt}"
    assert n_asm > 20
    defs = {
        "LO_SCALE": r"\bLO_SCALE\s*=",
        "split_h": r"\bsplit_h\s*\([^;{}]*\)\s*\{",
        "__cvta_generic_to_shared": r"\b__cvta_generic_to_shared\b",
    }
    for name, pat in defs.items():
        where = [f for f, src in srcs.items() if re.search(pat, src)]
        assert len(where) == 1, f"{name} is defined in {where}"


def test_product_never_imports_oracle():
    for f in os.listdir(PKG):
        if f.endswith(".py"):
            src = open(os.path.join(PKG, f)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f


@pytest.mark.parametrize("cfg", ["tiny", "c1"])
def test_synthetic_design_invariants(cfg):
    d = tm_synth.make_design(seed=1, **tm_synth.CONFIGS[cfg])
    lv = d.level
    assert (lv >= 0).all() and d.num_levels == 2 * d.meta["n_lv"] + 1
    assert (lv[d.net_src] < lv[d.net_dst]).all() and (lv[d.cell_src] < lv[d.cell_dst]).all()
    assert (lv[d.net_dst] % 2 == 1).all() and (lv[d.cell_dst] % 2 == 0).all()
    assert (lv[d.pis] == 0).all() and (lv[d.endpoints] % 2 == 1).all()
    assert len(set(d.endpoints.tolist())) == d.endpoints.size
    assert (np.diff(lv[d.endpoints]) >= 0).all()                       # grouped by level
    for i in range(0, d.endpoints.size, 97):
        row = d.mask_cols[d.mask_indptr[i]:d.mask_indptr[i + 1]]
        assert (np.diff(row) > 0).all() and (row < d.map_size ** 2).all()
    d2 = tm_synth.make_design(seed=1, **tm_synth.CONFIGS[cfg])
    assert np.array_equal(d.net_src, d2.net_src) and np.array_equal(d.image, d2.image)   # seeded
    tl = d.topo_levels()
    assert sum(len(x[0]) for x in tl) == d.n and sum(len(x[1]) for x in tl) == d.endpoints.size
    p2l, p2e = d.path_dicts()
    assert all(p2e[p] == t for nodes, tg, pids in tl for t, p in zip(tg, pids))


def test_timing_graph_surface_and_no_cpu_path():
    import tm_graph
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["tiny"])
    g = tm_graph.TimingGraph(d.n, (d.net_src, d.net_dst), (d.cell_src, d.cell_dst), pis=d.pis)
    g.ndata["h"] = torch.zeros(d.n, 128)
    assert g.nodes["pin"].data is g.ndata
    g.nodes["pin"].data["h"][[1, 2]] = 1.0                              # model.py:208-style row write
    assert float(g.ndata["h"].sum()) == 256.0
    g.edges["cell"].data["a"] = torch.zeros(g.number_of_edges(etype="cell"), 1)
    assert g.number_of_nodes() == d.n and g.number_of_edges(etype="net") == d.net_src.size
    src, dst = g.edges(etype="net")
    assert torch.equal(src, torch.from_numpy(d.net_src))
    assert tm_graph.as_timing_graph(g) is g
    with pytest.raises(RuntimeError, match="CUDA"):
        g.schedule()


def test_mask_csr_from_reference_sparse_format():
    import tm_graph
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["tiny"])
    rows = np.repeat(np.arange(d.endpoints.size), np.diff(d.mask_indptr))
    perm = np.random.default_rng(0).permutation(rows.size)                # uncoalesced order
    coo = torch.sparse_coo_tensor(np.stack([rows[perm], d.mask_cols[perm].astype(np.int64)]),
                                  torch.ones(rows.size, dtype=torch.int64), (d.endpoints.size, d.map_size ** 2))
    c = tm_graph.MaskCSR.from_sparse_coo(coo)
    assert torch.equal(c.indptr, torch.from_numpy(d.mask_indptr))
    assert torch.equal(c.cols, torch.from_numpy(d.mask_cols))


def test_module_state_dict_names_match_reference_fixture():
    """Parameter names / shapes of the drop-in modules == the reference's (golden fixture keys)."""
    from conftest import load_golden_step
    import tm_engine
    z, sd_m, sd_c = load_golden_step("tiny")
    model, cnn = tm_engine.build_models(8, device="cpu")
    assert {k: tuple(v.shape) for k, v in model.state_dict().items()} == {k: tuple(v.shape) for k, v in sd_m.items()}
    assert {k: tuple(v.shape) for k, v in cnn.state_dict().items()} == {k: tuple(v.shape) for k, v in sd_c.items()}
    model.load_state_dict(sd_m)
    cnn.load_state_dict(sd_c)
    # seeded construction reproduces the reference's initial weights (same creation order)
    torch.manual_seed(0)
    import model as M
    gnn = M.PathConv(out_feat_dim=128, hidden_feat_dim=128, cell_feat_dim=36, net_feat_dim=2)
    assert torch.equal(gnn.fc_cell_neigh.layers[0].weight, sd_m["gnn.fc_cell_neigh.layers.0.weight"])
    assert torch.equal(gnn.fc_attn2.weight, sd_m["gnn.fc_attn2.weight"])


def test_modules_pickle_roundtrip():
    import pickle
    import tm_engine
    model, cnn = tm_engine.build_models(8, device="cpu")
    m2, c2 = pickle.loads(pickle.dumps((model, cnn)))                     # train.py:86-89 format
    assert type(m2).__module__ == "model" and type(c2).__module__ == "Unet"
    assert torch.equal(m2.fcn.weight, model.fcn.weight)


DP_SCRIPT = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
import tm_dp
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
torch.manual_seed(0)
params = [torch.nn.Parameter(torch.zeros(3, 5)), torch.nn.Parameter(torch.zeros(7)), torch.nn.Parameter(torch.zeros(2, 2))]
for i, p in enumerate(params):
    p.grad = torch.full_like(p, float(rank + 1) * (i + 1))
params[1].grad = None                                  # unused parameter (fc_net_drive-like, D12)
b = tm_dp.GradBucket(params, world)
work = b.post(None)
b.finish(work)
flat_ptr = b.flat.data_ptr()
for i, p in enumerate(params):
    if p.grad is not None:
        assert p.grad.data_ptr() >= flat_ptr                # .grad is a view of the persistent flat buffer
exp = sum(r + 1 for r in range(world)) / world
assert torch.allclose(params[0].grad, torch.full((3, 5), exp)), params[0].grad
assert params[1].grad is None
assert torch.allclose(params[2].grad, torch.full((2, 2), 3 * exp))
shard = tm_dp.shard_designs(list(range(10)), rank, world)
assert shard == list(range(rank, 10, world))
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
'''


def test_data_parallel_buckets_gloo_world2(tmp_path):
    script = tmp_path / "dp.py"
    script.write_text(DP_SCRIPT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29613")
    procs = [subprocess.Popen([sys.executable, str(script), PKG], env=dict(env, RANK=str(r), WORLD_SIZE="2"),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_loader_reference_semantics(tmp_path):
    """tm_loader.load_single_design == the reference function (train.py:335-388) on a synthetic design written in
    the reference's tuple format: feat_reduce trim 42/3 -> 36/2, ndata['h'] / edata['a'] zeros, min-max norm from
    column num_ctypes on, critical-path oversampling (os_rate x when negatives outnumber positives 2:1), the 1/5
    validation split written once and reused; LoadedDesign orders a batch like the reference loop (levels ascending,
    DataLoader order inside a level)."""
    import tm_loader
    import tm_synth
    d = tm_synth.make_design(seed=3, **tm_synth.CONFIGS["tiny"])
    tup = tm_loader.design_tuple_from_synth(d, seed=1)
    tm_loader.save_design(str(tmp_path / "x.pkl"), tup)
    raw_cf = tup[0].ndata["cell_feat"].clone()
    ds, g, p2l, p2e, tl, img, pm = tm_loader.load_single_design("train", str(tmp_path), "x", 128, 2, [6, 1], False)
    P, crit = len(d.endpoints), tup[5]
    assert len(ds) == P + 2 * len(crit) and ds.paths[P:P + len(crit)] == crit
    assert torch.equal(g.ndata["cell_feat"], raw_cf[:, :-6]) and g.ndata["net_feat"].shape[1] == 2
    assert g.ndata["h"].shape == (d.n, 128) and float(g.ndata["h"].abs().sum()) == 0.0
    assert g.edges["cell"].data["a"].shape == (len(d.cell_src), 1)
    assert isinstance(img, torch.Tensor) and img.dtype == torch.float32 and tuple(pm.shape) == (P, d.map_size ** 2)
    # norm: columns >= num_ctypes scaled to [0, 1] by their own min / max, the one-hot block untouched
    gn = tm_loader.load_single_design("train", str(tmp_path), "x", 128, 0, [6, 1], True)[1]
    cf = gn.ndata["cell_feat"]
    assert torch.equal(cf[:, :34], raw_cf[:, :34])
    col = raw_cf[:, 35]
    assert torch.allclose(cf[:, 35], (col - col.min()) / (col.max() - col.min()))
    # test usage: split written once, then reused
    v1 = tm_loader.load_single_design("test", str(tmp_path), "x", 128, 1, [6, 1], False)[0].paths
    v2 = tm_loader.load_single_design("test", str(tmp_path), "x", 128, 1, [6, 1], False)[0].paths
    assert v1 == v2 and abs(len(v1) - P // 5) <= 2 and (tmp_path / "x_split.pkl").exists()
    # batch order of the fused path == order of the reference loop's predictions
    ld = tm_loader.LoadedDesign(str(tmp_path / "x.pkl"), "cpu")
    ids = [7, 3, 11, 0, 3, 25]
    want = []
    for lid in range(len(tl)):
        want += [p for p in ids if p2l[p] == lid]
    assert ld.order_batch(ids).tolist() == want
