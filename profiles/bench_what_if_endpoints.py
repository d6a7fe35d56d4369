"""What-if restricted to chosen endpoints (inc.what_if(pin_sets, endpoints=E)) against the unrestricted what_if.

  design: config 2 (100k cells, 256x256 U-Net image), tm_synth seed 0, one design with all of its endpoints; U-Net in
          the default tf32x3 mode; what_if_rows = n (one row per pin).
  E:      the 1, 8 and 64 endpoints with the largest prediction, the 64 endpoints on the deepest levels, all endpoints.
  candidates: K = 8 and 64 single-pin candidates, drawn by the norm of the input gradient of sum(pred[E]) (as an
          optimisation loop draws them) and uniformly from R(E), E's fan-in cone; each candidate's rows get a cell-type
          swap / new net features (one vectorised edit, no host reads).
  variants, timed alternately (REPEATS rounds of CUDA events around ITERS captured replays, median ms per call):
    restricted   : wi = inc.what_if(sets, endpoints=E), wi.capture() -> (K, T_E)
    unrestricted : wi = inc.what_if(sets), wi.capture() -> (K, T)
  per case: admitted candidates, mean cone pins, |R(E)|, and whether every restricted row is bitwise equal to the
          unrestricted row at E (rows the unrestricted call admitted).
  loop:   one optimisation iteration on the top-64 objective -- captured input gradient, what_if over the 64 pins with
          the largest gradient norm (the same vectorised edit), commit of the admitted candidate with the lowest
          objective -- host clock around the iteration ending in a device synchronise, median of ITERS iterations,
          with the restricted and with the unrestricted what_if.
Writes one JSON line (card name, power limit and clocks read in the same run) to --out and stdout.
Usage: python profiles/bench_what_if_endpoints.py [--out profiles/r12_bench_what_if_endpoints.json]
"""
import argparse
import gc
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import bench_configs as bc  # noqa: E402

importlib.import_module(bc.PKG)
import tm_engine  # noqa: E402
import tm_graph  # noqa: E402
import tm_lib  # noqa: E402
import tm_synth  # noqa: E402

DEV = torch.device("cuda", 0)
REPEATS, ITERS = 5, 5
NUM_CTYPES = 34


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def events(fn, iters=ITERS):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def ab(variants):
    for fn in variants.values():
        fn()
    torch.cuda.synchronize()
    t = {k: [] for k in variants}
    for _ in range(REPEATS):
        for k, fn in variants.items():
            t[k].append(events(fn))
    return {k: statistics.median(v) for k, v in t.items()}


def edit_rows(cf, nf, gen):
    """Every row at once: a cell-type swap where the row carries one cell type, new uniforms where it carries net
    features; device work only."""
    oh = cf[:, :NUM_CTYPES]
    has = oh.sum(dim=1) == 1.0
    shift = torch.randint(1, NUM_CTYPES, (cf.shape[0],), device=cf.device, generator=gen)
    j = (torch.argmax(oh, dim=1) + shift) % NUM_CTYPES
    new = torch.nn.functional.one_hot(j, NUM_CTYPES).to(cf.dtype)
    oh.copy_(torch.where(has[:, None], new, oh))
    net = nf.abs().sum(dim=1) > 0
    nf.copy_(torch.where(net[:, None], torch.rand(nf.shape, device=nf.device, generator=gen), nf))


def grad_pins(inc, T, E, k):
    seed = torch.zeros(T, dtype=torch.float32, device=DEV)
    seed[torch.from_numpy(E).to(DEV)] = 1.0
    g = inc.input_grads(seed)
    norm = g["cell_feat"].norm(dim=1) + g["net_feat"].norm(dim=1)
    return torch.topk(norm, k).indices.cpu().numpy()


def within_pins(b, E):
    fan = tm_graph.FaninCone(b.graph, keep_bits=True)
    fan.build(b.endpoints[torch.from_numpy(E).to(DEV)].contiguous(), torch.ones(E.size, device=DEV))
    n = b.graph.number_of_nodes()
    w = fan.bits.cpu().numpy().view(np.uint32)
    return np.nonzero((w[np.arange(n) >> 5] >> (np.arange(n) & 31).astype(np.uint32)) & 1)[0]


def case(inc, E, pins, gen):
    sets = [[int(p)] for p in pins]
    wr, wu = inc.what_if(sets, endpoints=E), inc.what_if(sets)
    edit_rows(wr.cell_feat, wr.net_feat, gen)
    wu.cell_feat.copy_(wr.cell_feat)
    wu.net_feat.copy_(wr.net_feat)
    rr, ru = wr.capture(), wu.capture()
    t = ab({"restricted": rr, "unrestricted": ru})
    pr, pu = rr().clone(), ru().clone()
    fr, fu = wr.fitted(), wu.fitted()
    both = torch.from_numpy(fr & fu).to(DEV)
    Et = torch.from_numpy(wr.endpoints).to(DEV)
    same = torch.equal(pr[both].view(torch.int32), pu[both][:, Et].view(torch.int32))
    sr, su = wr.cone_sizes(), wu.cone_sizes()
    out = {"K": len(sets), "T_E": int(E.size), "ms_per_call": t, "unrestricted_over_restricted":
           t["unrestricted"] / t["restricted"], "admitted": {"restricted": int(fr.sum()), "unrestricted": int(fu.sum())},
           "mean_cone_pins": {"restricted": float(sr.mean()), "unrestricted": float(su.mean())},
           "within_size": wr.within_size(), "rows_compared": int(both.sum()), "bitwise_equal_at_E": bool(same)}
    del rr, ru, wr, wu
    gc.collect()
    return out


def loop_iteration(inc, T, E, seed, grads, gen, restricted, n_cand=64):
    """gradient -> what_if over the n_cand pins with the largest gradient norm -> commit the best; host seconds."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    g = grads()
    norm = g["cell_feat"].norm(dim=1) + g["net_feat"].norm(dim=1)
    pins = torch.topk(norm, n_cand).indices.cpu().numpy()
    wi = inc.what_if([[int(p)] for p in pins], endpoints=E if restricted else None)
    edit_rows(wi.cell_feat, wi.net_feat, gen)
    pred = torch.nan_to_num(wi.run(), nan=0.0)
    obj = pred.sum(dim=1) if restricted else pred @ seed
    fitted = torch.from_numpy(wi.fitted()).to(obj.device)
    k = int(torch.argmin(torch.where(fitted, obj, torch.full_like(obj, float("inf")))).item())
    wi.commit(k)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, int(fitted.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_bench_what_if_endpoints.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    model, net = tm_engine.build_models(d.map_size, seed=0, device=DEV)
    step = tm_engine.DesignStep(model, net)
    b = tm_engine.DesignBatch.from_host(tm_engine.HostDesign(d, pin=True), DEV)
    torch.cuda.synchronize()
    sched = b.graph.schedule()
    n = int(sched.n)
    inc = step.incremental(b, what_if_rows=n)
    T = int(b.endpoints.numel())
    rng = np.random.default_rng(0)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(0)
    res = {"card": card(), "repeats": REPEATS, "iters": ITERS,
           "model": "U-Net tf32x3, all endpoints of the design", "design": "tm_synth c2 seed 0",
           "pins": n, "scheduled_pins": int(sched.n_sched), "levels": sched.num_levels, "endpoints": T,
           "what_if_rows": n, "cases": {}}
    order = torch.argsort(inc.pred, descending=True).cpu().numpy()
    deep = torch.argsort(b.endpoint_level.reshape(-1), descending=True, stable=True).cpu().numpy()
    objectives = {"top1": order[:1], "top8": order[:8], "top64": order[:64], "deepest64": deep[:64],
                  "all": np.arange(T)}
    for oname, E in objectives.items():
        E = np.sort(E)
        inside = within_pins(b, E)
        for K in (8, 64):
            for draw in ("grad", "uniform"):
                if draw == "grad":
                    pins = grad_pins(inc, T, E, K)
                else:
                    pins = rng.choice(inside, K, replace=inside.size < K)
                name = f"{oname}/K{K}/{draw}"
                res["cases"][name] = c = case(inc, E, pins, gen)
                print(json.dumps({name: c}), flush=True)
    # one optimisation iteration on the top-64 objective
    E = np.sort(objectives["top64"])
    seed = torch.zeros(T, dtype=torch.float32, device=DEV)
    seed[torch.from_numpy(E).to(DEV)] = 1.0
    grads = inc.capture_input_grads(seed)
    loop, admitted = {"restricted": [], "unrestricted": []}, {"restricted": [], "unrestricted": []}
    for it in range(ITERS + 1):
        for k in ("restricted", "unrestricted"):
            dt, n_adm = loop_iteration(inc, T, E, seed, grads, gen, k == "restricted")
            if it >= 1:
                loop[k].append(dt * 1e3)
                admitted[k].append(n_adm)
    res["loop_ms"] = {k: statistics.median(v) for k, v in loop.items()}
    res["loop_candidates_admitted"] = admitted
    print(json.dumps({"loop_ms": res["loop_ms"], "admitted": admitted}), flush=True)
    step.close()
    tm_lib.check_err_flags()
    line = json.dumps(res)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line, flush=True)


if __name__ == "__main__":
    main()
