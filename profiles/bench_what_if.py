"""What-if evaluation (IncrementalEvaluation.what_if -> WhatIf) against the update loop it replaces.

  design: config 2 (100k cells, 256x256 U-Net image), tm_synth seed 0, one design with all of its endpoints; U-Net in
          the default tf32x3 mode.
  cases:  K = 1, 8, 64 candidates x {one pin from the last quarter of the levels, eight such pins, one uniformly drawn
          scheduled pin} per candidate; every candidate's rows edited (cell-type swaps, new net features).
  variants, timed alternately (REPEATS rounds of CUDA events around ITERS calls, median in ms per call):
    what_if_replay : WhatIf.capture() replays: one CUDA graph scoring all K candidates
    update_loop    : per candidate, its rows written into the batch, a captured update (capture_update), the original
                     rows written back and the same captured update again (the revert) -- 2K updates
  breakdown: eager WhatIf.run phases with events between them (cone build = mark + plan + emit, self terms,
             propagation, head), median over ITERS calls; the cone build's kernels split by torch.profiler in a run of
             their own (mark vs plan + emit, device time per call).
  check: every candidate's row of the replay against the loop's captured update with that candidate's rows (bitwise).
Writes one JSON line (card name, power limit and clocks read in the same run) to --out and stdout.
Usage: python profiles/bench_what_if.py [--out profiles/r10_bench_what_if.json]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import bench_configs as bc  # noqa: E402

importlib.import_module(bc.PKG)
import tm_engine  # noqa: E402
import tm_lib  # noqa: E402
import tm_ops  # noqa: E402
import tm_synth  # noqa: E402
from tm_lib import call, stream  # noqa: E402

DEV = torch.device("cuda", 0)
REPEATS, ITERS = 5, 5
KS = (1, 8, 64)
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


def edit_rows(cf, nf, rng):
    """Cell-type one-hot swaps on rows carrying a cell type, new uniforms on rows carrying net features (in place)."""
    c, n = cf.cpu(), nf.cpu()
    oh = c[:, :NUM_CTYPES]
    out = oh.sum(1) == 1
    k = torch.argmax(oh, 1)
    j = (k + 1 + torch.from_numpy(rng.integers(0, NUM_CTYPES - 1, size=len(c)))) % NUM_CTYPES
    oh[out] = 0.0
    oh[out, j[out]] = 1.0
    sink = n.abs().sum(1) > 0
    n[sink] = torch.from_numpy(rng.random((int(sink.sum()), 2), dtype=np.float32))
    cf.copy_(c)
    nf.copy_(n)


def breakdown(wi):
    """Median ms of each phase of an eager WhatIf.run, events between the phases."""
    inc, c = wi.inc, wi.cones
    gp = inc._params()
    KT, Xw = wi.K * wi.T, wi._Xw
    width = Xw.shape[1]
    f0, f2 = inc.step.model.mlp_fuse.layers[0], inc.step.model.mlp_fuse.layers[2]

    def head():
        call("tm_gather_cols", KT, tm_ops.D, inc.H_ext, tm_ops.D, c.head_rows, Xw, width, 0, stream())
        call("tm_gather_cols", KT, width - tm_ops.D, inc.X[:, tm_ops.D:], width, wi._img_rows, Xw, width, tm_ops.D,
             stream())
        tm_ops.mlp2_forward(Xw, width, None, KT, f0.weight.detach(), f0.bias.detach(), f2.weight.detach(),
                            f2.bias.detach(), wi._pred2, 1)
        call("tm_what_if_mask", wi.K, wi.T, c.fitted, wi._pred2, stream())
    phases = {"cone_build": lambda: c.build(wi._seed_ptr, wi._seeds, wi._seed_slot, inc.S_ext),
              "self_terms": lambda: tm_ops.gnn_self_terms(inc.S_ext, wi.cell_feat, wi.net_feat, gp, wi._x_cell,
                                                          wi._x_net, cell_out=c.seed_rows[:wi._nc],
                                                          net_out=c.seed_rows[wi._nc:]),
              "propagation": lambda: tm_ops.gnn_forward_cone(c, inc.H_ext, inc.S_ext, gp),
              "head": head}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)]
    t = {k: [] for k in phases}
    for it in range(ITERS + 2):
        ev[0].record()
        for i, fn in enumerate(phases.values()):
            fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        if it >= 2:
            for i, k in enumerate(phases):
                t[k].append(ev[i].elapsed_time(ev[i + 1]))
    out = {k: statistics.median(v) for k, v in t.items()}
    # the cone build's three kernels, by device time (a profiled run of its own)
    n_prof = 5
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            phases["cone_build"]()
        torch.cuda.synchronize()
    ks = {"mark": 0.0, "plan": 0.0, "emit": 0.0}
    for e in prof.key_averages():
        dt = getattr(e, "device_time_total", None)
        dt = e.cuda_time_total if dt is None else dt
        for k in ks:
            if f"cones_{k}_kernel" in e.key:
                ks[k] += dt / 1000.0 / n_prof
    out["kernels_ms"] = ks
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_bench_what_if.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    model, net = tm_engine.build_models(d.map_size, seed=0, device=DEV)
    step = tm_engine.DesignStep(model, net)
    b = tm_engine.DesignBatch.from_host(tm_engine.HostDesign(d, pin=True), DEV)
    torch.cuda.synchronize()
    sched = b.graph.schedule()
    R = 8 * sched.n_sched
    inc = step.incremental(b, what_if_rows=R)
    lv = sched.level.cpu().numpy()
    L = sched.num_levels
    scheduled = np.nonzero(lv >= 0)[0]
    late = np.nonzero(lv >= (3 * L) // 4)[0]
    rng = np.random.default_rng(0)
    pool = torch.cuda.graph_pool_handle()
    res = {"card": card(), "repeats": REPEATS, "iters": ITERS,
           "model": "U-Net tf32x3, all endpoints of the design", "design": "tm_synth c2 seed 0",
           "pins": int(sched.n), "scheduled_pins": int(sched.n_sched), "levels": L,
           "endpoints": int(b.endpoints.numel()), "what_if_rows": R, "max_in_degree": inc.max_in_degree(),
           "cases": {}}
    for K in KS:
        for draw, src, per in (("late1", late, 1), ("late8", late, 8), ("uniform1", scheduled, 1)):
            sets = [np.sort(rng.choice(src, per, replace=False)) for _ in range(K)]
            wi = inc.what_if(sets)
            edit_rows(wi.cell_feat, wi.net_feat, rng)
            replay = wi.capture(pool=pool)
            got = replay().clone()
            # the loop it replaces: per candidate a captured update with its rows, then one with the original rows
            idx = [torch.from_numpy(s).to(DEV) for s in sets]
            orig = [(b.cell_feat[i].clone(), b.net_feat[i].clone()) for i in idx]
            cand = [wi.rows(k) for k in range(K)]
            ups = [inc.capture_update(s, pool=pool) for s in sets]

            def loop():
                for k in range(K):
                    b.cell_feat.index_copy_(0, idx[k], cand[k][1])
                    b.net_feat.index_copy_(0, idx[k], cand[k][2])
                    ups[k]()
                    b.cell_feat.index_copy_(0, idx[k], orig[k][0])
                    b.net_feat.index_copy_(0, idx[k], orig[k][1])
                    ups[k]()
            same = True
            for k in range(K):
                b.cell_feat.index_copy_(0, idx[k], cand[k][1])
                b.net_feat.index_copy_(0, idx[k], cand[k][2])
                p = ups[k]().clone()
                b.cell_feat.index_copy_(0, idx[k], orig[k][0])
                b.net_feat.index_copy_(0, idx[k], orig[k][1])
                ups[k]()
                same = same and bool(torch.equal(p.view(torch.int32), got[k].view(torch.int32)))
            t = ab({"what_if_replay": replay, "update_loop": loop})
            sizes = wi.cone_sizes()
            wi.run()
            bd = breakdown(wi)
            phase_sum = sum(v for k, v in bd.items() if k != "kernels_ms")
            case = {"K": K, "pins_per_candidate": per, "admitted": int(wi.fitted().sum()),
                    "cone_pins_mean": float(sizes.mean()), "cone_pins_total": int(sizes.sum()),
                    "cone_fraction_mean": float(sizes.mean()) / sched.n_sched,
                    "joined_nonempty_levels": int((np.diff(wi.cones.level_ptr.cpu().numpy()) > 0).sum()),
                    "ms_per_call": t, "loop_over_what_if": t["update_loop"] / t["what_if_replay"],
                    "what_if_vs_update_loop_bitwise": same, "eager_breakdown_ms": bd,
                    "head_share_of_eager": bd["head"] / phase_sum}
            res["cases"][f"K{K}_{draw}"] = case
            print(json.dumps({f"K{K}_{draw}": case}), flush=True)
            del ups
    step.close()
    tm_lib.check_err_flags()
    line = json.dumps(res)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line, flush=True)


if __name__ == "__main__":
    main()
