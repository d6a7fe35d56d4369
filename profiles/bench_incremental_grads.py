"""Incremental input gradients (IncrementalEvaluation.input_grads) against the frozen step they replace.

  design: config 2 (100k cells, 256x256 U-Net image), tm_synth seed 0, one design with all of its endpoints; U-Net in
          the default tf32x3 mode.
  seeds:  1.0 on the 1, 8 and 64 endpoints with the largest predicted arrival, on the 1 and 64 endpoints on the
          deepest levels, on 64 uniformly drawn endpoints, and on all T endpoints.
  variants, timed alternately (REPEATS rounds of CUDA events around ITERS replays, median in ms per call):
    cone_replay   : inc.capture_input_grads(seed) replays (feature gradients only: the image branch is frozen in inc)
    frozen_replay : step.capture(batch, input_grads=True, pred_grad=seed, param_grads=False) replays (also the image
                    gradient and the whole forward)
  detail: the cone's pins and fraction of the scheduled pins; the eager call's phases with events between them (cone
          build, head data gradient, G / result zeroing + scatter, A / LSE / HID recompute, backward sweep, self-MLP
          data gradients), median over ITERS calls.
  check:  the cone call's gradients against the frozen step's, max relative error (different back ends: fp32 class).
  loop:   one optimisation iteration -- gradient, what_if over the 64 pins with the largest feature-gradient norm (each
          candidate one pin, cell-type swap / new net features), commit of the admitted candidate with the lowest
          seeded objective -- host clock around the iteration ending in a device synchronise, median of ITERS iterations, for
          the cone call and for the frozen step as the gradient.
Writes one JSON line (card name, power limit and clocks read in the same run) to --out and stdout.
Usage: python profiles/bench_incremental_grads.py [--out profiles/r11_bench_incremental_grads.json]
"""
import argparse
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


def breakdown(inc, seed):
    """Median ms of each phase of an eager input_grads call, events between the phases."""
    t, ev = {}, []

    def mark(name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        ev.append((name, e))
    for it in range(ITERS + 2):
        ev.clear()
        mark("start")
        inc._grad_launch(seed, mark=mark)
        torch.cuda.synchronize()
        if it >= 2:
            for (_, a), (k, b) in zip(ev[:-1], ev[1:]):
                t.setdefault(k, []).append(a.elapsed_time(b))
    return {k: statistics.median(v) for k, v in t.items()}


def rel_err(got, ref):
    return float((got - ref).abs().max()) / max(float(ref.abs().max()), 1e-30)


def edit_pin(cf, nf, rng):
    """Cell-type swap on a row carrying a cell type, new uniforms on a row carrying net features (in place)."""
    oh = cf[:, :NUM_CTYPES]
    if float(oh.sum()) == 1.0:
        k = int(torch.argmax(oh))
        oh.zero_()
        oh[0, (k + 1 + int(rng.integers(0, NUM_CTYPES - 1))) % NUM_CTYPES] = 1.0
    if float(nf.abs().sum()) > 0:
        nf.copy_(torch.from_numpy(rng.random(nf.shape, dtype=np.float32)))


def loop_iteration(inc, b, seed, grads, rng, n_cand=64):
    """gradient -> what_if over the n_cand pins with the largest gradient norm -> commit the best; host seconds."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    g = grads()
    norm = g["cell_feat"].norm(dim=1) + g["net_feat"].norm(dim=1)
    pins = torch.topk(norm, n_cand).indices.cpu().numpy()
    wi = inc.what_if([[int(p)] for p in pins])
    for k in range(wi.K):
        _, cf, nf = wi.rows(k)
        edit_pin(cf, nf, rng)
    obj = torch.nan_to_num(wi.run(), nan=0.0) @ seed
    fitted = torch.from_numpy(wi.fitted()).to(obj.device)
    k = int(torch.argmin(torch.where(fitted, obj, torch.full_like(obj, float("inf")))).item())
    wi.commit(k)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, int(fitted.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_bench_incremental_grads.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    model, net = tm_engine.build_models(d.map_size, seed=0, device=DEV)
    step = tm_engine.DesignStep(model, net)
    b = tm_engine.DesignBatch.from_host(tm_engine.HostDesign(d, pin=True), DEV)
    torch.cuda.synchronize()
    sched = b.graph.schedule()
    inc = step.incremental(b, what_if_rows=64 * sched.n_sched // 8)
    T = int(b.endpoints.numel())
    rng = np.random.default_rng(0)
    pool = torch.cuda.graph_pool_handle()
    res = {"card": card(), "repeats": REPEATS, "iters": ITERS,
           "model": "U-Net tf32x3, all endpoints of the design", "design": "tm_synth c2 seed 0",
           "pins": int(sched.n), "scheduled_pins": int(sched.n_sched), "levels": sched.num_levels, "endpoints": T,
           "cases": {}}
    order = torch.argsort(inc.pred, descending=True)
    deep = torch.argsort(b.endpoint_level.reshape(-1), descending=True, stable=True)
    picks = {"top1": order[:1], "top8": order[:8], "top64": order[:64], "deepest1": deep[:1], "deepest64": deep[:64],
             "random64": torch.from_numpy(rng.choice(T, 64, replace=False)).to(DEV), "all": order}
    seed = torch.zeros(T, dtype=torch.float32, device=DEV)
    fseed = torch.zeros(T, dtype=torch.float32, device=DEV)
    cone_replay = inc.capture_input_grads(seed, pool=pool)
    frozen_replay = step.capture(b, input_grads=True, pred_grad=fseed, param_grads=False, pool=pool)
    for name, idx in picks.items():
        seed.zero_()
        seed[idx] = 1.0
        fseed.copy_(seed)
        g = {k: v.clone() for k, v in cone_replay().items()}
        frozen_replay()
        torch.cuda.synchronize()
        err = {k: rel_err(g[k], b.input_grads[k]) for k in g}
        t = ab({"cone_replay": cone_replay, "frozen_replay": frozen_replay})
        size = inc.grad_cone_size()
        case = {"seeded_endpoints": int(idx.numel()), "cone_pins": size, "cone_fraction": size / sched.n_sched,
                "ms_per_call": t, "frozen_over_cone": t["frozen_replay"] / t["cone_replay"],
                "max_rel_err_vs_frozen": err, "eager_breakdown_ms": breakdown(inc, seed)}
        res["cases"][name] = case
        print(json.dumps({name: case}), flush=True)
    # one optimisation iteration on the top-64 objective: gradient -> what_if over 64 pins -> commit
    seed.zero_()
    seed[picks["top64"]] = 1.0
    fseed.copy_(seed)

    def frozen_grads():
        frozen_replay()
        return b.input_grads
    loop, admitted = {"cone": [], "frozen": []}, []
    for it in range(ITERS + 1):
        for k, fn in (("cone", cone_replay), ("frozen", frozen_grads)):
            dt, n_adm = loop_iteration(inc, b, seed, fn, rng)
            if it >= 1:
                loop[k].append(dt * 1e3)
                admitted.append(n_adm)
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
