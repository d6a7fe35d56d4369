"""Incremental evaluation (DesignStep.incremental -> IncrementalEvaluation) against the full re-evaluation it replaces.

  design: config 2 (100k cells, 256x256 U-Net image), tm_synth seed 0, one design with all of its endpoints; U-Net in
          the default tf32x3 mode, train mode (batch statistics of the batch, as the reference validates).
  cases:  edit sets of 1, 8, 64 and 512 pins, drawn (a) uniformly from the scheduled pins and (b) from the last quarter
          of the levels.  The synthetic generator draws drivers from all earlier levels, so early seeds have wide cones;
          each case reports its cone's pins, fraction of the scheduled pins and non-empty levels.
  variants, timed alternately:
    captured_update   : IncrementalEvaluation.capture_update(pins) replays (one CUDA graph: S rows, cone build, cone
                        propagation, head netlist side)
    captured_evaluate : DesignStep.capture_evaluate replays (the whole forward, per-level propagation, plus metrics)
    eager_forward     : DesignStep.forward (persistent propagation)
  timing: every variant warmed up, then REPEATS alternating rounds of CUDA events around ITERS calls each; the median is
          reported in ms per call.  Inputs stay resident on the device.
  breakdown: a separate eager run per case with events between the four phases of an update (S rows / cone build /
             propagation / head), median over ITERS calls.
  check: after each case's edit, the captured update's predictions against DesignStep.forward on the edited features
         (bitwise).
Writes one JSON line (card name and power limit read in the same run) to --out and stdout.
Usage: python profiles/bench_incremental.py [--out profiles/r9_bench_incremental.json]
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

DEV = torch.device("cuda", 0)
REPEATS, ITERS = 7, 20
SIZES = (1, 8, 64, 512)
NUM_CTYPES = 34


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
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
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    t = {k: [] for k in variants}
    for _ in range(REPEATS):
        for k, fn in variants.items():
            t[k].append(events(fn))
    return {k: statistics.median(v) for k, v in t.items()}


def edit(b, pins, rng):
    """Cell-type one-hot swaps on cell-output rows, new uniforms on net sinks (host-side edit, one upload)."""
    cf, nf = b.cell_feat[pins].cpu(), b.net_feat[pins].cpu()
    oh = cf[:, :NUM_CTYPES]
    out = oh.sum(1) == 1
    k = torch.argmax(oh, 1)
    j = (k + 1 + torch.from_numpy(rng.integers(0, NUM_CTYPES - 1, size=len(pins)))) % NUM_CTYPES
    oh[out] = 0.0
    oh[out, j[out]] = 1.0
    sink = nf.abs().sum(1) > 0
    nf[sink] = torch.from_numpy(rng.random((int(sink.sum()), 2), dtype=np.float32))
    idx = torch.from_numpy(np.asarray(pins)).to(DEV)
    b.cell_feat[idx] = cf.to(DEV)
    b.net_feat[idx] = nf.to(DEV)


def breakdown(inc, pins):
    """Median ms of each phase of an eager update, events between the phases."""
    sel = inc._pins(pins)
    idx, nc, _ = sel
    gp = inc._params()
    phases = {"s_rows": lambda: tm_ops.gnn_self_terms(inc.S, inc.b.cell_feat, inc.b.net_feat, gp, idx[:nc], idx[nc:]),
              "cone_build": lambda: inc.cone.build(idx),
              "propagation": lambda: tm_ops.gnn_forward_cone(inc.cone, inc.H, inc.S, gp),
              "head": lambda: inc.step._head_netlist_side(inc.H, inc.b, inc._hs, out=inc._pred2)}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)]
    t = {k: [] for k in phases}
    for it in range(ITERS + 3):
        ev[0].record()
        for i, fn in enumerate(phases.values()):
            fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        if it >= 3:
            for i, k in enumerate(phases):
                t[k].append(ev[i].elapsed_time(ev[i + 1]))
    return {k: statistics.median(v) for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_bench_incremental.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    model, net = tm_engine.build_models(d.map_size, seed=0, device=DEV)
    step = tm_engine.DesignStep(model, net)
    host = tm_engine.HostDesign(d, pin=True)
    b_inc, b_cap = tm_engine.DesignBatch.from_host(host, DEV), tm_engine.DesignBatch.from_host(host, DEV)
    torch.cuda.synchronize()
    replay_eval = step.capture_evaluate(b_cap)
    inc = step.incremental(b_inc)
    sched = b_inc.graph.schedule()
    lv = sched.level.cpu().numpy()
    L = sched.num_levels
    scheduled = np.nonzero(lv >= 0)[0]
    late = np.nonzero(lv >= (3 * L) // 4)[0]
    rng = np.random.default_rng(0)
    res = {"card": card(), "repeats": REPEATS, "iters": ITERS,
           "model": "U-Net tf32x3, train mode (batch statistics), all endpoints of the design",
           "design": "tm_synth c2 seed 0", "pins": int(sched.n), "scheduled_pins": int(sched.n_sched), "levels": L,
           "endpoints": int(b_inc.endpoints.numel()), "cases": {}}
    for draw, pool in (("uniform", scheduled), ("last_quarter", late)):
        for k in SIZES:
            pins = np.sort(rng.choice(pool, k, replace=False))
            edit(b_inc, pins, rng)
            replay = inc.capture_update(pins)           # captures after one eager update of the edited rows
            pred = replay().clone()
            ref = step.forward(b_inc)
            torch.cuda.synchronize()
            cone = inc.cone_size()
            lp = inc.cone.level_ptr[:L + 1].cpu().numpy()
            t = ab({"captured_update": replay, "captured_evaluate": replay_eval,
                    "eager_forward": lambda: step.forward(b_cap)})
            res["cases"][f"{draw}_{k}"] = {
                "edited_pins": k, "cone_pins": cone, "cone_fraction": cone / sched.n_sched,
                "nonempty_cone_levels": int((np.diff(lp) > 0).sum()), "ms_per_call": t,
                "update_vs_capture_evaluate": t["captured_update"] / t["captured_evaluate"],
                "captured_update_vs_forward_bitwise": bool(torch.equal(pred.view(torch.int32), ref.view(torch.int32))),
                "eager_update_breakdown_ms": breakdown(inc, pins)}
            print(json.dumps({f"{draw}_{k}": res["cases"][f"{draw}_{k}"]}), flush=True)
    step.close()
    tm_lib.check_err_flags()
    line = json.dumps(res)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line, flush=True)


if __name__ == "__main__":
    main()
