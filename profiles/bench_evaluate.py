"""The fused evaluation step (DesignStep.evaluate / capture_evaluate) against the eager inference it replaces.

  variants, per config and K:
    eager_forward_metrics : DesignStep.forward + tm_ops.step_metrics (pooled over the batch), eager, one stream for the
                            propagation (the persistent kernel) with the image branch behind it
    eager_evaluate        : DesignStep.evaluate, eager (two streams, per-level propagation, per-design / per-level rows)
    captured_evaluate     : DesignStep.capture_evaluate replays (one CUDA graph)
  cases: config 2 (100k cells, 256x256 U-Net image; the headline design) and config 1 (5k cells, 64x64 image; BASELINE's
         inference config), each for K = 1 design with all of its endpoints and K = 8 joined designs (tm_synth seeds
         0..7, DesignBatch.concat).  U-Net in the default tf32x3 mode, train mode (batch-norm statistics of the batch,
         as the reference validates).
  timing: every variant is warmed up, then the variants are timed alternately REPEATS times, CUDA events around ITERS
          calls each; the median is reported in ms per call and designs/s.  The inputs stay resident on the device.
  check: captured against eager evaluate (predictions and metric table, bitwise) and against forward (max relative
         difference of the predictions, fp32-class).
Writes one JSON line (card name and power limit read in the same run) to --out and stdout.
Usage: python profiles/bench_evaluate.py [--out profiles/r8_bench_evaluate.json]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

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
KS = (1, 8)
CONFIGS = ("c2", "c1")


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


def bits(t):
    return t.detach().contiguous().view(torch.int32)


def run_case(cfg, K, designs):
    model, net = tm_engine.build_models(designs[0].map_size, seed=0, device=DEV)
    step = tm_engine.DesignStep(model, net)
    hosts = [tm_engine.HostDesign(d, pin=True) for d in designs[:K]]

    def batch():
        bs = [tm_engine.DesignBatch.from_host(h, DEV) for h in hosts]
        return bs[0] if K == 1 else tm_engine.DesignBatch.concat(bs)
    b_fwd, b_eval, b_cap = batch(), batch(), batch()
    torch.cuda.synchronize()

    def eager_forward_metrics():
        pred = step.forward(b_fwd)
        return pred, tm_ops.step_metrics(pred, b_fwd.arrival_time)

    replay = step.capture_evaluate(b_cap)
    variants = {"eager_forward_metrics": eager_forward_metrics,
                "eager_evaluate": lambda: step.evaluate(b_eval),
                "captured_evaluate": replay}
    t = ab(variants)
    pred_c, met_c = replay()
    pred_e, met_e = step.evaluate(b_eval)
    pred_f = step.forward(b_fwd)
    torch.cuda.synchronize()
    rel = float(((pred_c.double() - pred_f.double()).abs() / pred_f.double().abs().max()).max())
    out = {"endpoints": int(b_cap.endpoints.numel()), "pins": int(b_cap.graph.number_of_nodes()),
           "metric_rows": int(met_c.table.shape[0]),
           "ms_per_call": t,
           "designs_per_s": {k: K * 1e3 / ms for k, ms in t.items()},
           "captured_vs_eager_evaluate_bitwise": bool(torch.equal(pred_c, pred_e) and torch.equal(bits(met_c.table),
                                                                                                   bits(met_e.table))),
           "captured_vs_forward_max_rel_diff": rel,
           "batch_row": met_c.to_host().batch.tolist()}
    step.close()
    del variants, replay
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_bench_evaluate.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    res = {"card": card(), "Ks": list(KS), "repeats": REPEATS, "iters": ITERS,
           "model": "U-Net tf32x3, train mode (batch statistics), all endpoints of every design",
           "designs": "tm_synth seeds 0..K-1 of the config"}
    for cfg in CONFIGS:
        designs = [tm_synth.make_design(seed=s, **tm_synth.CONFIGS[cfg]) for s in range(max(KS))]
        res[cfg] = {f"K{K}": run_case(cfg, K, designs) for K in KS}
    tm_lib.check_err_flags()
    line = json.dumps(res)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line, flush=True)


if __name__ == "__main__":
    main()
