"""Several designs per fused design step (DesignBatch.concat + DesignStep): is a step over K designs cheaper per
design than K one-design steps?

  step : K in {1, 2, 4, 8} config-2 designs (tm_synth seeds 0..K-1) joined by DesignBatch.concat, stepped as one
         resident CUDA-graph replay, next to the one-design step (DesignBatch.from_host, the headline's form) on design
         0, for the U-Net in tf32x3, the U-Net with TM_UNET_MATH=bf16 (net.math = "bf16") and LayoutNet bf16 on a
         2x512x512 image.  ms per step and designs/s; every variant of a network is warmed up and then timed
         alternately REPEATS times, CUDA events around ITERS replays; the median is reported.
  memory: peak bytes allocated while a variant is built, captured and replayed, over what was allocated before.
  check: at K = 2 (full size), every gradient of the joined step against the mean of the two one-design steps, at
         tests/dp_equivalence.py's bar (1e-5 relative + 1e-6 of the largest magnitude); the number of elements
         outside it and the largest relative error are reported.
Writes one JSON line (card name and power limit read in the same run) to --out and stdout.
Usage: python profiles/bench_multi_design.py [--out profiles/r3_bench_multi_design.json]
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
import tm_synth  # noqa: E402

DEV = torch.device("cuda", 0)
REPEATS, ITERS = 5, 10
KS = (1, 2, 4, 8)
NETS = (("unet_tf32x3", "unet", None), ("unet_bf16", "unet", "bf16"), ("layoutnet_bf16", "layoutnet", "bf16"))


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


def models(cnn, math, map_size):
    model, net = tm_engine.build_models(map_size, seed=0, device=DEV, cnn=cnn)
    if math:
        net.math = math
    return model, net


def grads(model, net):
    return [None if p.grad is None else p.grad.detach().clone() for p in list(model.parameters()) + list(net.parameters())]


def grad_check(cnn, math, designs):
    """K = 2 joined step against the mean of the one-design steps (fresh models, same seed)."""
    model, net = models(cnn, math, designs[0].map_size)
    step = tm_engine.DesignStep(model, net)
    single = []
    for d in designs[:2]:
        step.run(tm_engine.DesignBatch.from_synth(d, DEV))
        torch.cuda.synchronize()
        single.append(grads(model, net))
    model2, net2 = models(cnn, math, designs[0].map_size)
    step2 = tm_engine.DesignStep(model2, net2)
    step2.run(tm_engine.DesignBatch.concat([tm_engine.DesignBatch.from_synth(d, DEV) for d in designs[:2]]))
    torch.cuda.synchronize()
    bad, worst = 0, 0.0
    for a, (g0, g1) in zip(grads(model2, net2), zip(*single)):
        if a is None:
            continue
        ref = (g0.double() + g1.double()) / 2
        err = (a.double() - ref).abs()
        bad += int((err > 1e-5 * ref.abs() + 1e-6 * ref.abs().max()).sum())
        worst = max(worst, float((err / ref.abs().max().clamp_min(1e-30)).max()))
    return {"elements_outside_dp_bar": bad, "max_err_over_max_abs": worst}


def run_net(name, cnn, math, designs):
    model, net = models(cnn, math, designs[0].map_size)
    step = tm_engine.DesignStep(model, net)
    variants, mem, keep = {}, {}, []
    hosts = [tm_engine.HostDesign(d, pin=True) for d in designs]

    def add(key, make):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        b = make()
        replay = step.capture(b)
        replay()
        torch.cuda.synchronize()
        mem[key] = torch.cuda.max_memory_allocated() - base
        keep.append(b)                                  # the batch's tensors are the graph's static inputs
        variants[key] = replay

    add("single_design_step", lambda: tm_engine.DesignBatch.from_host(hosts[0], DEV))
    for K in KS:
        add(f"K{K}", lambda K=K: tm_engine.DesignBatch.concat([tm_engine.DesignBatch.from_host(h, DEV)
                                                               for h in hosts[:K]]))
    t = ab(variants)
    step.close()
    out = {"ms_per_step": t,
           "designs_per_s": {k: (1 if k == "single_design_step" else int(k[1:])) * 1e3 / ms for k, ms in t.items()},
           "ms_per_design": {k: ms / (1 if k == "single_design_step" else int(k[1:])) for k, ms in t.items()},
           "peak_bytes_over_before": mem,
           "grad_check_K2": grad_check(cnn, math, designs)}
    del variants, keep
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_multi_design.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    res = {"card": card(), "Ks": list(KS), "repeats": REPEATS, "iters": ITERS,
           "designs": "config-2 netlists (tm_synth seeds 0..K-1); U-Net 3x256x256, LayoutNet 2x512x512 images"}
    unet_d = [tm_synth.make_design(seed=s, **tm_synth.CONFIGS["c2"]) for s in range(max(KS))]
    layout_d = [tm_synth.make_design(seed=s, img_channels=2, img_scale=4, **tm_synth.CONFIGS["c2"]) for s in range(max(KS))]
    for name, cnn, math in NETS:
        res[name] = run_net(name, cnn, math, layout_d if cnn == "layoutnet" else unet_d)
    tm_lib.check_err_flags()
    line = json.dumps(res)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line, flush=True)


if __name__ == "__main__":
    main()
