"""LayoutNet (model.py:216-247, the reference's default image network) on the device: its two tensor-bound layers on
both bf16 routes, the whole network in each math mode, and the fused config-2 design step next to the U-Net's.

  layers : encode.3 (7x7, 32->64 at 256x256) and encode.6 (9x9, 64->32 at 128x128) of a 2x512x512 input; forward,
           data gradient and weight gradient on the TMA-fed k x k kernels (tm_convkxk_bf16*, weight gradient with its
           fixed-order reduction) and on the cp.async-fed bf16 tensor-core route (tm_unet._conv / _conv_wgrad with
           math "bf16": tm_tc_conv2d_nhwc_splitk, tm_tc_conv2d_wgrad_nhwc + unpacking).  The bf16 operand copies
           (tm_to_bf16_rows) and the weight packing of the TMA route are outside the timed region; the network
           timing below includes them.  Algorithmic
           TFLOP/s = 2*k*k*Cin*Cout*H*W / time; share of the dense bf16 peak of bench_configs.peaks().
  network: LayoutNet forward + backward (batch 1, 2x512x512) in tf32x3, bf16 on the cp.async route
           (TM_CONV_TMA=0) and bf16 on the TMA route.
  step   : the fused DesignStep on the config-2 netlist: U-Net (3x256x256 image, the headline), LayoutNet tf32x3 and
           LayoutNet bf16 (2x512x512 image); a resident CUDA-graph replay and DesignStep.prepare() end to end
           (per-step values uploaded from pinned host memory before each replay).

Every shape is warmed up; A/B variants are timed alternately, REPEATS times, CUDA events around ITERS calls; the
median is reported.  The working sets fit in L2 (the largest activation is 16 MB), as they do in the step.
Prints one JSON line, with the card's name and power limit read in the same run.
Usage: python profiles/bench_layoutnet_step.py
"""
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
import model as M  # noqa: E402
import tm_engine  # noqa: E402
import tm_lib  # noqa: E402
import tm_synth  # noqa: E402
import tm_unet  # noqa: E402
from tm_lib import call, stream  # noqa: E402

DEV = torch.device("cuda", 0)
REPEATS, ITERS = 7, 20


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


def ab(variants, iters=ITERS):
    """{name: fn} -> {name: median ms}; every variant warmed up, then timed alternately REPEATS times."""
    for fn in variants.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    t = {k: [] for k in variants}
    for _ in range(REPEATS):
        for k, fn in variants.items():
            t[k].append(events(fn, iters))
    return {k: statistics.median(v) for k, v in t.items()}


def layer_routes(k, cin, cout, h, tpk):
    torch.manual_seed(k)
    B, w = 1, h
    npix = B * h * w
    x = torch.randn(npix, cin, device=DEV)
    dy = torch.randn(npix, cout, device=DEV)
    wt = torch.randn(cout, cin, k, k, device=DEV) * 0.02
    bias = torch.randn(cout, device=DEV)
    xb = torch.empty(npix, cin, dtype=torch.bfloat16, device=DEV)
    dyb = torch.empty(npix, cout, dtype=torch.bfloat16, device=DEV)
    call("tm_to_bf16_rows", npix, cin, x, cin, xb, cin, stream())
    call("tm_to_bf16_rows", npix, cout, dy, cout, dyb, cout, stream())
    wq, wd = tm_unet._pack_kxk_bf16(wt, True)
    wf, wb = tm_unet._pack(wt, True)
    y, dx = torch.empty(npix, cout, device=DEV), torch.empty(npix, cin, device=DEV)
    dw = torch.empty(cout, cin, k, k, device=DEV)
    err = tm_lib.err_flag(DEV)
    nb = tm_lib.ws_bytes("tm_convkxk_bf16_wgrad_ws", B, h, w, cin, cout, k)
    ws_t = tm_lib.workspace(nb, DEV)
    wsp = tm_unet._Ws(DEV)
    flop = 2.0 * k * k * cin * cout * npix
    dirs = {
        "fwd": {"tma": lambda: call("tm_convkxk_bf16", B, h, w, cin, cout, k, xb, wq, bias, y, cout, tm_unet.RELU, err, stream()),
                "cp_async": lambda: tm_unet._conv(x, cin, B, h, w, cin, cout, k, wf, bias, y, cout, tm_unet.RELU, math="bf16")},
        "dgrad": {"tma": lambda: call("tm_convkxk_bf16", B, h, w, cout, cin, k, dyb, wd, None, dx, cin, 0, err, stream()),
                  "cp_async": lambda: tm_unet._conv(dy, cout, B, h, w, cout, cin, k, wb, None, dx, cin, math="bf16")},
        "wgrad": {"tma": lambda: call("tm_convkxk_bf16_wgrad", B, h, w, cin, cout, k, xb, dyb, dw, ws_t, nb, err, stream()),
                  "cp_async": lambda: tm_unet._conv_wgrad(wsp, x, cin, dy, cout, B, h, w, cin, cout, k, False, math="bf16")},
    }
    out = {"shape": f"{k}x{k} {cin}->{cout} at {h}x{w}", "GFLOP": flop / 1e9}
    for d, v in dirs.items():
        t = ab(v)
        out[d] = {r: {"ms": ms, "TFLOPs": flop / ms / 1e9, "frac_of_bf16_peak": flop / ms / 1e9 / tpk} for r, ms in t.items()}
    return out


def network():
    torch.manual_seed(1)
    net = M.LayoutNet("max").to(DEV).train()
    x = torch.rand(1, 2, 512, 512, device=DEV)

    def both(math, tma):
        def fn():
            old_m, old_t = tm_unet.MATH, tm_unet.USE_TMA
            tm_unet.MATH, tm_unet.USE_TMA = math, tma
            try:
                out, st = tm_unet.layoutnet_forward(net, x, need_bwd=True)
                tm_unet.layoutnet_backward(net, st, torch.ones_like(out))
            finally:
                tm_unet.MATH, tm_unet.USE_TMA = old_m, old_t
        return fn
    t = ab({"tf32x3": both("tf32x3", True), "bf16_cp_async": both("bf16", False), "bf16_tma": both("bf16", True)}, iters=10)
    return {"fwd_bwd_ms": t}


def step_times():
    d_u = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    d_l = tm_synth.make_design(seed=0, img_channels=2, img_scale=4, **tm_synth.CONFIGS["c2"])
    cases = {}
    for name, d, cnn, math in (("unet", d_u, "unet", None), ("layoutnet_tf32x3", d_l, "layoutnet", None),
                               ("layoutnet_bf16", d_l, "layoutnet", "bf16")):
        model, net = tm_engine.build_models(d.map_size, seed=0, device=DEV, cnn=cnn)
        if math:
            net.math = math
        step = tm_engine.DesignStep(model, net)
        host = tm_engine.HostDesign(d, pin=True)
        batch = tm_engine.DesignBatch.from_host(host, DEV)
        replay = step.capture(batch)
        prep = step.prepare(host, DEV, graph=batch.graph)
        # the batch's tensors are the resident graph's static inputs: they must outlive the replays
        cases[name] = (replay, lambda p=prep, h=host: p.step(h), step, batch)
    t = ab({f"{n}_{kind}": fn for n, (r, e, _, _) in cases.items() for kind, fn in (("resident", r), ("prepare_e2e", e))},
           iters=20)
    for c in cases.values():
        c[2].close()
    return {"ms_per_step": t, "designs": {"unet": "config-2 netlist, 3x256x256 image",
                                          "layoutnet": "config-2 netlist, 2x512x512 image"}}


def main():
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    _, tpk = bc.peaks()
    out = {"card": card(), "bf16_peak_TFLOPs": tpk,
           "bf16_peak_source": "MEASURED_PEAKS.json" if os.path.isfile(os.path.join(ROOT, "MEASURED_PEAKS.json"))
           else "bench_configs.peaks() default (measured burst)",
           "layers": {"encode.3": layer_routes(7, 32, 64, 256, tpk), "encode.6": layer_routes(9, 64, 32, 128, tpk)},
           "layoutnet_512": network(),
           "step_c2": step_times()}
    tm_lib.check_err_flags()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
