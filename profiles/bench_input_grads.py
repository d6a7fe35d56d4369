"""Cost of the image gradient (d output / d input image) of the image networks.

  kernel : tm_conv_dgrad_narrow, standalone, on the two shapes it serves -- U-Net inc.double_conv.0 (k = 3, dy 16
           channels -> dx 3, 1x256x256, the config-2 image) and LayoutNet encode.0 (k = 9, dy 32 channels -> dx 2,
           1x512x512) -- with fp32 and bf16 dy; next to the generic route the same data gradient would otherwise take
           (tm_unet._conv on the dgrad-packed weight in tf32x3, NHWC output, then tm_nhwc_to_nchw).  Algorithmic
           GFLOP = 2*k*k*Cin*Cout*H*W; dy bytes = H*W*Cout*sizeof(dy).
  module : UNet (3x256x256) and LayoutNet (2x512x512) forward + backward through the nn.Module (autograd), with
           the input's requires_grad off and on, in tf32x3 and bf16 mode.

Every variant is warmed up; A/B variants are timed alternately, REPEATS times, CUDA events around ITERS calls; the
median is reported.  Working sets fit in L2 (dy is at most 34 MB).  Prints one JSON line (and writes it to --out),
with the card's name and power limit read in the same run.
Usage: python profiles/bench_input_grads.py [--out FILE]
"""
import argparse
import importlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import bench_configs as bc  # noqa: E402
from bench_layoutnet_step import ab, card  # noqa: E402

importlib.import_module(bc.PKG)
import model as M  # noqa: E402
import tm_lib  # noqa: E402
import tm_unet  # noqa: E402
import Unet as U  # noqa: E402
from tm_lib import call, stream  # noqa: E402

DEV = torch.device("cuda", 0)


def kernel(k, cout, cin, H):
    torch.manual_seed(k)
    B = 1
    npix = B * H * H
    dy = torch.randn(npix, cout, device=DEV)
    dyb = dy.bfloat16()
    w = torch.randn(cout, cin, k, k, device=DEV) * 0.05
    dx = torch.empty(B, cin, H, H, device=DEV)
    dx_rows = torch.empty(npix, cin, device=DEV)
    _, wb = tm_unet._pack(w, True)

    def generic():
        tm_unet._conv(dy, cout, B, H, H, cout, cin, k, wb, None, dx_rows, cin, math="tf32x3")
        call("tm_nhwc_to_nchw", B, cin, H, H, dx_rows, cin, dx, stream())
    t = ab({"narrow_fp32_dy": lambda: call("tm_conv_dgrad_narrow", B, H, H, cin, cout, k, dy, cout, 0, w, dx, stream()),
            "narrow_bf16_dy": lambda: call("tm_conv_dgrad_narrow", B, H, H, cin, cout, k, dyb, cout, 1, w, dx, stream()),
            "generic_tf32x3_then_nchw": generic}, iters=50)
    flop = 2.0 * k * k * cin * cout * npix
    return {"shape": f"k={k}, dy {cout} ch -> dx {cin} ch at {B}x{H}x{H}", "GFLOP": flop / 1e9,
            "dy_MB": {"fp32": npix * cout * 4 / 1e6, "bf16": npix * cout * 2 / 1e6},
            "ms": t, "TFLOPs": {n: flop / ms / 1e9 for n, ms in t.items()}}


def module(net, x):
    g = None

    def run(want_x):
        def fn():
            nonlocal g
            xi = x.detach().requires_grad_(want_x)
            out = net(xi)
            if g is None:
                g = torch.randn_like(out)
            out.backward(g)
        return fn
    return ab({"input_grad_off": run(False), "input_grad_on": run(True)}, iters=10)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    out = {"card": card(),
           "kernel": {"unet_inc": kernel(3, 16, 3, 256), "layoutnet_encode0": kernel(9, 32, 2, 512)},
           "module_fwd_bwd_ms": {}}
    torch.manual_seed(1)
    unet = U.UNet("max").to(DEV).train()
    lnet = M.LayoutNet("max").to(DEV).train()
    xu, xl = torch.rand(1, 3, 256, 256, device=DEV), torch.rand(1, 2, 512, 512, device=DEV)
    for math in ("tf32x3", "bf16"):
        unet.math = lnet.math = math
        out["module_fwd_bwd_ms"][f"unet_256_{math}"] = module(unet, xu)
        out["module_fwd_bwd_ms"][f"layoutnet_512_{math}"] = module(lnet, xl)
    tm_lib.check_err_flags()
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
