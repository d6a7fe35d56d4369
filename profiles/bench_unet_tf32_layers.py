"""U-Net (Unet.py:85-119) convolutions in tf32x3 mode at the headline's 3x256x256 image: every 3x3 layer and every
transposed convolution, per direction, on the TMA-fed kernels (tm_conv3x3_tf32*, tm_convt2x2_tf32*; K split and
folded for the deep layers) and on the cp.async route they replace (tm_tc_conv2d_nhwc_splitk,
tm_tc_conv2d_wgrad_nhwc + unpacking, and the CUDA-core transposed-conv kernels).  Weight packing is outside the timed
region.  Algorithmic TFLOP/s = 2 * taps * Cin * Cout * pixels / time (the 3xTF32 products count once).

Every shape is warmed up; the two routes are timed alternately, REPEATS times, CUDA events around ITERS calls; the
median is reported.  The working sets fit in L2, as they do in the step.  Prints one JSON line, with the card's name
and power limit read in the same run.
Usage: python profiles/bench_unet_tf32_layers.py
"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import bench_layoutnet_step as bl  # noqa: E402  (card, ab; imports the package)

import tm_lib  # noqa: E402
import tm_unet  # noqa: E402
from tm_lib import call, stream  # noqa: E402

DEV = bl.DEV
# (H, Cin, Cout) of the 3x3 layers, encoder then decoder; (H of the input map, Cin, Cout) of the transposed convs
CONV = [(256, 16, 16), (256, 16, 16), (128, 16, 32), (128, 32, 32), (64, 32, 64), (64, 64, 64), (32, 64, 128),
        (32, 128, 128), (64, 128, 64), (64, 64, 64), (128, 64, 32), (128, 32, 32), (256, 32, 16), (256, 16, 16)]
CONVT = [(32, 128, 64), (64, 64, 32), (128, 32, 16)]


def conv_layer(h, cin, cout):
    B, w = 1, h
    npix = B * h * w
    x, dy = torch.randn(npix, cin, device=DEV), torch.randn(npix, cout, device=DEV)
    wt = torch.randn(cout, cin, 3, 3, device=DEV) * 0.05
    y, dx = torch.empty(npix, cout, device=DEV), torch.empty(npix, cin, device=DEV)
    err = tm_lib.err_flag(DEV)
    tm_unet.MATH = "tf32x3"
    wq, wd = tm_unet._pack_tma(wt, w, True, "tf32")
    wf, wb = tm_unet._pack(wt, True)
    ws = tm_unet._Ws(DEV)
    nbw = tm_lib.ws_bytes("tm_conv3x3_tf32_wgrad_ws", B, h, w, cin, cout)
    dw = torch.empty(cout, cin, 3, 3, device=DEV)
    flop = 2.0 * 9 * cin * cout * npix
    dirs = {
        "fwd": {"tma": lambda: tm_unet._conv_tf(ws, x, cin, B, h, w, cin, cout, wq, y, cout),
                "cp_async": lambda: tm_unet._conv(x, cin, B, h, w, cin, cout, 3, wf, None, y, cout)},
        "dgrad": {"tma": lambda: tm_unet._conv_tf(ws, dy, cout, B, h, w, cout, cin, wd, dx, cin),
                  "cp_async": lambda: tm_unet._conv(dy, cout, B, h, w, cout, cin, 3, wb, None, dx, cin)},
        "wgrad": {"tma": lambda: call("tm_conv3x3_tf32_wgrad", B, h, w, cin, cin, cout, x, cin, dy, cout, dw, ws.get(nbw), nbw,
                                      err, stream()),
                  "cp_async": lambda: tm_unet._conv_wgrad(ws, x, cin, dy, cout, B, h, w, cin, cout, 3, False)},
    }
    out = {"shape": f"3x3 {cin}->{cout} at {h}x{w}", "GFLOP": flop / 1e9}
    for d, v in dirs.items():
        t = bl.ab(v)
        out[d] = {r: {"us": ms * 1e3, "TFLOPs": flop / ms / 1e9} for r, ms in t.items()}
    return out


def convt_layer(h, cin, cout):
    B, w = 1, h
    npix = B * h * w
    x = torch.randn(npix, cin, device=DEV)
    cat = torch.randn(4 * npix, 2 * cout, device=DEV)                # [skip | up] concat buffer: dy is its second half
    half = cat[:, cout:]
    wt = torch.randn(cin, cout, 2, 2, device=DEV) * 0.05
    bias = torch.randn(cout, device=DEV)
    dx = torch.empty(npix, cin, device=DEV)
    err = tm_lib.err_flag(DEV)
    wfq, wdq = torch.empty(4 * cout, cin, device=DEV), torch.empty(4, cin, cout, device=DEV)
    call("tm_convt2x2_pack_f32", cin, cout, wt, wfq, wdq, stream())
    wtf, wtT = torch.empty(cin, 4 * cout, device=DEV), torch.empty(4 * cout, cin, device=DEV)
    call("tm_convt_pack_weight", cin, cout, wt, wtf, wtT, stream())
    shape = (B, h, w, cin, cout)
    nb = tm_lib.ws_bytes("tm_convt2x2_tf32_ws", *shape)
    wsb = tm_lib.workspace(max(nb, 256), DEV)
    nbo = tm_lib.ws_bytes("tm_convt2x2_wgrad_ws", *shape)
    wso = tm_lib.workspace(nbo, DEV)
    dw, dwt, dbt = torch.empty(cin, cout, 2, 2, device=DEV), torch.empty(cin, 4 * cout, device=DEV), torch.empty(cout, device=DEV)
    flop = 2.0 * 4 * cin * cout * npix
    dirs = {
        "fwd": {"tma": lambda: call("tm_convt2x2_tf32", *shape, x, cin, wfq, bias, half, 2 * cout, wsb, nb, err, stream()),
                "cp_async": lambda: call("tm_convt2x2_nhwc", *shape, x, cin, wtf, bias, half, 2 * cout, 2 * h, 2 * w, 0, 0,
                                         stream())},
        "dgrad": {"tma": lambda: call("tm_convt2x2_tf32_dgrad", *shape, half, 2 * cout, wdq, dx, cin, wsb, nb, err, stream()),
                  "cp_async": lambda: call("tm_convt2x2_dgrad_nhwc", *shape, half, 2 * cout, 2 * h, 2 * w, 0, 0, wtT, dx, cin,
                                           stream())},
    }
    if tm_lib.ws_bytes("tm_convt2x2_tf32_wgrad_supported", *shape) == 1:
        def old_wgrad():
            call("tm_convt2x2_wgrad_nhwc", *shape, x, cin, half, 2 * cout, 2 * h, 2 * w, 0, 0, dwt, dbt, wso, nbo, stream())
            call("tm_convt_unpack_wgrad", cin, cout, dwt, dw, stream())
        dirs["wgrad"] = {"tma": lambda: call("tm_convt2x2_tf32_wgrad", *shape, x, cin, half, 2 * cout, dw, wsb, nb, err,
                                             stream()),
                         "cp_async": old_wgrad}
    out = {"shape": f"convT 2x2 {cin}->{cout} at {h}x{w}", "GFLOP": flop / 1e9}
    for d, v in dirs.items():
        t = bl.ab(v)
        out[d] = {r: {"us": ms * 1e3, "TFLOPs": flop / ms / 1e9} for r, ms in t.items()}
    return out


def main():
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    out = {"card": bl.card(), "conv3x3": [conv_layer(*s) for s in CONV], "convt2x2": [convt_layer(*s) for s in CONVT]}
    tot = {r: sum(l[d][r]["us"] for l in out["conv3x3"] + out["convt2x2"] for d in ("fwd", "dgrad", "wgrad") if d in l)
           for r in ("tma", "cp_async")}
    out["sum_us"] = tot
    tm_lib.check_err_flags()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
