"""Cost of the input gradients of the fused design step (``DesignStep.run(input_grads=True)``).

  step    : the config-2 design step captured as a CUDA graph, ``input_grads`` off and on, for the U-Net in tf32x3 (the
            headline step, 3x256x256 image) and LayoutNet in bf16 mode (2x512x512 image).
  kernel  : tm_selfmlp_gen_bwd1_dx (the net pins' feature gradient fused into the first-layer backward of fc_net_self)
            against tm_selfmlp_gen_bwd1 alone, over the config-2 step's net-class pins (feature rows gathered).
  cell_dx : the cell pins' feature gradient, dX = dh W1 (dh stored, 256 -> 36) scattered to the feature rows, on
            tm_tc_gemm_nn in tf32x3 over the config-2 step's cell-class pins.

Every variant is warmed up; A/B variants are timed alternately, 7 times, CUDA events around ITERS calls; the median is
reported.  Prints one JSON line (and writes it to --out), with the card's name and power limit read in the same run.
Usage: python profiles/bench_step_input_grads.py [--out FILE]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import bench_configs  # noqa: E402,F401  (puts the package on sys.path and imports it)
from bench_layoutnet_step import ab, card  # noqa: E402

import tm_engine  # noqa: E402
import tm_lib  # noqa: E402
import tm_ops  # noqa: E402
import tm_synth  # noqa: E402
from tm_lib import call, stream  # noqa: E402

DEV = torch.device("cuda", 0)


def step(cnn, math):
    kw = dict(img_channels=2, img_scale=4) if cnn == "layoutnet" else {}
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"], **kw)
    model, net = tm_engine.build_models(d.map_size, seed=0, device=DEV, cnn=cnn)
    net.math = math
    st = tm_engine.DesignStep(model, net)
    replays = {}
    for on in (False, True):
        b = tm_engine.DesignBatch.from_synth(d, DEV)
        replays["input_grads_on" if on else "input_grads_off"] = st.capture(b, input_grads=on)
    t = ab(replays, iters=10)
    st.close()
    return {"image": f"{cnn} {math}", "pins": int(d.n), "ms": t,
            "added_ms": t["input_grads_on"] - t["input_grads_off"]}


def kernels():
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    b = tm_engine.DesignBatch.from_synth(d, DEV)
    sched = b.graph.schedule()
    n = d.n
    torch.manual_seed(0)
    G = torch.randn(n, 128, device=DEV)
    out = {}

    # net pins: Linear(2, 256) -> ReLU -> Linear(256, 128), hidden layer generated
    npins = sched.net_class
    M = int(npins.numel())
    X = b.net_feat
    W1, b1 = torch.randn(256, 2, device=DEV) * 0.5, torch.randn(256, device=DEV) * 0.3
    W2 = torch.randn(128, 256, device=DEV) * 0.1
    dW1, db1 = torch.empty(256, 2, device=DEV), torch.empty(256, device=DEV)
    dX = torch.zeros(n, 2, device=DEV)
    nb = tm_lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")
    ws = tm_lib.workspace(nb, DEV)
    t = ab({"gen_bwd1": lambda: call("tm_selfmlp_gen_bwd1", M, G, 128, npins, X, 2, npins, 2, W1, b1, W2, dW1, db1,
                                     ws, nb, stream()),
            "gen_bwd1_dx": lambda: call("tm_selfmlp_gen_bwd1_dx", M, G, 128, npins, X, 2, npins, 2, W1, b1, W2, dW1,
                                        db1, dX, 2, ws, nb, stream())}, iters=50)
    out["net_pins"] = {"rows": M, "ms": t, "added_ms": t["gen_bwd1_dx"] - t["gen_bwd1"]}

    # cell pins: dX[c_rows] = dh @ W1, dh (rows, 256) stored, W1 (256, 36)
    cpins = sched.cell_class
    Mc = int(cpins.numel())
    dh = torch.randn(Mc, 256, device=DEV)
    Wc = torch.randn(256, 36, device=DEV) * 0.1
    dXc = torch.zeros(n, 36, device=DEV)
    old = tm_ops.MATH
    tm_ops.MATH = "tf32x3"
    t = ab({"gemm_nn_tf32x3": lambda: tm_ops.gemm_nn(Mc, 36, 256, dh, 256, Wc, 36, dXc, 36, c_rows=cpins)}, iters=50)
    tm_ops.MATH = old
    out["cell_pins"] = {"rows": Mc, "ms": t, "GFLOP": 2.0 * Mc * 256 * 36 / 1e9,
                        "MB_moved": (Mc * (256 + 36) * 4 + Mc * 4) / 1e6}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    out = {"card": card(), "kernels": kernels(),
           "step_c2": {"unet_tf32x3": step("unet", "tf32x3"), "layoutnet_bf16": step("layoutnet", "bf16")}}
    tm_lib.check_err_flags()
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
