"""Cost of an input-gradient step against a frozen predictor (``DesignStep.run(input_grads=True, param_grads=False)``).

  step    : the config-2 design step captured as a CUDA graph, the training step with ``input_grads=True`` against the
            frozen step, for the U-Net in tf32x3 (3x256x256 image) and LayoutNet in bf16 mode (2x512x512 image) -- the
            two configurations profiles/r6_bench_step_input_grads.json measured.
  rows_dx : tm_selfmlp_rows_dx (fc_cell_self's data gradient in one pass) against tm_selfmlp_rows_dh + tm_tc_gemm_nn
            (tf32x3) over the config-2 cell-class pins, feature rows scattered; the two outputs are compared.
  null    : each weight-gradient-free kernel form against its full call at config-2 sizes: tm_selfmlp_gen_bwd1_dx
            (dW1 = db1 = NULL), tm_fuse_backward (dWt = NULL), tm_gnn_backward (GHID = GZC = NULL) on the per-level
            (fp16-split cell kernels) and the persistent back end.

Every variant is warmed up; A/B variants are timed alternately, 7 times, CUDA events around the calls; the median is
reported.  Prints one JSON line (and writes it to --out), with the card's name and power limit read in the same run.
Usage: python profiles/bench_frozen_step.py [--out FILE]
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
    replays, outs = {}, {}
    for name, pg in (("training_input_grads", True), ("frozen", False)):
        b = tm_engine.DesignBatch.from_synth(d, DEV)
        replays[name] = st.capture(b, input_grads=True, param_grads=pg)
        outs[name] = b
    t = ab(replays, iters=10)
    ig = [outs[k].input_grads for k in replays]
    same = {k: bool(torch.equal(ig[0][k], ig[1][k])) for k in ("image", "net_feat", "cell_feat")}
    c0, c1 = ig[0]["cell_feat"].double(), ig[1]["cell_feat"].double()
    st.close()
    return {"image": f"{cnn} {math}", "pins": int(d.n), "ms": t, "saved_ms": t["training_input_grads"] - t["frozen"],
            "bitwise_equal_after_replays": same,
            "cell_feat_max_abs_diff_over_max": float((c0 - c1).abs().max() / c0.abs().max())}


def rows_dx():
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    b = tm_engine.DesignBatch.from_synth(d, DEV)
    sched = b.graph.schedule()
    cp = sched.cell_class
    M, n = int(cp.numel()), d.n
    torch.manual_seed(0)
    G = torch.randn(n, 128, device=DEV)
    W2 = torch.randn(128, 256, device=DEV) * 0.1
    W1 = torch.randn(256, 36, device=DEV) * 0.1
    H = torch.relu(torch.randn(M, 256, device=DEV))
    dX_f, dX_r = torch.zeros(n, 36, device=DEV), torch.zeros(n, 36, device=DEV)
    dh = torch.empty(M, 256, device=DEV)
    nb = tm_lib.ws_bytes("tm_selfmlp_rows_dh_ws_bytes")
    ws = tm_lib.workspace(nb, DEV)
    old = tm_ops.MATH
    tm_ops.MATH = "tf32x3"

    def fused():
        call("tm_selfmlp_rows_dx", M, G, 128, cp, W2, H, 256, None, W1, 36, dX_f, 36, cp, ws, nb, stream())

    def two_pass():
        call("tm_selfmlp_rows_dh", M, G, 128, cp, W2, H, 256, None, dh, 256, ws, nb, stream())
        tm_ops.gemm_nn(M, 36, 256, dh, 256, W1, 36, dX_r, 36, c_rows=cp)
    t = ab({"rows_dx": fused, "rows_dh+gemm_nn": two_pass}, iters=50)
    tm_ops.MATH = old
    ref = (((G[cp.long()].double() @ W2.double()) * (H > 0)) @ W1.double())
    err = {k: float((v[cp.long()].double() - ref).abs().max() / ref.abs().max()) for k, v in
           (("rows_dx", dX_f), ("rows_dh+gemm_nn", dX_r))}
    return {"rows": M, "ms": t, "max_abs_err_over_max_vs_fp64": err,
            "max_abs_diff_between_the_two_over_max": float((dX_f - dX_r).abs().max() / dX_r.abs().max()),
            "hidden_gradient_MB_not_written": M * 256 * 4 / 1e6}


def null_forms():
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS["c2"])
    model, net = tm_engine.build_models(d.map_size, seed=0, device=DEV)
    b = tm_engine.DesignBatch.from_synth(d, DEV)
    sched = b.graph.schedule()
    n = d.n
    torch.manual_seed(1)
    out = {}
    # fc_net_self data gradient
    npins = sched.net_class
    M = int(npins.numel())
    G = torch.randn(n, 128, device=DEV)
    W1, b1 = torch.randn(256, 2, device=DEV) * 0.5, torch.randn(256, device=DEV) * 0.3
    W2 = torch.randn(128, 256, device=DEV) * 0.1
    dW1, db1 = torch.empty(256, 2, device=DEV), torch.empty(256, device=DEV)
    dXa, dXb = torch.zeros(n, 2, device=DEV), torch.zeros(n, 2, device=DEV)
    nb = tm_lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")
    ws = tm_lib.workspace(nb, DEV)
    t = ab({"full": lambda: call("tm_selfmlp_gen_bwd1_dx", M, G, 128, npins, b.net_feat, 2, npins, 2, W1, b1, W2, dW1,
                                 db1, dXa, 2, ws, nb, stream()),
            "null": lambda: call("tm_selfmlp_gen_bwd1_dx", M, G, 128, npins, b.net_feat, 2, npins, 2, W1, b1, W2, None,
                                 None, dXb, 2, ws, nb, stream())}, iters=50)
    out["gen_bwd1_dx"] = {"rows": M, "ms": t, "bitwise_equal": bool(torch.equal(dXa, dXb))}
    # mask fusion
    J = b.width
    feat, wt = torch.randn(J, device=DEV), torch.randn(J, 128, device=DEV) * 0.01
    T = int(b.endpoints.numel())
    gy = torch.randn(T, 128, device=DEV)
    cptr, ct = b.mask_rows.csc()
    dwt, dFa, dFb = torch.empty(J, 128, device=DEV), torch.empty(J, device=DEV), torch.empty(J, device=DEV)
    t = ab({"full": lambda: call("tm_fuse_backward", T, J, 128, cptr, ct, gy, 128, feat, wt, dwt, dFa, stream()),
            "null": lambda: call("tm_fuse_backward", T, J, 128, cptr, ct, gy, 128, feat, wt, None, dFb, stream())},
           iters=50)
    out["fuse_backward"] = {"J": J, "T": T, "ms": t, "bitwise_equal": bool(torch.equal(dFa, dFb))}
    # propagation backward, both back ends
    step = tm_engine.DesignStep(model, net)
    gp = [p.detach() for p in step.gnn_params]
    cn1w, cn2w = tm_ops._f32c(gp[8]), tm_ops._f32c(gp[10])
    ncr = max(sched.n_cell_rows, 1)
    GA = torch.empty(ncr, 128, device=DEV)
    GHID, GZC = torch.empty(ncr, 256, device=DEV), torch.empty(ncr, 128, device=DEV)
    nbg = tm_lib.ws_bytes("tm_gnn_ws_bytes")
    wsg = tm_lib.workspace(nbg, DEV)
    G0 = torch.zeros(n, 128, device=DEV)
    G0[b.endpoints.long()] = torch.randn(T, 128, device=DEV)
    for name, impl in (("per_level_h16", 16), ("persistent", 3)):
        old = tm_lib.lib().tm_gnn_set_impl(impl)
        try:
            H, saved = tm_ops.gnn_forward(sched, b.cell_feat, b.net_feat, gp, save=True)
            Ga, Gb = G0.clone(), G0.clone()

            def run(Gx, wg):
                Gx.copy_(G0)                                  # (the sweep consumes G: every call starts from the seed)
                call("tm_gnn_backward", sched.struct, saved["H"], Gx, cn1w, cn2w, saved["A"], saved["LSE"], saved["HID"],
                     GA, GHID if wg else None, GZC if wg else None, wsg, nbg, stream())
            run(Ga, True)
            run(Gb, False)
            torch.cuda.synchronize()
            equal = bool(torch.equal(Ga, Gb))
            t = ab({"full": lambda: run(Ga, True), "null": lambda: run(Gb, False)}, iters=10)
        finally:
            tm_lib.lib().tm_gnn_set_impl(old)
        out[f"gnn_backward_{name}"] = {"ms": t, "bitwise_equal": equal}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(DEV)
    out = {"card": card(), "rows_dx": rows_dx(), "null": null_forms(),
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
