"""Pin the oracle (oracle/restate.py, oracle/levelize.py) to the reference, against the committed fixtures
generated from the UNMODIFIED reference (oracle/make_golden.py -> tests/golden/*.npz)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLD, assert_close, design_to_oracle, load_golden_step
from oracle import levelize, restate
import tm_synth


@pytest.fixture(scope="module")
def tiny():
    return tm_synth.make_design(seed=0, **tm_synth.CONFIGS["tiny"])


def test_step_matches_golden(tiny):
    z, sd_m, sd_c = load_golden_step("tiny")
    out = restate.design_step(sd_m, sd_c, design_to_oracle(tiny))
    assert_close(out["feat_map"], z["feat_map"], 1e-5, 1e-6, "feat_map")
    assert_close(out["H"], z["H"], 1e-5, 1e-6, "H")
    assert_close(out["pred"], z["pred"], 1e-5, 1e-6, "pred")
    assert_close(out["loss"], z["loss"], 1e-5, 1e-6, "loss")
    for k in z.files:
        if not k.startswith("grad."):
            continue
        name = k[len("grad.model."):] if k.startswith("grad.model.") else "cnn." + k[len("grad.cnn."):]
        g = out["grads"][name]
        if z[k].size == 0:                                   # fc_net_drive / fc_attn2: never used
            assert g is None, name
        else:
            assert_close(g, z[k], 1e-4, 1e-5, name)
    for k in z.files:
        if k.startswith("after.cnn.") and "running" in k:
            assert_close(out["bn_stats"][k[len("after.cnn."):]], z[k], 1e-5, 1e-6, k)


def test_layoutnet_matches_golden():
    z = np.load(os.path.join(GOLD, "layoutnet.npz"))
    sd = {k[2:]: torch.from_numpy(z[k]).requires_grad_(True) for k in z.files if k.startswith("p.")}
    y = restate.layoutnet_forward(sd, torch.from_numpy(z["x"]))
    assert_close(y, z["y"], 1e-5, 1e-6, "y")
    y.square().sum().backward()
    for k, p in sd.items():
        assert_close(p.grad, z["g." + k], 1e-4, 1e-5, k)


@pytest.mark.parametrize("cfg", ["tiny", "c1"])
def test_levels_match_golden(cfg):
    d = tm_synth.make_design(seed=0, **tm_synth.CONFIGS[cfg])
    z = np.load(os.path.join(GOLD, f"levels_{cfg}.npz"))
    src = np.concatenate([d.net_src, d.cell_src, [d.n]])     # + the unreachable island of make_golden
    dst = np.concatenate([d.net_dst, d.cell_dst, [d.n + 1]])
    lv = levelize.node_levels(d.n + 2, src, dst, d.pis)
    assert np.array_equal(lv, z["node_level"])               # bit-exact pin -> level
    assert np.array_equal(np.nonzero(lv >= 0)[0], z["remaining"])
    assert np.array_equal(d.level, z["node_level"][:d.n])    # the generator's own levels
    assert np.array_equal(d.level[d.endpoints], z["targets_level"])
    if cfg == "tiny":                                        # frontier form, literal restatement
        levels, removed = levelize.topo_levels_frontier(d.n + 2, src, dst, d.pis, d.endpoints,
                                                        {int(e): i for i, e in enumerate(d.endpoints)})
        assert removed == [d.n, d.n + 1]
        for lid, (nodes, targets, pids) in enumerate(levels):
            assert np.array_equal(np.asarray(nodes), np.nonzero(lv == lid)[0])
            assert np.array_equal(np.asarray(pids, np.int64), np.nonzero(z["targets_level"] == lid)[0])
    # critical paths and masks
    preds = [[] for _ in range(d.n)]
    for s, t in zip(src[:-1].tolist(), dst[:-1].tolist()):
        preds[t].append(s)
    off = np.concatenate([[0], np.cumsum(z["path_len"])])
    xy = d.pin_xy
    mi, mc = [0], []
    for i, e in enumerate(d.endpoints):
        p = levelize.find_critical_path(e, d.level, preds)
        assert p == z["path_flat"][off[i]:off[i + 1]].tolist()
        mc.extend(levelize.path_mask_columns(p, xy, d.map_size))
        mi.append(len(mc))
    assert np.array_equal(np.asarray(mi, np.int32), d.mask_indptr)
    assert np.array_equal(np.asarray(mc, np.int32), d.mask_cols)


def test_in_csr_definition(tiny):
    indptr, idx = levelize.in_csr(tiny.n, tiny.cell_src, tiny.cell_dst)
    assert indptr[-1] == tiny.cell_src.size
    for v in range(0, tiny.n, 37):
        row = idx[indptr[v]:indptr[v + 1]]
        assert np.array_equal(row, np.sort(tiny.cell_src[tiny.cell_dst == v]))


def test_bf16_unet_free_running_gradients_are_tie_limited(pkg):
    """Evidence for the way tests/test_gpu_configs.py::test_config4_unet_bf16 checks gradients.  The bf16-rounded
    oracle against ITSELF -- same network, same rounding points, fp32 against fp64 accumulation (differences of
    1e-7 before the first rounding): the outputs agree at the bf16 bar, the parameter gradients do not (relative
    L2 distance of several per cent), because bf16 quantisation noise regenerates at every layer and re-routes
    ReLU / max-pool gates.  No implementation can therefore meet rtol 2e-2 per element on free-running gradients;
    teacher-forcing the gates (restate._force) removes the ambiguity and is what the GPU test does."""
    import Unet as U
    torch.manual_seed(4)
    sd = {k: v.detach().clone() for k, v in U.UNet("max").state_dict().items()}
    x = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(1))
    names = [k for k, v in sd.items() if v.is_floating_point() and "running" not in k]

    def run(dtype, forced=None):
        P = {k: (v.to(dtype).clone().requires_grad_(True) if k in names else (v.to(dtype) if v.is_floating_point() else v.clone()))
             for k, v in sd.items()}
        out, _ = restate.unet_forward(P, x.to(dtype), "max", rounding="bf16", forced=forced)
        g = torch.randn(out.shape, generator=torch.Generator().manual_seed(2)).to(dtype)
        return out.detach(), torch.autograd.grad(out, [P[k] for k in names], g)

    o32, g32 = run(torch.float32)
    # the fp64 run, its contraction outputs captured through the hook the GPU test forces through
    cap = {}
    orig_force = restate._force
    restate._force = lambda y, forced, key: (cap.setdefault(key, y.detach()), y)[1]
    try:
        o64, g64 = run(torch.float64)
    finally:
        restate._force = orig_force
    scale = float(o64.abs().max())
    assert float((o32.double() - o64).abs().max()) <= 2e-2 * scale            # forward: fine at the bf16 bar
    rels = [float((a.double() - b).norm() / b.norm()) for a, b in zip(g32, g64)]
    assert max(rels) > 2e-2, f"free-running bf16 gradients unexpectedly agree ({max(rels):.3e})"
    # with the gates forced to the fp64 run's, the fp32 run's gradients agree per element at the bar
    _, g32f = run(torch.float32, forced=cap)
    for k, a, b in zip(names, g32f, g64):
        err = (a.double() - b).abs()
        tol = 2e-2 * float(b.abs().max()) + 2e-2 * b.abs()
        assert bool((err <= tol).all()), f"{k}: forced fp32 run differs from the fp64 run ({float(err.max()):.3e})"
