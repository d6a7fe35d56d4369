"""Which kernel serves each product of the four two-layer MLPs that run through ``tm_ops.mlp2_*``, in every arithmetic
mode, and where a misaligned operand sends a product that has a fused kernel.  Host logic only (no device).  A change
of this table is a change of which kernels the step launches."""
import pytest

import tm_ops

MATHS = ("tf32x3", "tf32", "tc6", "tc3", "bf16", "fp32")
MLPS = {"fc_cell_self": (36, 256, 128), "fc_net_self": (2, 256, 128), "mlp_alpha": (1, 64, 32), "mlp_fuse": (288, 576, 1)}

GEMM = dict(hidden="stored", lin1="gemm", lin2="gemm", dw2="gemm", dh="gemm", dw1="gemm", dx="gemm", dx_only="gemm")
SMALLK = dict(hidden="generated", lin1="tm_tc_mlp2_smallk_forward", lin2="tm_tc_mlp2_smallk_forward",
              dw2="tm_tc_mlp2_smallk_wgrad2", dh="gemm", dw1="tm_tc_mlp1_bwd_fused", dx="gemm", dx_only="gemm")
GEN_SPLIT = dict(hidden="generated", lin1="tm_selfmlp_gen_forward", lin2="tm_selfmlp_gen_forward",
                 dw2="tm_selfmlp_gen_wgrad2", dh="tm_selfmlp_gen_bwd1", dw1="tm_selfmlp_gen_bwd1",
                 dx="tm_selfmlp_gen_bwd1_dx", dx_only="tm_selfmlp_gen_bwd1_dx")
ROWS_SPLIT = dict(GEMM, lin1="tm_selfmlp_lin1_relu", lin2="tm_selfmlp_rows_forward", dh="tm_selfmlp_rows_dh",
                  dx_only="tm_selfmlp_rows_dx")


def _expected(mlp, math):
    if mlp == "fc_cell_self":
        return ROWS_SPLIT if math == "tf32x3" else GEMM
    if mlp == "fc_net_self":
        return GEN_SPLIT if math == "tf32x3" else GEMM if math == "fp32" else SMALLK
    if mlp == "mlp_alpha":
        return GEMM if math == "fp32" else SMALLK
    return GEMM


@pytest.mark.parametrize("math", MATHS)
@pytest.mark.parametrize("mlp", sorted(MLPS))
def test_route_of_each_mlp(mlp, math):
    assert tm_ops.mlp2_route(1000, *MLPS[mlp], math=math) == _expected(mlp, math)


@pytest.mark.parametrize("misaligned, expected", [
    # fc_net_self: the forward and the backward leave the fused kernels independently
    ("out", dict(GEN_SPLIT, lin1="tm_tc_mlp2_smallk_forward", lin2="tm_tc_mlp2_smallk_forward")),
    ("g", dict(SMALLK, lin1="tm_selfmlp_gen_forward", lin2="tm_selfmlp_gen_forward")),
])
def test_generated_route_with_a_misaligned_operand(misaligned, expected):
    assert tm_ops.mlp2_route(1000, *MLPS["fc_net_self"], math="tf32x3", **{f"{misaligned}_aligned": False}) == expected


@pytest.mark.parametrize("misaligned, expected", [
    # fc_cell_self: the fused second layer needs the fused first layer's row maxima
    ("x", dict(GEMM, dh="tm_selfmlp_rows_dh", dx_only="tm_selfmlp_rows_dx")),
    ("out", dict(ROWS_SPLIT, lin2="gemm")),
    ("g", dict(ROWS_SPLIT, dh="gemm", dx_only="gemm")),
    ("dx", dict(ROWS_SPLIT, dx_only="gemm")),
])
def test_stored_route_with_a_misaligned_operand(misaligned, expected):
    assert tm_ops.mlp2_route(1000, *MLPS["fc_cell_self"], math="tf32x3", **{f"{misaligned}_aligned": False}) == expected


def test_no_rows_store_an_empty_hidden_layer():
    assert tm_ops.mlp2_route(0, *MLPS["fc_net_self"], math="tf32x3") == dict(GEMM, dh="tm_selfmlp_rows_dh")
    assert tm_ops.mlp2_route(0, *MLPS["fc_cell_self"], math="tf32x3") == dict(ROWS_SPLIT, lin1="gemm", lin2="gemm")
