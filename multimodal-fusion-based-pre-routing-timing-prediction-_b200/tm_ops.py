"""Host-side operators over ``libtm_b200``: GNN propagation, mask fusion, MLPs.

Two layers:

* plain functions (``gnn_forward`` / ``gnn_backward`` / ``fusion_*`` / ``mlp2_*``) that launch the
  CUDA kernels on the current stream and return raw tensors -- used by the fused design step
  (``tm_engine.py``) with no autograd bookkeeping;
* ``torch.autograd.Function`` wrappers (``GnnPropagateFn``, ``MaskFusionFn``, ``LinearFn``) over the
  same functions -- used by the drop-in ``nn.Module`` surface (``model.py``) so that the reference's
  ``train.py`` loop (``loss.backward(retain_graph=True)``, anomaly mode) works unchanged.
  Saved buffers are never freed or overwritten in ``backward`` (SURVEY.md D9).

Reference semantics: src/model.py:10-24 (MLP), :88-116,:138-213 (PathConv), :269-292 (PathModel),
src/train.py:500-501 (mask fusion).
"""
import os

import torch

import tm_lib
from tm_lib import call, stream

D = 128
BIAS, RELU, MASK, ACCUM = 1, 2, 4, 8

# Arithmetic of the dense contractions (MLPs, weight gradients):
#   "tf32x3" tcgen05 kind::tf32, x = hi + lo with hi = the fp32 word itself (the tensor core reads its
#          upper 19 bits) and lo = x - trunc(x); hi*hi + hi*lo + lo*hi, fp32 accumulate in TMEM:
#          ~21-bit products, fp32-class accuracy -- the default for the rtol 1e-3 path;
#   "tf32" single-pass TF32 (11-bit operands);
#   "tc6"  bf16 operands split into three terms (24 bits), 6 MMAs;  "tc3": two terms, 3 MMAs;
#   "bf16" tcgen05 with plain bf16 operands (rtol 2e-2 class);
#   "fp32" the CUDA-core FFMA kernels (tm_gemm_nn / tm_gemm_tn).
MATH = os.environ.get("TM_MATH", "tf32x3")
FUSE_RUNS = os.environ.get("TM_FUSE_RUNS", "1") != "0"    # run-length / prefix-table mask fusion forward
TC_MIN_N = 4           # Linear(hid, 1) (the head's last layer): a 128 x 32 tensor-core tile would be 97 % padding
TC_MIN_K = 16          # contractions shorter than this stay on the CUDA-core kernel (K = 1, 2: pure bandwidth)


def _precision(math=None):
    m = math or MATH
    if m not in ("tf32x3", "tf32", "tc6", "tc3", "bf16", "fp32"):
        raise ValueError(f"unknown math mode {m!r}")
    return {"tf32x3": 3, "tf32": 4, "tc6": 2, "tc3": 1, "bf16": 0, "fp32": None}[m]


def _colsum(R, C, X, ld, rows, out, accumulate):
    nb = tm_lib.ws_bytes("tm_colsum_ws", R, C)
    call("tm_colsum", R, C, X, ld, rows, out, accumulate, tm_lib.workspace(nb, out.device), nb, stream())


class _Aux:
    """Helper stream for bandwidth-bound side work (bias-gradient column sums) that is independent of
    the tensor-core GEMM enqueued next to it: the persistent GEMM CTAs fill the shared memory of every
    SM but leave thread / register room, so a plain streaming kernel co-resides with them."""
    stream = None
    pending = []

    @classmethod
    def run(cls, fn, *tensors):
        if not torch.cuda.is_available():
            return fn()
        if cls.stream is None:
            cls.stream = torch.cuda.Stream()
        cur = torch.cuda.current_stream()
        if torch.cuda.is_current_stream_capturing() or cur == cls.stream:
            return fn()
        # every tensor passed in stays referenced by the caller until its aux_join(), so no
        # record_stream (which would stall the caching allocator's reuse of these large buffers)
        cls.stream.wait_stream(cur)
        with torch.cuda.stream(cls.stream):
            fn()
        cls.pending.append(cur)

    @classmethod
    def join(cls):
        """Make the current stream wait for everything posted from it."""
        if cls.stream is not None and cls.pending:
            torch.cuda.current_stream().wait_stream(cls.stream)
            cls.pending = []


def aux_join():
    _Aux.join()


def _f32c(t):
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _rowmajor(t):
    """2-D tensor usable as a strided row-major operand (unit inner stride)."""
    if t.dtype != torch.float32 or t.stride(-1) != 1:
        t = t.float().contiguous()
    return t


# --------------------------------------------------------------------------------------------
# thin wrappers
# --------------------------------------------------------------------------------------------
def gemm_nn(M, N, K, A, lda, B, ldb, C, ldc, a_rows=None, c_rows=None, bias=None, mask=None, ldmask=0, flags=0,
            b_is_nk=False, math=None):
    """C = epi(A @ B).  B is [K,N] row-major, or [N,K] (an nn.Linear weight as stored) with b_is_nk."""
    if bias is not None:
        flags |= BIAS
    if mask is not None:
        flags |= MASK
    prec = _precision(math)
    if N == 1 and b_is_nk and mask is None and not (flags & ACCUM) and M > 0:
        call("tm_rowdot", M, K, A, lda, a_rows, B, bias, C, ldc, c_rows, 1 if flags & RELU else 0, stream())
        return
    if prec is None or K < TC_MIN_K or N < TC_MIN_N:
        if b_is_nk:
            B, ldb = transpose(B[:, :K] if B.shape[1] != K else B), N
        call("tm_gemm_nn", M, N, K, A, lda, a_rows, B, ldb, C, ldc, c_rows, bias, mask, ldmask, flags, stream())
    else:
        if not b_is_nk and B.dim() == 2 and B.is_contiguous() and B.shape == (K, N) and B.numel() <= (1 << 22):
            # a [K,N] weight: hand the tensor cores the K-major [N,K] form (one tiny transpose
            # instead of an MN-major operand re-staged by every CTA)
            B, ldb, b_is_nk = transpose(B), K, True
        call("tm_tc_gemm_nn", M, N, K, A, lda, a_rows, B, ldb, 1 if b_is_nk else 0, C, ldc, c_rows, bias, mask,
             ldmask, flags, prec, tm_lib.err_flag(C.device), stream())


def gemm_tn(M, N, R, A, lda, B, ldb, C, ldc, a_rows=None, b_rows=None, colsum_a=None, colsum_b=None,
            accumulate=0, math=None):
    """C (+)= A^T @ B over the R rows; optional column sums of A / B (bias gradients)."""
    prec = _precision(math)
    if prec is None or (M < TC_MIN_K and N < TC_MIN_K):
        nb = tm_lib.ws_bytes("tm_gemm_tn_ws", M, N, R)
        ws = tm_lib.workspace(nb, C.device)
        call("tm_gemm_tn", M, N, R, A, lda, a_rows, B, ldb, b_rows, C, ldc, colsum_a, colsum_b, accumulate,
             ws, nb, stream())
        return
    nb = tm_lib.ws_bytes("tm_tc_gemm_tn_ws", M, N, R)
    ws = tm_lib.workspace(nb, C.device)
    if colsum_a is not None:
        _Aux.run(lambda: _colsum(R, M, A, lda, a_rows, colsum_a, accumulate), A, colsum_a, a_rows)
    if colsum_b is not None:
        _Aux.run(lambda: _colsum(R, N, B, ldb, b_rows, colsum_b, accumulate), B, colsum_b, b_rows)
    call("tm_tc_gemm_tn", M, N, R, A, lda, a_rows, B, ldb, b_rows, C, ldc, accumulate, prec, ws, nb,
         tm_lib.err_flag(C.device), stream())


def transpose(w):
    """(rows, cols) -> (cols, rows), contiguous."""
    w = _f32c(w)
    out = torch.empty(w.shape[1], w.shape[0], dtype=torch.float32, device=w.device)
    call("tm_transpose", w.shape[0], w.shape[1], w, out, stream())
    return out


def colsum(X, R, C, ld, out=None, accumulate=0):
    if out is None:
        out = torch.empty(C, dtype=torch.float32, device=X.device)
    _colsum(R, C, X, ld, None, out, accumulate)
    return out


# --------------------------------------------------------------------------------------------
# two-layer MLP (model.py:10-24 with sizes (in, hid, out)):  y = W2 relu(W1 x + b1) + b2
# --------------------------------------------------------------------------------------------
def _rows_aligned(t, ld):
    """Every row of ``t`` (row stride ``ld`` floats) starts on a 16-byte boundary: the fused kernels' vector loads."""
    return ld % 4 == 0 and t.data_ptr() % 16 == 0


def mlp2_route(n_rows, kin, hid, nout, math=None, x_aligned=True, out_aligned=True, g_aligned=True, dx_aligned=True):
    """The kernel that serves each product of the MLP kin -> hid -> nout over ``n_rows`` rows in arithmetic ``math``
    (default ``MATH``), given whether the rows of the input x, of the output, of the output's gradient g and of the
    input's gradient dx are 16-byte aligned.  Host logic only: ``mlp2_forward`` and ``mlp2_backward`` launch what it names.

    Returns a dict.  "hidden" is "generated" -- a Linear(<=2, hid) first layer costs 2 FMAs per hidden activation, so
    the kernels recompute the activations in their operand loaders and never store them -- or "stored".  The products:
    "lin1" / "lin2" the two forward layers (one kernel for both when the hidden layer is generated), "dw2" (dW2, db2),
    "dh" the hidden layer's gradient, "dw1" (dW1, db1), "dx" the data gradient next to the parameter gradients and
    "dx_only" the data gradient alone.  "gemm" is ``gemm_nn`` / ``gemm_tn``; a ``tm_*`` name is that kernel, where
    ``tm_selfmlp_gen_bwd1_dx`` is ``tm_selfmlp_gen_bwd1`` with dX in its epilogue.  The ``tm_selfmlp_*`` kernels
    (tm_selfmlp.cu) serve the reference's sizes at tf32x3 on the fp16 two-term split: 256 hidden units, 128 outputs for
    the second layer and its gradients, at most 48 inputs (a multiple of 4) for a stored first layer."""
    prec = _precision(math)
    split = prec == 3 and hid == 256
    split_out = split and nout == 128
    split_in = split and kin % 4 == 0 and kin <= 48
    if kin <= 2 and prec is not None and n_rows > 0 and hid >= TC_MIN_K:
        fwd = "tm_selfmlp_gen_forward" if split_out and out_aligned else "tm_tc_mlp2_smallk_forward"
        if split_out and g_aligned:
            return dict(hidden="generated", lin1=fwd, lin2=fwd, dw2="tm_selfmlp_gen_wgrad2", dh="tm_selfmlp_gen_bwd1",
                        dw1="tm_selfmlp_gen_bwd1", dx="tm_selfmlp_gen_bwd1_dx", dx_only="tm_selfmlp_gen_bwd1_dx")
        return dict(hidden="generated", lin1=fwd, lin2=fwd, dw2="tm_tc_mlp2_smallk_wgrad2", dh="gemm",
                    dw1="tm_tc_mlp1_bwd_fused", dx="gemm", dx_only="gemm")
    lin1 = "tm_selfmlp_lin1_relu" if split_in and n_rows > 0 and x_aligned else "gemm"
    # the fused second layer scales each row by the row maximum tm_selfmlp_lin1_relu writes
    lin2 = "tm_selfmlp_rows_forward" if lin1 != "gemm" and split_out and out_aligned else "gemm"
    dh = "tm_selfmlp_rows_dh" if split_out and g_aligned else "gemm"
    dx_only = "tm_selfmlp_rows_dx" if dh != "gemm" and split_in and dx_aligned else "gemm"
    return dict(hidden="stored", lin1=lin1, lin2=lin2, dw2="gemm", dh=dh, dw1="gemm", dx="gemm", dx_only=dx_only)


def mlp2_forward(x, ldx, rows, n_rows, w1, b1, w2, b2, out, ldo, out_rows=None, h_out=None):
    """x rows (optionally gathered by ``rows``) -> out rows (optionally scattered by ``out_rows``), on the kernels
    ``mlp2_route`` names.  Returns the hidden activations (n_rows, hid) needed by ``mlp2_backward``, or None when the
    route generates them.  ``h_out``: a contiguous (n_rows, hid) float32 tensor the stored hidden activations are
    written to (and returned) instead of a new one."""
    hid, kin = w1.shape
    nout = w2.shape[0]
    dev = out.device
    r = mlp2_route(n_rows, kin, hid, nout, x_aligned=_rows_aligned(x, ldx), out_aligned=_rows_aligned(out, ldo))
    if r["lin1"] == "tm_selfmlp_gen_forward":
        nb = tm_lib.ws_bytes("tm_selfmlp_ws_bytes")
        call("tm_selfmlp_gen_forward", n_rows, x, ldx, rows, kin, _f32c(w1), _f32c(b1), _f32c(w2), _f32c(b2), out, ldo,
             out_rows, tm_lib.workspace(nb, dev), nb, stream())
        return None
    if r["lin1"] == "tm_tc_mlp2_smallk_forward":
        call("tm_tc_mlp2_smallk_forward", n_rows, hid, nout, x, ldx, rows, kin, _f32c(w1), _f32c(b1), _f32c(w2), _f32c(b2),
             out, ldo, out_rows, _precision(), tm_lib.err_flag(dev), stream())
        return None
    h = torch.empty(n_rows, hid, dtype=torch.float32, device=dev) if h_out is None else h_out
    rowmax = None
    if r["lin1"] == "tm_selfmlp_lin1_relu":
        nb = tm_lib.ws_bytes("tm_selfmlp_lin1_ws_bytes")
        if r["lin2"] == "tm_selfmlp_rows_forward":
            rowmax = torch.empty(n_rows, dtype=torch.float32, device=dev)
        call("tm_selfmlp_lin1_relu", n_rows, x, ldx, rows, kin, _f32c(w1), _f32c(b1), h, hid, rowmax,
             tm_lib.workspace(nb, dev), nb, stream())
    else:
        gemm_nn(n_rows, hid, kin, x, ldx, _f32c(w1), kin, h, hid, a_rows=rows, bias=b1, flags=RELU, b_is_nk=True)
    if r["lin2"] == "tm_selfmlp_rows_forward":
        nb = tm_lib.ws_bytes("tm_selfmlp_ws_bytes")
        call("tm_selfmlp_rows_forward", n_rows, h, hid, None, rowmax, _f32c(w2), _f32c(b2), out, ldo, out_rows,
             tm_lib.workspace(nb, dev), nb, stream())
    else:
        gemm_nn(n_rows, nout, hid, h, hid, _f32c(w2), hid, out, ldo, c_rows=out_rows, bias=b2, b_is_nk=True)
    return h


def _hidden_grad(r, n_rows, g, ldg, g_rows, w2, h, h_rows, dh):
    """dh[r] = (g[g_rows] @ w2) * (h[r] > 0), r = h_rows or the row itself."""
    nout, hid = w2.shape
    if r["dh"] == "tm_selfmlp_rows_dh":
        nb = tm_lib.ws_bytes("tm_selfmlp_rows_dh_ws_bytes")
        call("tm_selfmlp_rows_dh", n_rows, g, ldg, g_rows, w2, h, h.stride(0), h_rows, dh, dh.stride(0),
             tm_lib.workspace(nb, dh.device), nb, stream())
    else:
        gemm_nn(n_rows, hid, nout, g, ldg, w2, hid, dh, hid, a_rows=g_rows, c_rows=h_rows, mask=h, ldmask=hid)


def mlp2_backward(x, ldx, rows, n_rows, w1, w2, h, g, ldg, g_rows=None, need_dx=False, b1=None, wgrad_stream=None,
                  h_rows=None, dx_out=None, need_wgrad=True):
    """Gradients of a two-layer MLP, on the kernels ``mlp2_route`` names.  ``g``: dLoss/d(out) rows (optionally gathered
    by ``g_rows``).  ``h``: the hidden activations mlp2_forward returned, or None when they were generated on the fly
    (then ``b1`` is required).  Returns (dw1, db1, dw2, db2, dx or None).
    ``wgrad_stream`` (with ``need_dx``): the data gradient is computed first on the current stream and the four
    parameter gradients on ``wgrad_stream`` (which waits for it); the caller joins that stream before reading them.
    ``h_rows``: row of ``h`` that belongs to MLP row i (default i) -- set when ``rows`` / ``g_rows`` are a subset of
    the rows the forward pass ran on (``tm_graph.BackwardCone``).
    ``dx_out`` (with ``need_dx``; required when ``rows`` gathers): the data gradient of MLP row i is written to row
    ``rows[i]`` of ``dx_out`` -- the row of ``x`` it read, so ``rows`` must be distinct -- and ``dx_out`` is returned as dx;
    its other rows are left as they are.  The parameter gradients are the same bits as without ``need_dx``.
    ``need_wgrad=False`` (with ``need_dx``): the data gradient alone, the same launches without the parameter-gradient
    ones; returns (None, None, None, None, dx).  dx is the same bits as with the parameter gradients, except where the
    route has a kernel for the data gradient alone (a stored hidden layer of the reference's sizes, ``fc_cell_self``:
    ``tm_selfmlp_rows_dx`` sums the second product in another order)."""
    hid, kin = w1.shape
    nout = w2.shape[0]
    dev = g.device
    if not need_wgrad and not need_dx:
        raise RuntimeError("mlp2_backward: need_wgrad=False needs need_dx")
    if need_dx and h_rows is not None:
        raise RuntimeError("mlp2_backward: h_rows has no dx path")
    if need_dx and dx_out is None:
        if rows is not None:
            raise RuntimeError("mlp2_backward: a data gradient of gathered rows needs dx_out")
        dx_out = torch.empty(n_rows, kin, dtype=torch.float32, device=dev)
    dw1 = db1 = dw2 = db2 = None
    if need_wgrad:
        dw2 = torch.empty(nout, hid, dtype=torch.float32, device=dev)
        db2 = torch.empty(nout, dtype=torch.float32, device=dev)
        dw1 = torch.empty(hid, kin, dtype=torch.float32, device=dev)
        db1 = torch.empty(hid, dtype=torch.float32, device=dev)
    if n_rows == 0:
        if need_wgrad:
            for t in (dw1, db1, dw2, db2):
                t.zero_()
        return dw1, db1, dw2, db2, dx_out
    r = mlp2_route(n_rows, kin, hid, nout, g_aligned=_rows_aligned(g, ldg),
                   dx_aligned=need_dx and _rows_aligned(dx_out, dx_out.stride(0)))
    if (h is None) != (r["hidden"] == "generated"):
        raise RuntimeError(f"mlp2_backward: h is not what mlp2_forward returns for this MLP in {MATH} "
                           f"(hidden layer {r['hidden']})")
    w1, w2 = _f32c(w1), _f32c(w2)
    if h is None:
        if b1 is None:
            raise RuntimeError("mlp2_backward: generated hidden activations need b1")
        b1 = _f32c(b1)
        if need_wgrad and r["dw2"] == "tm_selfmlp_gen_wgrad2":
            # bias gradient and max |g| in one pass, then the fused weight-gradient kernel (hidden layer generated as
            # a tcgen05 operand, accumulators resident in TMEM)
            gmax = torch.empty(1, dtype=torch.float32, device=dev)
            nbc = tm_lib.ws_bytes("tm_colsum_ws", n_rows, nout)
            call("tm_colsum_absmax", n_rows, nout, g, ldg, g_rows, db2, gmax, tm_lib.workspace(nbc, dev), nbc, stream())
            nb = tm_lib.ws_bytes("tm_selfmlp_wgrad2_ws_bytes")
            call("tm_selfmlp_gen_wgrad2", n_rows, g, ldg, g_rows, x, ldx, rows, kin, w1, b1, gmax, dw2,
                 tm_lib.workspace(nb, dev), nb, stream())
        elif need_wgrad:
            _Aux.run(lambda: _colsum(n_rows, nout, g, ldg, g_rows, db2, 0), g, db2, g_rows)
            nb = tm_lib.ws_bytes("tm_tc_gemm_tn_ws", nout, hid, n_rows)
            call("tm_tc_mlp2_smallk_wgrad2", nout, hid, n_rows, g, ldg, g_rows, x, ldx, rows, kin, w1, b1, dw2,
                 _precision(), tm_lib.workspace(nb, dev), nb, tm_lib.err_flag(dev), stream())
        if r["dw1"] == "tm_selfmlp_gen_bwd1":
            nb = tm_lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")
            if need_dx:                                      # dW1 / db1 NULL: the data gradient alone
                call("tm_selfmlp_gen_bwd1_dx", n_rows, g, ldg, g_rows, x, ldx, rows, kin, w1, b1, w2,
                     dw1, db1, dx_out, dx_out.stride(0), tm_lib.workspace(nb, dev), nb, stream())
            else:
                call("tm_selfmlp_gen_bwd1", n_rows, g, ldg, g_rows, x, ldx, rows, kin, w1, b1, w2,
                     dw1, db1, tm_lib.workspace(nb, dev), nb, stream())
        else:
            if need_wgrad:
                nb = tm_lib.ws_bytes("tm_tc_mlp1_bwd_ws", hid)
                call("tm_tc_mlp1_bwd_fused", n_rows, hid, nout, g, ldg, g_rows, transpose(w2), None, 0, x, ldx, rows, kin,
                     w1, b1, dw1, db1, tm_lib.workspace(nb, dev), nb, tm_lib.err_flag(dev), stream())
            if need_dx:
                # no fused data-gradient kernel on this route: the hidden layer is materialised for the data
                # gradient alone (the parameter gradients above are untouched)
                hm = torch.empty(n_rows, hid, dtype=torch.float32, device=dev)
                gemm_nn(n_rows, hid, kin, x, ldx, w1, kin, hm, hid, a_rows=rows, bias=b1, flags=RELU, b_is_nk=True)
                dh = torch.empty(n_rows, hid, dtype=torch.float32, device=dev)
                _hidden_grad(r, n_rows, g, ldg, g_rows, w2, hm, None, dh)
                gemm_nn(n_rows, kin, hid, dh, hid, w1, kin, dx_out, dx_out.stride(0), c_rows=rows)
        aux_join()
        return dw1, db1, dw2, db2, dx_out
    if not need_wgrad and r["dx_only"] == "tm_selfmlp_rows_dx":
        # one pass: the hidden layer's gradient never leaves the SM
        nb = tm_lib.ws_bytes("tm_selfmlp_rows_dh_ws_bytes")
        call("tm_selfmlp_rows_dx", n_rows, g, ldg, g_rows, w2, h, h.stride(0), None, w1, kin, dx_out,
             dx_out.stride(0), rows, tm_lib.workspace(nb, dev), nb, stream())
        return None, None, None, None, dx_out
    on_side = need_dx and wgrad_stream is not None
    if need_wgrad and not on_side:
        gemm_tn(nout, hid, n_rows, g, ldg, h, hid, dw2, hid, a_rows=g_rows, b_rows=h_rows, colsum_a=db2)
    # with h_rows, dh lives in the rows of h it belongs to, so the ReLU mask of the epilogue reads the matching row
    dh = torch.empty(n_rows if h_rows is None else h.shape[0], hid, dtype=torch.float32, device=dev)
    _hidden_grad(r, n_rows, g, ldg, g_rows, w2, h, h_rows, dh)
    if need_wgrad and not on_side:
        gemm_tn(hid, kin, n_rows, dh, hid, x, ldx, dw1, kin, a_rows=h_rows, b_rows=rows, colsum_a=db1)
    if need_dx:
        gemm_nn(n_rows, kin, hid, dh, hid, w1, kin, dx_out, dx_out.stride(0), c_rows=rows)
    if need_wgrad and on_side:
        wgrad_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(wgrad_stream):
            gemm_tn(nout, hid, n_rows, g, ldg, h, hid, dw2, hid, a_rows=g_rows, colsum_a=db2)
            gemm_tn(hid, kin, n_rows, dh, hid, x, ldx, dw1, kin, b_rows=rows, colsum_a=db1)
            aux_join()
    aux_join()
    return dw1, db1, dw2, db2, dx_out


# --------------------------------------------------------------------------------------------
# GNN propagation
# --------------------------------------------------------------------------------------------
GNN_PARAM_NAMES = ("fc_cell_self.layers.0.weight", "fc_cell_self.layers.0.bias",
                   "fc_cell_self.layers.2.weight", "fc_cell_self.layers.2.bias",
                   "fc_net_self.layers.0.weight", "fc_net_self.layers.0.bias",
                   "fc_net_self.layers.2.weight", "fc_net_self.layers.2.bias",
                   "fc_cell_neigh.layers.0.weight", "fc_cell_neigh.layers.0.bias",
                   "fc_cell_neigh.layers.2.weight", "fc_cell_neigh.layers.2.bias")


def gnn_forward(sched, cell_feat, net_feat, params, save=True, impl=None, x_rows=None):
    """Full propagation over every level.  ``params``: the 12 tensors of GNN_PARAM_NAMES.
    Returns ``(H, saved)``; H is (N, 128) with zeros on pins outside the schedule.
    ``impl``: back end for this call (``tm_gnn_set_impl`` bits; None = the process default, which runs the
    forward as ONE persistent cluster kernel).  The persistent kernel owns every SM while it runs, so a
    caller that overlaps the propagation with other streams (``DesignStep``) asks for 0, the chain of
    small per-level kernels that co-resides with them.
    ``x_rows`` = (rows of ``cell_feat`` for ``sched.cell_class``, rows of ``net_feat`` for ``sched.net_class``) when the
    schedule is a sub-netlist whose pins are renumbered (``tm_graph.ConeGraph``); default: the pin ids themselves."""
    (cs1w, cs1b, cs2w, cs2b, ns1w, ns1b, ns2w, ns2b, cn1w, cn1b, cn2w, cn2b) = [_f32c(p) for p in params]
    if cn2w.shape[0] != D or cs2w.shape[0] != D or ns2w.shape[0] != D or cn1w.shape != (256, D):
        raise RuntimeError("the CUDA propagation kernels are built for out_feat_dim = hidden_feat_dim = 128 "
                           "with 256-wide MLPs (the reference configuration, options.py:10)")
    cell_feat, net_feat = _rowmajor(cell_feat), _rowmajor(net_feat)
    tm_lib.require_cuda(cell_feat, "cell_feat")
    dev = cell_feat.device
    n = sched.n
    S = torch.empty(n, D, dtype=torch.float32, device=dev)
    nc, nn_ = int(sched.cell_class.numel()), int(sched.net_class.numel())
    xc, xn = x_rows if x_rows is not None else (sched.cell_class, sched.net_class)
    hc = mlp2_forward(cell_feat, cell_feat.stride(0), xc, nc, cs1w, cs1b, cs2w, cs2b, S, D, out_rows=sched.cell_class)
    hn = mlp2_forward(net_feat, net_feat.stride(0), xn, nn_, ns1w, ns1b, ns2w, ns2b, S, D, out_rows=sched.net_class)
    # every scheduled pin's row is written by its level's kernel: only pins outside the schedule need the zero fill
    # (170 MB = 42 us of the config-2 step when every pin is scheduled, as in the reference's designs)
    if sched.n_sched == n and os.environ.get("TM_H_FILL") != "1":
        H = torch.empty(n, D, dtype=torch.float32, device=dev)
    else:
        H = torch.zeros(n, D, dtype=torch.float32, device=dev)
    ncr = sched.n_cell_rows
    A = LSE = HID = None
    if save:
        A = torch.empty(max(ncr, 1), D, dtype=torch.float32, device=dev)
        LSE = torch.empty(max(ncr, 1), D, dtype=torch.float32, device=dev)
        HID = torch.empty(max(ncr, 1), 256, dtype=torch.float32, device=dev)
    w1t, w2t = transpose(cn1w), transpose(cn2w)
    nb = tm_lib.ws_bytes("tm_gnn_ws_bytes")
    old = tm_lib.lib().tm_gnn_set_impl(impl) if impl is not None else None
    try:
        call("tm_gnn_forward", sched.struct, 0, sched.num_levels, H, S, w1t, cn1b, w2t, cn2b, A, LSE, HID,
             tm_lib.workspace(nb, dev), nb, stream())
    finally:
        if old is not None:
            tm_lib.lib().tm_gnn_set_impl(old)
    saved = dict(H=H, A=A, LSE=LSE, HID=HID, hc=hc, hn=hn, cell_feat=cell_feat, net_feat=net_feat, x_rows=x_rows) if save else None
    return H, saved


def gnn_self_terms(S, cell_feat, net_feat, params, cell_pins, net_pins, cell_out=None, net_out=None):
    """Rewrite the rows of the hoisted self terms ``S`` (N, 128) of the given pins: ``cell_pins`` (int32 device, pins
    on even levels) through ``fc_cell_self(cell_feat[pin])``, ``net_pins`` (odd levels) through
    ``fc_net_self(net_feat[pin])`` -- the split of ``Schedule.cell_class`` / ``net_class``.  With those two class lists
    these are exactly the launches ``gnn_forward`` makes; a pin's row does not depend on which other pins are listed
    (every route of ``mlp2_route`` scales per row and tiles rows independently).  Other rows are left alone.
    ``cell_out`` / ``net_out`` (int32 device, as long as the pin lists): write row i to ``S[cell_out[i]]`` instead
    of ``S[cell_pins[i]]`` (what-if evaluation: candidate rows into their virtual rows)."""
    (cs1w, cs1b, cs2w, cs2b, ns1w, ns1b, ns2w, ns2b) = [_f32c(p) for p in params[:8]]
    cell_feat, net_feat = _rowmajor(cell_feat), _rowmajor(net_feat)
    nc, nn_ = int(cell_pins.numel()), int(net_pins.numel())
    if nc:
        mlp2_forward(cell_feat, cell_feat.stride(0), cell_pins, nc, cs1w, cs1b, cs2w, cs2b, S, D,
                     out_rows=cell_pins if cell_out is None else cell_out)
    if nn_:
        mlp2_forward(net_feat, net_feat.stride(0), net_pins, nn_, ns1w, ns1b, ns2w, ns2b, S, D,
                     out_rows=net_pins if net_out is None else net_out)


def gnn_forward_cone(cone, H, S, params):
    """Re-propagate H (N, 128) in place over a sub-schedule -- ``cone`` a ``tm_graph.ForwardCone`` after ``build``, or a
    whole ``Schedule`` -- from the self terms ``S``: the persistent forward kernel over the schedule's levels, whatever
    ``tm_gnn_set_impl`` says, nothing saved.  Rows of the schedule's pins are rewritten (the same bits as the persistent
    ``gnn_forward`` writes for them given the same sources), every other row is only read."""
    cn1w, cn1b, cn2w, cn2b = [_f32c(p) for p in params[8:12]]
    w1t, w2t = transpose(cn1w), transpose(cn2w)
    nb = tm_lib.ws_bytes("tm_gnn_ws_bytes")
    call("tm_gnn_forward_cone", cone.struct, H, S, w1t, cn1b, w2t, cn2b, tm_lib.workspace(nb, H.device), nb, stream())


def gnn_backward(sched, saved, params, G, cone=None, need_dx=False, need_wgrad=True):
    """``G`` (N,128): dLoss/dH, consumed (overwritten with dLoss/d pre-activation).
    Returns the 12 parameter gradients in GNN_PARAM_NAMES order.
    ``cone`` (``tm_graph.BackwardCone`` of the endpoints that seeded G): the weight-gradient contractions run over
    the cone's rows only -- every other row of dLoss/dz is exactly zero.
    ``need_dx``: returns ``(grads, dcell_feat, dnet_feat)``, the gradients with respect to the features, shaped like
    the ``cell_feat`` / ``net_feat`` the forward read.  The self-term S enters each pin's pre-activation linearly, so
    after the sweep G is dLoss/dS and the feature gradient is the self MLPs' data gradient of it.  Rows the
    propagation never reads are exactly zero: net-class pins in ``dcell_feat``, cell-class pins in ``dnet_feat``,
    unscheduled pins in both.  The parameter gradients are the same bits as without ``need_dx``.
    ``need_wgrad=False`` (with ``need_dx``): the feature gradients alone, ``(None, dcell_feat, dnet_feat)``; the sweep
    stores no weight-gradient operands and no parameter gradient is computed.  G and dnet_feat are the same bits;
    dcell_feat comes from the fused ``fc_cell_self`` data-gradient kernel (``tm_selfmlp_rows_dx``)."""
    if need_dx and cone is not None:
        raise RuntimeError("gnn_backward: a BackwardCone has no feature-gradient path")
    if not need_wgrad and not need_dx:
        raise RuntimeError("gnn_backward: need_wgrad=False needs need_dx")
    (cs1w, cs1b, cs2w, cs2b, ns1w, ns1b, ns2w, ns2b, cn1w, cn1b, cn2w, cn2b) = [_f32c(p) for p in params]
    dev = G.device
    ncr = sched.n_cell_rows
    GA = torch.empty(max(ncr, 1), D, dtype=torch.float32, device=dev)
    GHID = GZC = None                                           # the fc_cell_neigh weight-gradient operands
    if need_wgrad:
        GHID = torch.empty(max(ncr, 1), 256, dtype=torch.float32, device=dev)
        GZC = torch.empty(max(ncr, 1), D, dtype=torch.float32, device=dev)
    nb = tm_lib.ws_bytes("tm_gnn_ws_bytes")
    call("tm_gnn_backward", sched.struct, saved["H"], G, cn1w, cn2w, saved["A"], saved["LSE"], saved["HID"],
         GA, GHID, GZC, tm_lib.workspace(nb, dev), nb, stream())
    if need_wgrad:
        dcn2w = torch.empty(D, 256, dtype=torch.float32, device=dev)
        dcn2b = torch.empty(D, dtype=torch.float32, device=dev)
        dcn1w = torch.empty(256, D, dtype=torch.float32, device=dev)
        dcn1b = torch.empty(256, dtype=torch.float32, device=dev)
        cr = cone.crows if cone is not None else None
        if cr is not None:
            ncr = int(cr.numel())
        if ncr > 0:
            gemm_tn(D, 256, ncr, GZC, D, saved["HID"], 256, dcn2w, 256, a_rows=cr, b_rows=cr, colsum_a=dcn2b)
            gemm_tn(256, D, ncr, GHID, 256, saved["A"], D, dcn1w, D, a_rows=cr, b_rows=cr, colsum_a=dcn1b)
            aux_join()
        else:
            for t in (dcn2w, dcn2b, dcn1w, dcn1b):
                t.zero_()
    cf, nf = saved["cell_feat"], saved["net_feat"]
    cpins, npins, cpos, npos = sched.cell_class, sched.net_class, None, None
    xc, xn = saved.get("x_rows") or (cpins, npins)            # feature rows of the two classes
    if cone is not None:
        if saved.get("x_rows") is not None:
            raise RuntimeError("gnn_backward: a BackwardCone on top of a renumbered sub-netlist is not supported")
        cpins, npins = cone.cell_pins, cone.net_pins
        xc, xn = cpins, npins
        cpos = cone.cell_pos if saved["hc"] is not None else None
        npos = cone.net_pos if saved["hn"] is not None else None
    dcf = torch.zeros(cf.shape, dtype=torch.float32, device=dev) if need_dx else None
    dnf = torch.zeros(nf.shape, dtype=torch.float32, device=dev) if need_dx else None
    dcs1w, dcs1b, dcs2w, dcs2b, _ = mlp2_backward(cf, cf.stride(0), xc, int(cpins.numel()), cs1w, cs2w, saved["hc"], G, D,
                                                  g_rows=cpins, b1=cs1b, h_rows=cpos, need_dx=need_dx, dx_out=dcf,
                                                  need_wgrad=need_wgrad)
    dns1w, dns1b, dns2w, dns2b, _ = mlp2_backward(nf, nf.stride(0), xn, int(npins.numel()), ns1w, ns2w, saved["hn"], G, D,
                                                  g_rows=npins, b1=ns1b, h_rows=npos, need_dx=need_dx, dx_out=dnf,
                                                  need_wgrad=need_wgrad)
    if not need_wgrad:
        return None, dcf, dnf
    grads = (dcs1w, dcs1b, dcs2w, dcs2b, dns1w, dns1b, dns2w, dns2b, dcn1w, dcn1b, dcn2w, dcn2b)
    return (grads, dcf, dnf) if need_dx else grads


def gnn_cone_scratch(sched, device):
    """The buffers ``gnn_backward_cone`` works in, sized by the parent ``sched``: A / LSE / GA (n_cell_rows, 128) and HID
    (max(n_cell_rows, pins on even levels), 256), which after the sweep holds the ``fc_cell_self`` hidden rows."""
    ncr = max(sched.n_cell_rows, 1)
    hid_rows = max(ncr, int(sched.cell_class.numel()))
    f32 = lambda r, c: torch.empty(r, c, dtype=torch.float32, device=device)     # noqa: E731
    return dict(A=f32(ncr, D), LSE=f32(ncr, D), GA=f32(ncr, D), HID=f32(hid_rows, 256))


def gnn_backward_cone(cone, H, G, params, cell_feat, net_feat, dcell, dnet, scratch, mark=None):
    """The feature gradients of ``gnn_backward(..., need_dx=True, need_wgrad=False)`` over a ``tm_graph.FaninCone``
    after ``build``, from the final ``H`` of a forward (every source of a cone pin is final there):

    1. ``tm_gnn_save_cone``: A / LSE / HID of the cone's cell pins recomputed from H (what the forward would have saved);
    2. ``tm_gnn_backward_cone``: the persistent data-gradient sweep over the cone; ``G`` (n, 128) holds dLoss/dH on the
       cone's pins on entry (the head's gradient; zero elsewhere in the cone) and dLoss/dS on exit;
    3. the self-MLP data gradients over the cone's class lists, with device row counts: ``fc_cell_self``'s hidden rows
       recomputed (``tm_selfmlp_lin1_relu_dcount``) then ``tm_selfmlp_rows_dx_dcount``; ``fc_net_self`` through
       ``tm_selfmlp_gen_bwd1_dx_dcount``.  Those are the routes ``mlp2_route`` gives the full backward (they depend on
       the row count only through ``n_rows > 0``); in another arithmetic than tf32x3 there is no device-count kernel
       and this raises.

    Rows of ``dcell`` / ``dnet`` (shaped like the features) of the cone's pins are written; the caller zeroes the rest.
    Every row written is the same bits as the full backward's.  ``scratch``: ``gnn_cone_scratch``.  ``mark(phase)``,
    when given, is called after each of the three stages ("recompute", "backward", "self_dx": diagnostics)."""
    (cs1w, cs1b, cs2w, cs2b, ns1w, ns1b, ns2w, ns2b, cn1w, cn1b, cn2w, cn2b) = [_f32c(p) for p in params]
    cell_feat, net_feat = _rowmajor(cell_feat), _rowmajor(net_feat)
    cap_c, cap_n = cone.n_cell_cap, cone.n_net_cap
    rc = mlp2_route(cap_c, cs1w.shape[1], cs1w.shape[0], cs2w.shape[0], x_aligned=_rows_aligned(cell_feat, cell_feat.stride(0)),
                    dx_aligned=_rows_aligned(dcell, dcell.stride(0)))
    rn = mlp2_route(cap_n, ns1w.shape[1], ns1w.shape[0], ns2w.shape[0], g_aligned=_rows_aligned(G, D),
                    dx_aligned=_rows_aligned(dnet, dnet.stride(0)))
    if (cap_c and (rc["lin1"], rc["dx_only"]) != ("tm_selfmlp_lin1_relu", "tm_selfmlp_rows_dx")) or \
            (cap_n and rn["dx_only"] != "tm_selfmlp_gen_bwd1_dx"):
        raise RuntimeError(f"gnn_backward_cone: the self-term MLPs route to {rc['dx_only']} / {rn['dx_only']} in {MATH}; "
                           "only the fused tf32x3 kernels take a device row count")
    dev = H.device
    nb = tm_lib.ws_bytes("tm_gnn_ws_bytes")
    ws = tm_lib.workspace(nb, dev)
    call("tm_gnn_save_cone", cone.struct, H, transpose(cn1w), cn1b, transpose(cn2w), scratch["A"], scratch["LSE"],
         scratch["HID"], ws, nb, stream())
    if mark:
        mark("recompute")
    call("tm_gnn_backward_cone", cone.struct, H, G, cn1w, cn2w, scratch["A"], scratch["LSE"], scratch["HID"],
         scratch["GA"], ws, nb, stream())
    if mark:
        mark("backward")
    hc = scratch["HID"]                                        # free after the sweep: fc_cell_self's hidden rows
    counts = cone.counts
    if cap_c:
        nb = tm_lib.ws_bytes("tm_selfmlp_lin1_ws_bytes")
        call("tm_selfmlp_lin1_relu_dcount", cap_c, counts[1:], cell_feat, cell_feat.stride(0), cone.cell_pins,
             cs1w.shape[1], cs1w, cs1b, hc, 256, tm_lib.workspace(nb, dev), nb, stream())
        nb = tm_lib.ws_bytes("tm_selfmlp_rows_dh_ws_bytes")
        call("tm_selfmlp_rows_dx_dcount", cap_c, counts[1:], G, D, cone.cell_pins, cs2w, hc, 256, None, cs1w,
             cs1w.shape[1], dcell, dcell.stride(0), cone.cell_pins, tm_lib.workspace(nb, dev), nb, stream())
    if cap_n:
        nb = tm_lib.ws_bytes("tm_selfmlp_bwd1_ws_bytes")
        call("tm_selfmlp_gen_bwd1_dx_dcount", cap_n, counts[2:], G, D, cone.net_pins, net_feat, net_feat.stride(0),
             cone.net_pins, ns1w.shape[1], ns1w, ns1b, ns2w, dnet, dnet.stride(0), tm_lib.workspace(nb, dev), nb,
             stream())
    if mark:
        mark("self_dx")


class GnnPropagateFn(torch.autograd.Function):
    """H = propagate(cell_feat, net_feat; 12 PathConv parameters) over a fixed Schedule."""

    @staticmethod
    def forward(ctx, sched, cell_feat, net_feat, need, *params):
        H, saved = gnn_forward(sched, cell_feat, net_feat, [p.detach() for p in params], save=need)
        ctx.sched, ctx.saved = sched, saved
        ctx.params = [p.detach() for p in params]
        return H

    @staticmethod
    def backward(ctx, gH):
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            raise NotImplementedError("PathConv: gradients w.r.t. cell_feat / net_feat are not implemented; the "
                                      "propagation differentiates its parameters only (set requires_grad=False on "
                                      "the features)")
        G = gH.contiguous().clone()                      # consumed in place by the sweep
        grads = gnn_backward(ctx.sched, ctx.saved, ctx.params, G)
        return (None, None, None, None) + tuple(grads)


def step_metrics(pred, arrival, required=None, label=None):
    """One launch, one (8,) device tensor [mse, r2, correct, tp, fn, tn, fp, T] instead of the seven
    ``.item()`` round trips of train.py:513-549.  ``label``: int64 (0 = non-critical)."""
    pred, arrival = _f32c(pred.detach().reshape(-1)), _f32c(arrival.detach().reshape(-1))
    tm_lib.require_cuda(pred, "pred")
    out = torch.empty(8, dtype=torch.float32, device=pred.device)
    req = None if required is None else _f32c(required.detach().reshape(-1))
    lab = None if label is None else label.detach().reshape(-1).to(torch.int64).contiguous()
    call("tm_step_metrics", int(pred.numel()), pred, arrival, req, lab, out, stream())
    return out


EVAL_COLUMNS = ("mse", "r2", "correct", "tp", "fn", "tn", "fp", "count", "mape")


def eval_metrics(pred, arrival, seg_ptr, seg_idx, required=None, label=None):
    """``step_metrics`` per segment, one launch: segment s is the endpoints ``seg_idx[seg_ptr[s]:seg_ptr[s + 1]]``
    (int32 device tensors).  Returns the (n_seg, 9) float32 device tensor whose columns are ``EVAL_COLUMNS``: the eight
    of ``step_metrics`` (the last one the segment's endpoint count) and the mean absolute percentage error."""
    pred, arrival = _f32c(pred.detach().reshape(-1)), _f32c(arrival.detach().reshape(-1))
    tm_lib.require_cuda(pred, "pred")
    if seg_ptr.dtype != torch.int32 or seg_idx.dtype != torch.int32:
        raise ValueError("eval_metrics: seg_ptr and seg_idx must be int32")
    n_seg = int(seg_ptr.numel()) - 1
    out = torch.empty(max(n_seg, 0), len(EVAL_COLUMNS), dtype=torch.float32, device=pred.device)
    req = None if required is None else _f32c(required.detach().reshape(-1))
    lab = None if label is None else label.detach().reshape(-1).to(torch.int64).contiguous()
    call("tm_eval_metrics", n_seg, seg_ptr.contiguous(), seg_idx.contiguous(), pred, arrival, req, lab, out, stream())
    return out


# --------------------------------------------------------------------------------------------
# mask fusion
# --------------------------------------------------------------------------------------------
def fusion_forward(mask_rows, feat, fcn_w, fcn_b, out, ldo):
    """out[t, 0:128] = fcn(mask_t * feat)  (train.py:501 + model.py:272).  Returns fcn_w^T."""
    J = int(feat.numel())
    if fcn_w.shape != (D, J):
        raise RuntimeError(f"fcn must be Linear({J}, 128); got weight {tuple(fcn_w.shape)}")
    wt = transpose(fcn_w)
    if FUSE_RUNS:
        run_ptr, run_lo, run_hi = mask_rows.runs()
        nb = tm_lib.ws_bytes("tm_fuse_runs_ws", J)
        call("tm_fuse_forward_runs", mask_rows.T, J, D, run_ptr, run_lo, run_hi, feat, wt, _f32c(fcn_b), out, ldo,
             tm_lib.workspace(nb, feat.device), nb, stream())
    else:
        csr = mask_rows.csr
        call("tm_fuse_forward", mask_rows.T, J, D, csr.indptr, csr.cols, mask_rows.rows, feat, wt, _f32c(fcn_b),
             out, ldo, stream())
    return wt


def fusion_backward(mask_rows, feat, wt, g, ldg, need_wgrad=True):
    """Returns (dfeat (J,), dfcn_w (128,J), dfcn_b (128,)); ``need_wgrad=False``: (dfeat, None, None), dfeat the same
    bits."""
    J = int(feat.numel())
    dev = feat.device
    cptr, ct = mask_rows.csc()
    dwt = torch.empty(J, D, dtype=torch.float32, device=dev) if need_wgrad else None
    dF = torch.empty(J, dtype=torch.float32, device=dev)
    call("tm_fuse_backward", mask_rows.T, J, D, cptr, ct, g, ldg, feat, wt, dwt, dF, stream())
    if not need_wgrad:
        return dF, None, None
    db = colsum(g, mask_rows.T, D, ldg)
    return dF, transpose(dwt), db


def fusion_forward_multi(rows, tab, ep_off, feat, fcn_w, fcn_b, out, ldo):
    """Mask fusion of K designs in one launch: ``rows`` their ``MaskRows``, ``tab`` the device table of their
    run / CSC buffers, ``ep_off`` int32 (K+1,) endpoint offsets, ``feat`` (K*J,) their feature maps.  Row t of ``out``
    is what ``fusion_forward`` gives for its design.  K = 1 is ``fusion_forward``.  Returns fcn_w^T."""
    K = len(rows)
    if K == 1:
        return fusion_forward(rows[0], feat, fcn_w, fcn_b, out, ldo)
    J = int(feat.numel()) // K
    if fcn_w.shape != (D, J):
        raise RuntimeError(f"fcn must be Linear({J}, 128); got weight {tuple(fcn_w.shape)}")
    wt = transpose(fcn_w)
    nb = tm_lib.ws_bytes("tm_fuse_runs_multi_ws", K, J)
    call("tm_fuse_forward_runs_multi", K, sum(r.T for r in rows), J, D, tab, ep_off, feat, wt, _f32c(fcn_b), out, ldo,
         tm_lib.workspace(nb, feat.device), nb, stream())
    return wt


def fusion_backward_multi(rows, tab, ep_off, feat, wt, g, ldg, need_wgrad=True):
    """Returns (dfeat (K*J,), dfcn_w (128,J) summed over the designs, dfcn_b (128,)).  K = 1 is ``fusion_backward``.
    ``need_wgrad=False``: (dfeat, None, None)."""
    K = len(rows)
    if K == 1:
        return fusion_backward(rows[0], feat, wt, g, ldg, need_wgrad)
    J = int(feat.numel()) // K
    dev = feat.device
    dwt = torch.empty(J, D, dtype=torch.float32, device=dev) if need_wgrad else None
    dF = torch.empty(K * J, dtype=torch.float32, device=dev)
    call("tm_fuse_backward_multi", K, J, D, tab, ep_off, g, ldg, feat, wt, dwt, dF, stream())
    if not need_wgrad:
        return dF, None, None
    db = colsum(g, sum(r.T for r in rows), D, ldg)
    return dF, transpose(dwt), db


class MaskFusionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mask_rows, feat_flat, fcn_w, fcn_b):
        feat = _f32c(feat_flat.detach()).reshape(-1)
        out = torch.empty(mask_rows.T, D, dtype=torch.float32, device=feat.device)
        wt = fusion_forward(mask_rows, feat, fcn_w.detach(), fcn_b.detach(), out, D)
        ctx.mask_rows, ctx.feat, ctx.wt, ctx.shape = mask_rows, feat, wt, feat_flat.shape
        return out

    @staticmethod
    def backward(ctx, g):
        g = _f32c(g)
        dF, dw, db = fusion_backward(ctx.mask_rows, ctx.feat, ctx.wt, g, D)
        return None, dF.reshape(ctx.shape), dw, db


class MaskedFeatureMap:
    """What the caller may pass as ``path_map`` instead of the dense (T, map^2) product of
    train.py:500-501: the selected sparse mask rows plus the flattened CNN feature map."""

    def __init__(self, mask_rows, feat_map):
        self.mask_rows = mask_rows
        self.feat_map = feat_map

    def to_dense(self):
        csr = self.mask_rows.csr
        T, J = self.mask_rows.T, csr.width
        dense = torch.zeros(T, J, dtype=torch.float32, device=self.feat_map.device)
        rl = self.mask_rows.rows.long()
        deg = (csr.indptr[rl + 1] - csr.indptr[rl]).long()
        t_of = torch.repeat_interleave(torch.arange(T, device=deg.device), deg)
        first = torch.cumsum(deg, 0) - deg
        slot = torch.repeat_interleave(csr.indptr[rl].long(), deg) + \
            (torch.arange(int(deg.sum()), device=deg.device) - first[t_of])
        dense[t_of, csr.cols[slot].long()] = 1.0
        return dense * self.feat_map.reshape(1, -1)


# --------------------------------------------------------------------------------------------
# nn.Linear on the fp32 GEMM core (model.py:15; F.linear semantics, optional fused ReLU)
# --------------------------------------------------------------------------------------------
class LinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, relu):
        x2 = _rowmajor(x.detach().reshape(-1, x.shape[-1]))
        tm_lib.require_cuda(x2, "Linear input")
        M, K = x2.shape
        N = w.shape[0]
        y = torch.empty(M, N, dtype=torch.float32, device=x2.device)
        gemm_nn(M, N, K, x2, x2.stride(0), _f32c(w.detach()), K, y, N,
                bias=None if b is None else _f32c(b.detach()), flags=RELU if relu else 0, b_is_nk=True)
        ctx.save = (x2, w.detach(), y if relu else None)
        ctx.has_bias, ctx.xshape = b is not None, x.shape
        ctx.need_dx = x.requires_grad
        return y.reshape(x.shape[:-1] + (N,))

    @staticmethod
    def backward(ctx, g):
        x2, w, y = ctx.save
        N, K = w.shape
        M = x2.shape[0]
        g2 = _f32c(g.reshape(M, N))
        if y is not None:                                  # ReLU backward on the incoming gradient
            gm = torch.empty_like(g2)
            call("tm_leaky_relu_backward", g2.numel(), y, g2, 0.0, gm, stream())
            g2 = gm
        dev = x2.device
        dw = torch.empty(N, K, dtype=torch.float32, device=dev)
        db = torch.empty(N, dtype=torch.float32, device=dev) if ctx.has_bias else None
        if M > 0:
            gemm_tn(N, K, M, g2, N, x2, x2.stride(0), dw, K, colsum_a=db)
            aux_join()
        else:
            dw.zero_()
            if db is not None:
                db.zero_()
        dx = None
        if ctx.need_dx:
            dx = torch.empty(M, K, dtype=torch.float32, device=dev)
            gemm_nn(M, K, N, g2, N, _f32c(w), K, dx, K)
            dx = dx.reshape(ctx.xshape)
        return dx, dw, db, None


def linear(x, w, b=None, relu=False):
    return LinearFn.apply(x, w, b, relu)
