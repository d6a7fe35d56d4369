"""Image branch on libtm_b200: U-Net (src/Unet.py:85-119) and LayoutNet (src/model.py:216-247).

Activations are NHWC fp32 on the device; skip connections and transposed-conv outputs are written
straight into the two halves of a shared concat buffer (``torch.cat`` of Unet.py:67 costs
nothing).  BatchNorm always uses batch statistics -- the reference never calls ``.eval()``
(train.py:436-437) -- and updates the running statistics exactly like ``nn.BatchNorm2d``
(momentum 0.1, unbiased variance).  Every contraction is a ``tm_conv2d_nhwc`` /
``tm_convt2x2_nhwc`` implicit GEMM; nothing here calls cuDNN or ATen convolution.
"""
import os

import torch

import tm_lib
from tm_lib import call, stream

RELU = 2


def _empty(*shape, dev):
    return torch.empty(*shape, dtype=torch.float32, device=dev)


class _Ws:
    """One growing scratch buffer shared by the split-reduction kernels of a pass."""

    def __init__(self, dev):
        self.dev, self.buf = dev, None

    def get(self, nbytes):
        if self.buf is None or self.buf.numel() < nbytes:
            self.buf = tm_lib.workspace(nbytes, self.dev)
        return self.buf


# arithmetic of the convolutions: "tc3" (split-bf16 x3 on tcgen05, fp32-class), "bf16" (tcgen05,
# plain bf16 operands) or "fp32" (CUDA-core implicit GEMM).  Per network: net.math overrides.
MATH = None            # None -> follow tm_ops.MATH
_CUR = None            # math mode of the network currently being run (net.math)


def _prec(math):
    import tm_ops
    return tm_ops._precision(math or _CUR or MATH or tm_ops.MATH)


def _enter(net):
    global _CUR
    _CUR = getattr(net, "math", None)


USE_TMA = os.environ.get("TM_CONV_TMA", "1") != "0"   # bf16 / tf32x3 mode: TMA-fed 3x3 and transposed convolutions


def _cpad(c):
    return max(16, (c + 15) // 16 * 16)


def _tma_fmt():
    """Operand format of the TMA-fed kernels for the current arithmetic: "bf16" (bf16 mode), "tf32" (tf32x3: fp32
    operands read in place, 3xTF32 products) or None (tc6, tc3, tf32, fp32 keep the cp.async / CUDA-core kernels)."""
    return {0: "bf16", 3: "tf32"}.get(_prec(None)) if USE_TMA else None


def _tma_ok(B, H, W, cin, cout):
    """-> the TMA operand format when it serves the current arithmetic and the kernels take the shape (H, W powers
    of two; channels multiples of 16), else None."""
    fmt = _tma_fmt()
    if fmt is None or cout > 128 or _cpad(cin) > 128:
        return None
    fn = f"tm_conv3x3_{fmt}_supported"
    if (tm_lib.ws_bytes(fn, B, H, W, _cpad(cin), cout) == 1
            and (cin % 16 != 0 or tm_lib.ws_bytes(fn, B, H, W, cout, cin) == 1)):
        return fmt
    return None


def _to_bf16(x, ldx, npix, C):
    """fp32 rows (stride ldx) -> compact bf16 [npix][pad16(C)]: the TMA operand of the next convolution."""
    out = torch.empty(npix, _cpad(C), dtype=torch.bfloat16, device=x.device)
    call("tm_to_bf16_rows", npix, C, x, ldx, out, _cpad(C), stream())
    return out


def _pack_tma(w, W, need_dgrad, fmt="bf16"):
    """-> ((forward operand, P), (data-gradient operand, P) or None) for images W wide; bf16 or fp32 ("tf32")."""
    cout, cin = w.shape[0], w.shape[1]
    dev = w.device
    wc = w.detach().float().contiguous()
    dtype, pack = (torch.bfloat16, "tm_conv3x3_pack_bf16") if fmt == "bf16" else (torch.float32, "tm_conv3x3_pack_f32")

    def one(nc, kc, dgrad):
        kp = _cpad(kc)
        P = tm_lib.ws_bytes(f"tm_conv3x3_{fmt}_pack", W, kp, nc)
        q = torch.empty(9, P * nc, P * kp, dtype=dtype, device=dev)
        call(pack, cout, cin, wc, q, P, kp, dgrad, stream())
        return q, P
    return one(cout, cin, 0), (one(cin, cout, 1) if need_dgrad else None)


FUSE_BN_STATS = os.environ.get("TM_FUSE_BN_STATS", "1") != "0"   # BN statistics in the convolution's epilogue


def _conv_tma(xb, B, H, W, cinp, cout, wq, y, ldy, want_stats=False):
    """-> (stats buffer, number of partials) when the epilogue also took the batch-norm statistics, else None."""
    q, P = wq
    stats = None
    if want_stats and FUSE_BN_STATS and P * cout <= 128:
        nb = tm_lib.ws_bytes("tm_conv3x3_bf16_stats_bytes", cout, P)
        stats = (torch.empty(nb, dtype=torch.uint8, device=y.device), nb // (16 * cout))
    call("tm_conv3x3_bf16", B, H, W, cinp, cout, P, xb, q, None, y, ldy, 0, stats[0] if stats else None,
         tm_lib.err_flag(y.device), stream())
    return stats


def _conv_tf(ws, x, ldx, B, H, W, cinp, cout, wq, y, ldy, want_stats=False):
    """tf32x3 on the TMA kernels, x read in place.  Deep layers split K (workspace); only unsplit launches take the
    batch-norm statistics in their epilogue.  -> (stats buffer, number of partials) or None."""
    q, P = wq
    nb = tm_lib.ws_bytes("tm_conv3x3_tf32_ws", B, H, W, cinp, cout, P)
    stats = None
    if want_stats and FUSE_BN_STATS and nb == 0 and P * cout <= 128:
        ns = tm_lib.ws_bytes("tm_conv3x3_bf16_stats_bytes", cout, P)
        stats = (torch.empty(ns, dtype=torch.uint8, device=y.device), ns // (16 * cout))
    call("tm_conv3x3_tf32", B, H, W, cinp, cout, P, x, ldx, q, None, y, ldy, 0, stats[0] if stats else None,
         ws.get(nb) if nb else None, nb, tm_lib.err_flag(y.device), stream())
    return stats


def _wgrad_tf(ws, x, ldx, dy, lddy, B, H, W, cinp, cin, cout):
    if min(cin, cout) >= 64:
        # measured slower on the TMA kernel (profiles/bench_unet_tf32_layers.py: 128 -> 128 at 32x32 70 us against
        # 31 us): few pixels, 32-pixel stages and one-tap stages; these stay on the cp.async tf_gemm route
        return _conv_wgrad(ws, x, ldx, dy, lddy, B, H, W, cin, cout, 3, False)[0]
    dev = dy.device
    dw = _empty(cout, cin, 3, 3, dev=dev)
    nb = tm_lib.ws_bytes("tm_conv3x3_tf32_wgrad_ws", B, H, W, cinp, cout)
    call("tm_conv3x3_tf32_wgrad", B, H, W, cinp, cin, cout, x, ldx, dy, lddy, dw, ws.get(nb), nb, tm_lib.err_flag(dev),
         stream())
    return dw


def _wgrad_tma(ws, xb, dyb, B, H, W, cin, cout):
    dev = dyb.device
    dw = _empty(cout, cin, 3, 3, dev=dev)
    nb = tm_lib.ws_bytes("tm_conv3x3_bf16_wgrad_ws", B, H, W, _cpad(cin), cout)
    call("tm_conv3x3_bf16_wgrad", B, H, W, _cpad(cin), cin, cout, xb, dyb, dw, ws.get(nb), nb, tm_lib.err_flag(dev), stream())
    return dw


def _conv(x, ldx, B, H, W, cin, cout, k, wf, bias, y, ldy, flags=0, math=None):
    prec = _prec(math)
    if prec is None:
        call("tm_conv2d_nhwc", B, H, W, cin, cout, k, x, ldx, wf, bias, y, ldy, flags, stream())
    else:
        nb = tm_lib.ws_bytes("tm_tc_conv2d_splitk_ws", B, H, W, cin, cout, k, prec)   # 0: the layer fills the GPU unsplit
        call("tm_tc_conv2d_nhwc_splitk", B, H, W, cin, cout, k, x, ldx, wf, bias, y, ldy, flags, prec,
             tm_lib.workspace(nb, y.device) if nb else None, nb, tm_lib.err_flag(y.device), stream())


def _conv_wgrad(ws, x, ldx, dy, lddy, B, H, W, cin, cout, k, want_bias, math=None):
    dev = dy.device
    dwf = _empty(k * k * cin, cout, dev=dev)
    dbias = _empty(cout, dev=dev) if want_bias else None
    prec = _prec(math)
    if prec is None:
        nb = tm_lib.ws_bytes("tm_conv2d_wgrad_ws", B, H, W, cin, cout, k)
        call("tm_conv2d_wgrad_nhwc", B, H, W, cin, cout, k, x, ldx, dy, lddy, dwf, dbias, ws.get(nb), nb, stream())
    else:
        nb = tm_lib.ws_bytes("tm_tc_conv2d_wgrad_ws", B, H, W, cin, cout, k)
        call("tm_tc_conv2d_wgrad_nhwc", B, H, W, cin, cout, k, x, ldx, dy, lddy, dwf, prec, ws.get(nb), nb,
             tm_lib.err_flag(dev), stream())
        if want_bias:
            nbc = tm_lib.ws_bytes("tm_colsum_ws", B * H * W, cout)
            call("tm_colsum", B * H * W, cout, dy, lddy, None, dbias, 0, tm_lib.workspace(nbc, dev), nbc, stream())
    dw = _empty(cout, cin, k, k, dev=dev)
    call("tm_conv_unpack_wgrad", cout, cin, k, dwf, dw, stream())
    return dw, dbias


def _pack(w, need_bwd=True):
    cout, cin, k, _ = w.shape
    dev = w.device
    w = w.detach().float().contiguous()
    wf = _empty(k * k * cin, cout, dev=dev)
    wb = _empty(k * k * cout, cin, dev=dev) if need_bwd else None
    call("tm_conv_pack_weight", cout, cin, k, w, wf, wb, stream())
    return wf, wb


EVAL = False          # set by unet_forward: nn.Module.eval() -> BatchNorm uses its running statistics
SEG = 1               # set by unet_forward / unet_backward: > 1 -> BatchNorm statistics per image of the batch


def _bn_relu_fwd(ws, x, ldx, npix, C, bn, y, ldy, update_stats, yb=None, stats=None):
    dev = x.device
    mean, invstd = _empty(C, dev=dev), _empty(C, dev=dev)
    if EVAL:
        if bn.running_mean is None:
            raise NotImplementedError("eval-mode BatchNorm without running statistics (track_running_stats=False)")
        call("tm_bn_relu_eval", npix, C, x, ldx, bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var,
             float(bn.eps), y, ldy, mean, invstd, yb, stream())
        return mean, invstd
    rm = bn.running_mean if update_stats else None
    rv = bn.running_var if update_stats else None
    if SEG > 1:
        # each image its own statistics; the running statistics take SEG updates, image 0 first
        mean, invstd = _empty(SEG * C, dev=dev), _empty(SEG * C, dev=dev)
        nb = tm_lib.ws_bytes("tm_bn_seg_ws", SEG, npix // SEG, C)
        call("tm_bn_relu_forward_seg", SEG, npix // SEG, C, x, ldx, bn.weight.detach(), bn.bias.detach(), rm, rv,
             float(bn.momentum), float(bn.eps), y, ldy, mean, invstd, yb, ws.get(nb), nb, stream())
    else:
        nb = tm_lib.ws_bytes("tm_bn_ws", npix, C)
        call("tm_bn_relu_forward", npix, C, x, ldx, bn.weight.detach(), bn.bias.detach(), rm, rv,
             float(bn.momentum), float(bn.eps), y, ldy, mean, invstd, yb, stats[0] if stats else None,
             stats[1] if stats else 0, ws.get(nb), nb, stream())
    if update_stats and bn.num_batches_tracked is not None:
        bn.num_batches_tracked += SEG
    return mean, invstd


def _bn_relu_bwd(ws, x, ldx, dy, lddy, npix, C, gamma, beta, mean, invstd, dx, lddx, dxb=None):
    """dx (fp32, may be None) and / or dxb (compact bf16) receive the gradient w.r.t. the BN input.  The ReLU mask
    is rebuilt from x and the saved statistics (bit-identical to the forward), so the activation is not read."""
    dev = x.device
    dg, db = _empty(C, dev=dev), _empty(C, dev=dev)
    if SEG > 1:
        nb = tm_lib.ws_bytes("tm_bn_seg_ws", SEG, npix // SEG, C)
        call("tm_bn_relu_backward_seg", SEG, npix // SEG, C, x, ldx, None, 0, dy, lddy, gamma, beta, mean, invstd, dx,
             lddx, dg, db, dxb, ws.get(nb), nb, stream())
        return dg, db
    nb = tm_lib.ws_bytes("tm_bn_ws", npix, C)
    call("tm_bn_relu_backward", npix, C, x, ldx, None, 0, dy, lddy, gamma, beta, mean, invstd, dx, lddx, dg, db, dxb,
         ws.get(nb), nb, stream())
    return dg, db


# --------------------------------------------------------------------------------------------
# U-Net
# --------------------------------------------------------------------------------------------
def _double_conv_fwd(ws, st, name, mods, x, ldx, B, H, W, cin, cout, out, ldo, update_stats, need_bwd):
    """conv3x3 -> BN -> ReLU -> conv3x3 -> BN -> ReLU (Unet.py:15-22); final activation -> out."""
    conv1, bn1, conv2, bn2 = mods
    dev = x.device
    npix = B * H * W
    cmid = conv1.weight.shape[0]
    r1, r2 = _empty(npix, cmid, dev=dev), _empty(npix, cout, dev=dev)
    route = _tma_ok(B, H, W, cin, cmid) if _tma_ok(B, H, W, cmid, cout) else None
    if route == "tf32":
        # tf32x3 mode: the TMA-fed kernels read the fp32 activations in place (x: compact rows, or 16 zero-padded
        # channels for the 3-channel input)
        wq1, wd1 = _pack_tma(conv1.weight, W, need_bwd and cin % 16 == 0, "tf32")
        wq2, wd2 = _pack_tma(conv2.weight, W, need_bwd, "tf32")
        a1 = _empty(npix, cmid, dev=dev)
        s1 = _conv_tf(ws, x, ldx, B, H, W, _cpad(cin), cmid, wq1, r1, cmid, want_stats=SEG == 1)
        m1, i1 = _bn_relu_fwd(ws, r1, cmid, npix, cmid, bn1, a1, cmid, update_stats, stats=s1)
        s2 = _conv_tf(ws, a1, cmid, B, H, W, cmid, cout, wq2, r2, cout, want_stats=SEG == 1)
        m2, i2 = _bn_relu_fwd(ws, r2, cout, npix, cout, bn2, out, ldo, update_stats, stats=s2)
        st[name] = dict(tf=True, x=x, ldx=ldx, a1=a1, wd1=wd1, wd2=wd2, B=B, H=H, W=W, cin=cin, cmid=cmid, cout=cout,
                        r1=r1, r2=r2, out=out, ldo=ldo, m1=m1, i1=i1, m2=m2, i2=i2, g1=bn1.weight.detach(),
                        g2=bn2.weight.detach(), be1=bn1.bias.detach(), be2=bn2.bias.detach())
        return
    if route == "bf16":
        # bf16 mode: TMA-fed tcgen05 convolutions on compact bf16 copies of the activations (kept for wgrad)
        xb = _to_bf16(x, ldx, npix, cin)
        wq1, wd1 = _pack_tma(conv1.weight, W, need_bwd and cin % 16 == 0)
        wq2, wd2 = _pack_tma(conv2.weight, W, need_bwd)
        # the convolution epilogue's statistics cover the whole batch: per-image statistics (SEG > 1) take their own pass
        s1 = _conv_tma(xb, B, H, W, _cpad(cin), cmid, wq1, r1, cmid, want_stats=SEG == 1)
        a1b = torch.empty(npix, cmid, dtype=torch.bfloat16, device=dev)
        # the mid activation exists only as the bf16 operand of conv2 (the backward rebuilds its ReLU mask from r1)
        m1, i1 = _bn_relu_fwd(ws, r1, cmid, npix, cmid, bn1, None, 0, update_stats, yb=a1b, stats=s1)
        s2 = _conv_tma(a1b, B, H, W, cmid, cout, wq2, r2, cout, want_stats=SEG == 1)
        m2, i2 = _bn_relu_fwd(ws, r2, cout, npix, cout, bn2, out, ldo, update_stats, stats=s2)
        st[name] = dict(tma=True, xb=xb if need_bwd else None, a1b=a1b if need_bwd else None, wd1=wd1, wd2=wd2,
                        x=x, ldx=ldx, B=B, H=H, W=W, cin=cin, cmid=cmid, cout=cout, r1=r1, r2=r2, out=out,
                        ldo=ldo, m1=m1, i1=i1, m2=m2, i2=i2, g1=bn1.weight.detach(), g2=bn2.weight.detach(),
                        be1=bn1.bias.detach(), be2=bn2.bias.detach())
        return
    a1 = _empty(npix, cmid, dev=dev)
    wf1, wb1 = _pack(conv1.weight, need_bwd)
    wf2, wb2 = _pack(conv2.weight, need_bwd)
    _conv(x, ldx, B, H, W, cin, cmid, 3, wf1, None, r1, cmid)
    m1, i1 = _bn_relu_fwd(ws, r1, cmid, npix, cmid, bn1, a1, cmid, update_stats)
    _conv(a1, cmid, B, H, W, cmid, cout, 3, wf2, None, r2, cout)
    m2, i2 = _bn_relu_fwd(ws, r2, cout, npix, cout, bn2, out, ldo, update_stats)
    st[name] = dict(x=x, ldx=ldx, B=B, H=H, W=W, cin=cin, cmid=cmid, cout=cout, r1=r1, a1=a1, r2=r2, out=out,
                    ldo=ldo, m1=m1, i1=i1, m2=m2, i2=i2, wb1=wb1, wb2=wb2, g1=bn1.weight.detach(),
                    g2=bn2.weight.detach(), be1=bn1.bias.detach(), be2=bn2.bias.detach())


def _dgrad_image(dr, lddr, bf16, s, w, dimg):
    """Gradient w.r.t. the network's input image from the gradient of its first convolution's output: the narrow
    direct kernel (2-4 image channels), written straight to NCHW."""
    call("tm_conv_dgrad_narrow", s["B"], s["H"], s["W"], s["cin"], w.shape[0], w.shape[2], dr, lddr, int(bf16), w, dimg,
         stream())


def _double_conv_bwd(ws, s, dout, lddo, grads, prefix, dx, lddx, dimg=None, w1=None, wg=True):
    """dout: gradient w.r.t. the block output (strided).  Writes dx (if not None); dimg (NCHW, optional): the gradient
    w.r.t. the block input when it is the input image, through the first convolution's weight w1.  ``wg=False``: no
    weight gradient is computed and nothing is added to ``grads`` (the batch-norm backward still reduces: dx needs it)."""
    B, H, W, cin, cmid, cout = s["B"], s["H"], s["W"], s["cin"], s["cmid"], s["cout"]
    npix = B * H * W
    dev = dout.device
    da1 = _empty(npix, cmid, dev=dev)
    if s.get("tf"):
        dr2 = _empty(npix, cout, dev=dev)
        dg2, db2 = _bn_relu_bwd(ws, s["r2"], cout, dout, lddo, npix, cout, s["g2"], s["be2"], s["m2"], s["i2"],
                                dr2, cout)
        dw2 = _wgrad_tf(ws, s["a1"], cmid, dr2, cout, B, H, W, cmid, cmid, cout) if wg else None
        _conv_tf(ws, dr2, cout, B, H, W, cout, cmid, s["wd2"], da1, cmid)
        dr1 = _empty(npix, cmid, dev=dev)
        dg1, db1 = _bn_relu_bwd(ws, s["r1"], cmid, da1, cmid, npix, cmid, s["g1"], s["be1"], s["m1"], s["i1"],
                                dr1, cmid)
        dw1 = _wgrad_tf(ws, s["x"], s["ldx"], dr1, cmid, B, H, W, _cpad(cin), cin, cmid) if wg else None
        if dx is not None:
            _conv_tf(ws, dr1, cmid, B, H, W, cmid, cin, s["wd1"], dx, lddx)
        if dimg is not None:
            _dgrad_image(dr1, cmid, False, s, w1, dimg)
    elif s.get("tma"):
        # the batch-norm backward emits its result directly as the bf16 operand shared by the weight and the
        # data gradient; the fp32 copy is never needed
        dr2b = torch.empty(npix, cout, dtype=torch.bfloat16, device=dev)
        dg2, db2 = _bn_relu_bwd(ws, s["r2"], cout, dout, lddo, npix, cout, s["g2"], s["be2"], s["m2"], s["i2"],
                                None, 0, dxb=dr2b)
        dw2 = _wgrad_tma(ws, s["a1b"], dr2b, B, H, W, cmid, cout) if wg else None
        _conv_tma(dr2b, B, H, W, cout, cmid, s["wd2"], da1, cmid)
        dr1b = torch.empty(npix, cmid, dtype=torch.bfloat16, device=dev)
        dg1, db1 = _bn_relu_bwd(ws, s["r1"], cmid, da1, cmid, npix, cmid, s["g1"], s["be1"], s["m1"], s["i1"],
                                None, 0, dxb=dr1b)
        dw1 = _wgrad_tma(ws, s["xb"], dr1b, B, H, W, cin, cmid) if wg else None
        if dx is not None:
            _conv_tma(dr1b, B, H, W, cmid, cin, s["wd1"], dx, lddx)
        if dimg is not None:
            _dgrad_image(dr1b, cmid, True, s, w1, dimg)
    else:
        dr2 = _empty(npix, cout, dev=dev)
        dg2, db2 = _bn_relu_bwd(ws, s["r2"], cout, dout, lddo, npix, cout, s["g2"], s["be2"], s["m2"], s["i2"],
                                dr2, cout)
        dr1 = _empty(npix, cmid, dev=dev)
        dw2 = _conv_wgrad(ws, s["a1"], cmid, dr2, cout, B, H, W, cmid, cout, 3, False)[0] if wg else None
        _conv(dr2, cout, B, H, W, cout, cmid, 3, s["wb2"], None, da1, cmid)
        dg1, db1 = _bn_relu_bwd(ws, s["r1"], cmid, da1, cmid, npix, cmid, s["g1"], s["be1"], s["m1"], s["i1"],
                                dr1, cmid)
        dw1 = _conv_wgrad(ws, s["x"], s["ldx"], dr1, cmid, B, H, W, cin, cmid, 3, False)[0] if wg else None
        if dx is not None:
            _conv(dr1, cmid, B, H, W, cmid, cin, 3, s["wb1"], None, dx, lddx)
        if dimg is not None:
            _dgrad_image(dr1, cmid, False, s, w1, dimg)
    if not wg:
        return
    grads[prefix + ".0.weight"] = dw1
    grads[prefix + ".1.weight"], grads[prefix + ".1.bias"] = dg1, db1
    grads[prefix + ".3.weight"] = dw2
    grads[prefix + ".4.weight"], grads[prefix + ".4.bias"] = dg2, db2


def _dc_mods(dc):
    seq = dc.double_conv
    return seq[0], seq[1], seq[3], seq[4]


def unet_forward(net, x, need_bwd=True, update_stats=True, per_image=False):
    """``net``: the UNet module (parameter container).  x: (B,3,H,W) or (3,H,W) on a CUDA device.
    Returns (out (B,1,H/2,W/2), state).  ``per_image``: train-mode BatchNorm normalises every image with its own
    statistics, as B batch-of-one calls would (the fused step over several designs); default: batch statistics,
    like ``nn.BatchNorm2d``."""
    _enter(net)
    global EVAL, SEG
    EVAL = not net.training
    if EVAL and need_bwd:
        raise NotImplementedError("UNet in eval mode is inference only here (BatchNorm backward with frozen statistics is not "
                                  "built): call it under torch.no_grad(), or keep the module in train mode like the reference")
    squeeze = x.dim() == 3
    if squeeze:                                        # train.py:465 passes (C,H,W)
        x = x.unsqueeze(0)
    x = x.detach().float().contiguous()
    tm_lib.require_cuda(x, "UNet input")
    B, C, H, W = x.shape
    if C != 3 or H % 8 or W % 8:
        raise RuntimeError("UNet expects (B,3,H,W) with H and W multiples of 8")
    SEG = B if per_image and not EVAL else 1
    dev = x.device
    mode = 0 if net.pooling == "max" else 1
    ws = _Ws(dev)
    st = {"ws": ws, "mode": mode, "B": B, "H": H, "W": W, "seg": SEG, "squeeze": squeeze,
          "w_in": net.inc.double_conv[0].weight.detach().float().contiguous()}
    # tf32x3 mode reads the input in place: 16 channels, zero padded (a 12-byte pixel stride is no TMA stride)
    c0 = 16 if _tma_fmt() == "tf32" else 3
    x0 = (torch.zeros if c0 > 3 else torch.empty)(B * H * W, c0, dtype=torch.float32, device=dev)
    call("tm_nchw_to_nhwc", B, 3, H, W, x, x0, c0, stream())
    chans = [16, 32, 64, 128]
    Hs = [H, H // 2, H // 4, H // 8]
    Ws_ = [W, W // 2, W // 4, W // 8]
    cat = [_empty(B * Hs[i] * Ws_[i], 2 * chans[i], dev=dev) for i in range(3)]     # [skip | up]
    x4 = _empty(B * Hs[3] * Ws_[3], 128, dev=dev)
    enc = [net.inc, net.down1.maxpool_conv[1], net.down2.maxpool_conv[1], net.down3.maxpool_conv[1]]
    cur, ld, cin = x0, c0, 3
    st["pool"] = []
    for i in range(4):
        if i > 0:                                      # Down = pool -> DoubleConv (Unet.py:33-36)
            pooled = _empty(B * Hs[i] * Ws_[i], chans[i - 1], dev=dev)
            idx = torch.empty(B * Hs[i] * Ws_[i] * chans[i - 1], dtype=torch.uint8, device=dev) if mode == 0 else None
            call("tm_pool2x2_forward", B, Hs[i - 1], Ws_[i - 1], chans[i - 1], mode, cur, ld, pooled, chans[i - 1],
                 idx, 0, stream())
            st["pool"].append(dict(idx=idx, src_ld=ld, C=chans[i - 1], H=Hs[i - 1], W=Ws_[i - 1]))
            cur, ld, cin = pooled, chans[i - 1], chans[i - 1]
        out, ldo = (cat[i], 2 * chans[i]) if i < 3 else (x4, 128)
        _double_conv_fwd(ws, st, f"enc{i}", _dc_mods(enc[i]), cur, ld, B, Hs[i], Ws_[i], cin, chans[i], out, ldo,
                         update_stats, need_bwd)
        cur, ld = out, ldo
    # decoder: Up = ConvTranspose2d(k2,s2) -> cat([skip, up]) -> DoubleConv (Unet.py:53-68)
    ups = [net.up1, net.up2, net.up3]
    y, ldy, cy = x4, 128, 128
    for j, up in enumerate(ups):
        i = 2 - j                                      # resolution index of the skip
        cout_t = cy // 2
        half = cat[i][:, chans[i]:]                    # second half of the concat buffer
        wup = up.up.weight.detach().float().contiguous()
        fmt = _tma_fmt()
        if fmt and tm_lib.ws_bytes(f"tm_convt2x2_{fmt}_supported", B, Hs[i + 1], Ws_[i + 1], cy, cout_t) != 1:
            fmt = None
        if fmt == "tf32":
            # tf32x3 mode: the same one-tap TMA convolution on the fp32 activation, read in place
            wfq = _empty(4 * cout_t, cy, dev=dev)
            wdq = _empty(4, cy, cout_t, dev=dev) if need_bwd else None
            call("tm_convt2x2_pack_f32", cy, cout_t, wup, wfq, wdq, stream())
            nb = tm_lib.ws_bytes("tm_convt2x2_tf32_ws", B, Hs[i + 1], Ws_[i + 1], cy, cout_t)
            call("tm_convt2x2_tf32", B, Hs[i + 1], Ws_[i + 1], cy, cout_t, y, ldy, wfq, up.up.bias.detach(), half,
                 2 * chans[i], ws.get(nb) if nb else None, nb, tm_lib.err_flag(dev), stream())
            st[f"up{j}"] = dict(x=y, ldx=ldy, cin=cy, cout=cout_t, wdf=wdq, i=i)
        elif fmt == "bf16":
            # bf16 mode: one-tap TMA convolution whose epilogue scatters the 2x2 output windows
            yb = _to_bf16(y, ldy, B * Hs[i + 1] * Ws_[i + 1], cy)
            wfq = torch.empty(4 * cout_t, cy, dtype=torch.bfloat16, device=dev)
            wdq = torch.empty(4, cy, cout_t, dtype=torch.bfloat16, device=dev) if need_bwd else None
            call("tm_convt2x2_pack_bf16", cy, cout_t, wup, wfq, wdq, stream())
            call("tm_convt2x2_bf16", B, Hs[i + 1], Ws_[i + 1], cy, cout_t, yb, wfq, up.up.bias.detach(), half,
                 2 * chans[i], tm_lib.err_flag(dev), stream())
            st[f"up{j}"] = dict(x=y, ldx=ldy, cin=cy, cout=cout_t, wdq=wdq, xb=yb if need_bwd else None, i=i)
        else:
            wt, wtT = _empty(cy, 4 * cout_t, dev=dev), _empty(4 * cout_t, cy, dev=dev)
            call("tm_convt_pack_weight", cy, cout_t, wup, wt, wtT, stream())
            call("tm_convt2x2_nhwc", B, Hs[i + 1], Ws_[i + 1], cy, cout_t, y, ldy, wt, up.up.bias.detach(), half,
                 2 * chans[i], Hs[i], Ws_[i], 0, 0, stream())
            st[f"up{j}"] = dict(x=y, ldx=ldy, cin=cy, cout=cout_t, wtT=wtT, i=i)
        out = _empty(B * Hs[i] * Ws_[i], chans[i], dev=dev)
        _double_conv_fwd(ws, st, f"dec{j}", _dc_mods(up.conv), cat[i], 2 * chans[i], B, Hs[i], Ws_[i], 2 * chans[i],
                         chans[i], out, chans[i], update_stats, need_bwd)
        y, ldy, cy = out, chans[i], chans[i]
    # OutConv: 1x1 conv (bias) -> pool -> ReLU (Unet.py:74-78)
    oc = net.outc.conv[0]
    wo = oc.weight.detach().float().reshape(-1).contiguous()         # (1,16,1,1) -> [16]
    o_raw = _empty(B * H * W, 1, dev=dev)
    call("tm_conv1x1_c1_forward", B * H * W, 16, y, ldy, wo, oc.bias.detach(), o_raw, 1, stream())
    out = _empty(B, 1, H // 2, W // 2, dev=dev)
    oidx = torch.empty(B * (H // 2) * (W // 2), dtype=torch.uint8, device=dev) if mode == 0 else None
    call("tm_pool2x2_forward", B, H, W, 1, mode, o_raw, 1, out, 1, oidx, RELU, stream())
    st.update(y3=y, ld3=ldy, wo=wo, out=out, oidx=oidx, cat=cat, chans=chans, Hs=Hs, Ws=Ws_)
    return out, st


def unet_backward(net, st, gout, need_dx=False, need_wgrad=True):
    """gout: (B,1,H/2,W/2).  Returns {state_dict-style name: gradient} for every parameter; with ``need_dx``
    (grads, dx), dx the gradient w.r.t. the input image in its layout: (B,3,H,W), or (3,H,W) for a 3-D input.
    ``need_wgrad=False`` (a frozen network): no weight-gradient kernel runs on any route and ``grads`` is empty; dx is
    the same bits."""
    _enter(net)
    global SEG
    SEG = st["seg"]
    B, H, W, mode = st["B"], st["H"], st["W"], st["mode"]
    ws, chans, Hs, Ws_, cat = st["ws"], st["chans"], st["Hs"], st["Ws"], st["cat"]
    dev = gout.device
    gout = gout.detach().float().contiguous()
    grads = {}
    d_oraw = _empty(B * H * W, 1, dev=dev)
    call("tm_pool2x2_backward", B, H, W, 1, mode, gout, 1, st["out"], 1, st["oidx"], d_oraw, 1, RELU, None, 0, stream())
    if need_wgrad:
        dw, db = _empty(1, 16, 1, 1, dev=dev), _empty(1, dev=dev)
        nb = tm_lib.ws_bytes("tm_conv1x1_c1_wgrad_ws", 16)
        call("tm_conv1x1_c1_wgrad", B * H * W, 16, st["y3"], st["ld3"], d_oraw, 1, dw, db, ws.get(nb), nb, stream())
        grads["outc.conv.0.weight"], grads["outc.conv.0.bias"] = dw, db
    dy = _empty(B * H * W, 16, dev=dev)
    call("tm_conv1x1_c1_dgrad", B * H * W, 16, d_oraw, 1, st["wo"], dy, 16, stream())
    lddy = 16
    dskip = [None, None, None]
    names = ["up1", "up2", "up3"]
    for j in (2, 1, 0):
        i = 2 - j
        dcat = _empty(B * Hs[i] * Ws_[i], 2 * chans[i], dev=dev)
        _double_conv_bwd(ws, st[f"dec{j}"], dy, lddy, grads, f"{names[j]}.conv.double_conv", dcat, 2 * chans[i],
                         wg=need_wgrad)
        dskip[i] = dcat                                  # first half = gradient of the skip tensor
        u = st[f"up{j}"]
        half = dcat[:, chans[i]:]
        dy = _empty(B * Hs[i + 1] * Ws_[i + 1], u["cin"], dev=dev)
        if u.get("wdq") is not None:
            # bf16 mode: weight and data gradient on the TMA path, both from one bf16 copy of the gradient half
            npo = B * Hs[i] * Ws_[i]
            halfb = _to_bf16(half, 2 * chans[i], npo, u["cout"])
            if need_wgrad:
                dwu, dbt = _empty(u["cin"], u["cout"], 2, 2, dev=dev), _empty(u["cout"], dev=dev)
                nb = tm_lib.ws_bytes("tm_convt2x2_bf16_wgrad_ws", B, Hs[i + 1], Ws_[i + 1], u["cin"], u["cout"])
                call("tm_convt2x2_bf16_wgrad", B, Hs[i + 1], Ws_[i + 1], u["cin"], u["cout"], u["xb"], halfb, dwu, ws.get(nb),
                     nb, tm_lib.err_flag(dev), stream())
                nbc = tm_lib.ws_bytes("tm_colsum_ws", npo, u["cout"])
                call("tm_colsum", npo, u["cout"], half, 2 * chans[i], None, dbt, 0, tm_lib.workspace(nbc, dev), nbc, stream())
            call("tm_convt2x2_bf16_dgrad", B, Hs[i + 1], Ws_[i + 1], u["cin"], u["cout"], halfb, u["wdq"], dy, u["cin"],
                 tm_lib.err_flag(dev), stream())
        else:
            tf = u.get("wdf") is not None
            shape = (B, Hs[i + 1], Ws_[i + 1], u["cin"], u["cout"])
            if need_wgrad and tf and tm_lib.ws_bytes("tm_convt2x2_tf32_wgrad_supported", *shape) == 1:
                # tf32x3 mode: weight gradient on the TMA path (its N side needs 32-channel boxes: Cout >= 32)
                nb = tm_lib.ws_bytes("tm_convt2x2_tf32_ws", *shape)
                dwu, dbt = _empty(u["cin"], u["cout"], 2, 2, dev=dev), _empty(u["cout"], dev=dev)
                call("tm_convt2x2_tf32_wgrad", *shape, u["x"], u["ldx"], half, 2 * chans[i], dwu, ws.get(nb), nb,
                     tm_lib.err_flag(dev), stream())
                npo = B * Hs[i] * Ws_[i]
                nbc = tm_lib.ws_bytes("tm_colsum_ws", npo, u["cout"])
                call("tm_colsum", npo, u["cout"], half, 2 * chans[i], None, dbt, 0, tm_lib.workspace(nbc, dev), nbc,
                     stream())
            elif need_wgrad:
                nb = tm_lib.ws_bytes("tm_convt2x2_wgrad_ws", *shape)
                dwt, dbt = _empty(u["cin"], 4 * u["cout"], dev=dev), _empty(u["cout"], dev=dev)
                call("tm_convt2x2_wgrad_nhwc", *shape, u["x"], u["ldx"], half,
                     2 * chans[i], Hs[i], Ws_[i], 0, 0, dwt, dbt, ws.get(nb), nb, stream())
                dwu = _empty(u["cin"], u["cout"], 2, 2, dev=dev)
                call("tm_convt_unpack_wgrad", u["cin"], u["cout"], dwt, dwu, stream())
            if tf:
                nb = tm_lib.ws_bytes("tm_convt2x2_tf32_ws", *shape)
                call("tm_convt2x2_tf32_dgrad", *shape, half, 2 * chans[i], u["wdf"], dy, u["cin"],
                     ws.get(nb) if nb else None, nb, tm_lib.err_flag(dev), stream())
            else:
                call("tm_convt2x2_dgrad_nhwc", *shape, half, 2 * chans[i], Hs[i],
                     Ws_[i], 0, 0, u["wtT"], dy, u["cin"], stream())
        if need_wgrad:
            grads[f"{names[j]}.up.weight"], grads[f"{names[j]}.up.bias"] = dwu, dbt
        lddy = u["cin"]
    # encoder, deepest first; dy is the gradient of x4
    enc_names = ["inc.double_conv", "down1.maxpool_conv.1.double_conv", "down2.maxpool_conv.1.double_conv",
                 "down3.maxpool_conv.1.double_conv"]
    for i in (3, 2, 1, 0):
        s = st[f"enc{i}"]
        if i > 0:
            dpool = _empty(B * Hs[i] * Ws_[i], chans[i - 1], dev=dev)
            _double_conv_bwd(ws, s, dy, lddy, grads, enc_names[i], dpool, chans[i - 1], wg=need_wgrad)
            p = st["pool"][i - 1]
            dprev = _empty(B * Hs[i - 1] * Ws_[i - 1], chans[i - 1], dev=dev)
            # pooling backward and the gradient arriving through the skip connection (first half of dcat) in one pass
            call("tm_pool2x2_backward", B, Hs[i - 1], Ws_[i - 1], chans[i - 1], mode, dpool, chans[i - 1], None, 0,
                 p["idx"], dprev, chans[i - 1], 0, dskip[i - 1], 2 * chans[i - 1], stream())
            dy, lddy = dprev, chans[i - 1]
        else:
            dx = _empty(B, 3, H, W, dev=dev) if need_dx else None
            _double_conv_bwd(ws, s, dy, lddy, grads, enc_names[0], None, 0, dimg=dx, w1=st["w_in"], wg=need_wgrad)
    if not need_dx:
        return grads
    return grads, (dx[0] if st["squeeze"] else dx)


UNET_PARAM_ORDER = None


def unet_param_names(net):
    return [k for k, _ in net.named_parameters()]


class UNetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, x, need, *params):
        # `need` is decided by the caller: grad mode is always off inside Function.forward
        out, st = unet_forward(net, x, need_bwd=need, update_stats=net.training)
        ctx.net, ctx.st, ctx.x_dtype = net, st, x.dtype
        ctx.names = unet_param_names(net)
        return out

    @staticmethod
    def backward(ctx, gout):
        if not ctx.needs_input_grad[1]:
            grads = unet_backward(ctx.net, ctx.st, gout)
            return (None, None, None) + tuple(grads[k] for k in ctx.names)
        # frozen parameters (requires_grad=False): the image gradient alone, no weight-gradient kernel
        wg = any(ctx.needs_input_grad[3:])
        grads, dx = unet_backward(ctx.net, ctx.st, gout, need_dx=True, need_wgrad=wg)
        return (None, dx.to(ctx.x_dtype), None) + tuple(grads.get(k) for k in ctx.names)


# --------------------------------------------------------------------------------------------
# LayoutNet (model.py:216-247): conv9 -> ReLU -> pool -> conv7 -> ReLU -> pool -> conv9 -> ReLU
#                               -> conv7 -> LeakyReLU(0.1)
# --------------------------------------------------------------------------------------------
LAYOUT_SPEC = [(0, 2, 32, 9, True), (3, 32, 64, 7, True), (6, 64, 32, 9, False), (8, 32, 1, 7, False)]


def _tma_kxk_ok(B, H, W, cin, cout, k):
    """bf16 mode and a shape the TMA-fed k x k kernels take.  encode.0 (Cin = 2) and encode.8 (Cout = 1) never do:
    padded to 16 channels they would waste 8x / 16x of every MMA."""
    return (USE_TMA and _prec(None) == 0 and cin % 16 == 0 and cout % 16 == 0
            and tm_lib.ws_bytes("tm_convkxk_bf16_supported", B, H, W, cin, cout, k) == 1)


def _pack_kxk_bf16(w, need_dgrad):
    """-> (forward operand [k*k][Cout][Cin], data-gradient operand [k*k][Cin][Cout] or None), bf16."""
    cout, cin, k, _ = w.shape
    wc = w.detach().float().contiguous()

    def one(nc, kc, dgrad):
        q = torch.empty(k * k, nc, kc, dtype=torch.bfloat16, device=w.device)
        call("tm_convkxk_pack_bf16", cout, cin, k, wc, q, kc, dgrad, stream())
        return q
    return one(cout, cin, 0), (one(cin, cout, 1) if need_dgrad else None)


def layoutnet_forward(net, x, need_bwd=True):
    _enter(net)
    squeeze = x.dim() == 3
    if squeeze:
        x = x.unsqueeze(0)
    x = x.detach().float().contiguous()
    tm_lib.require_cuda(x, "LayoutNet input")
    B, C, H, W = x.shape
    dev = x.device
    mode = 0 if net.pooling == "max" else 1
    ws = _Ws(dev)
    cur = _empty(B * H * W, C, dev=dev)
    call("tm_nchw_to_nhwc", B, C, H, W, x, cur, C, stream())
    st = dict(ws=ws, mode=mode, B=B, layers=[], squeeze=squeeze)
    h, w = H, W
    for li, (idx, cin, cout, k, pool) in enumerate(LAYOUT_SPEC):
        conv = net.encode[idx]
        last = li == len(LAYOUT_SPEC) - 1
        y = _empty(B * h * w, cout, dev=dev)
        rec = dict(x=cur, y=y, cin=cin, cout=cout, k=k, H=h, W=w, pool=None, name=f"encode.{idx}")
        if li == 0:                                       # for the gradient w.r.t. the input image
            rec["w"] = conv.weight.detach().float().contiguous()
        if _tma_kxk_ok(B, h, w, cin, cout, k):
            # bf16 mode: TMA-fed tcgen05 k x k convolution; the bf16 copy of x is kept for the weight gradient
            xb = _to_bf16(cur, cin, B * h * w, cin)
            wq, wd = _pack_kxk_bf16(conv.weight, need_bwd and li > 0)
            call("tm_convkxk_bf16", B, h, w, cin, cout, k, xb, wq, conv.bias.detach(), y, cout, 0 if last else RELU,
                 tm_lib.err_flag(dev), stream())
            rec.update(tma=True, xb=xb if need_bwd else None, wd=wd)
        else:
            wf, wb = _pack(conv.weight, need_bwd)
            _conv(cur, cin, B, h, w, cin, cout, k, wf, conv.bias.detach(), y, cout, 0 if last else RELU)
            rec.update(tma=False, wb=wb)
        if last:
            act = _empty(B * h * w, cout, dev=dev)
            call("tm_leaky_relu_forward", B * h * w * cout, y, 0.1, act, stream())
            rec["act"] = act
            cur = act
        elif pool:
            pooled = _empty(B * (h // 2) * (w // 2), cout, dev=dev)
            pidx = torch.empty(B * (h // 2) * (w // 2) * cout, dtype=torch.uint8, device=dev) if mode == 0 else None
            call("tm_pool2x2_forward", B, h, w, cout, mode, y, cout, pooled, cout, pidx, 0, stream())
            rec["pool"] = pidx if mode == 0 else True
            cur, h, w = pooled, h // 2, w // 2
        else:
            cur = y
        st["layers"].append(rec)
    out = cur.reshape(B, 1, h, w)                         # C == 1: NHWC == NCHW
    st["out_hw"] = (h, w)
    return (out[0] if squeeze else out), st


def layoutnet_backward(net, st, gout, need_dx=False, need_wgrad=True):
    """gout: the output's gradient.  Returns {state_dict-style name: gradient}; with ``need_dx`` (grads, dx), dx the
    gradient w.r.t. the input image in its layout: (B,2,H,W), or (2,H,W) for a 3-D input.  ``need_wgrad=False``: no
    weight- or bias-gradient kernel runs and ``grads`` is empty; dx is the same bits."""
    _enter(net)
    B, mode, ws = st["B"], st["mode"], st["ws"]
    dev = gout.device
    g = gout.detach().float().contiguous().reshape(-1, 1)
    grads = {}
    n_layers = len(st["layers"])
    for li in range(n_layers - 1, -1, -1):
        r = st["layers"][li]
        h, w, cin, cout, k = r["H"], r["W"], r["cin"], r["cout"], r["k"]
        npix = B * h * w
        if li == n_layers - 1:
            dy = _empty(npix, cout, dev=dev)
            call("tm_leaky_relu_backward", npix * cout, r["act"], g, 0.1, dy, stream())
        else:
            if r["pool"] is not None:
                dyp = _empty(npix, cout, dev=dev)
                call("tm_pool2x2_backward", B, h, w, cout, mode, g, cout, None, 0,
                     r["pool"] if mode == 0 else None, dyp, cout, 0, None, 0, stream())
                g = dyp
            dy = _empty(npix, cout, dev=dev)
            call("tm_leaky_relu_backward", npix * cout, r["y"], g, 0.0, dy, stream())   # ReLU
        if r["tma"]:
            # one bf16 copy of dy feeds the weight and the data gradient; the bias gradient sums the fp32 dy
            dyb = _to_bf16(dy, cout, npix, cout)
        if need_wgrad and r["tma"]:
            dw, db = _empty(cout, cin, k, k, dev=dev), _empty(cout, dev=dev)
            nb = tm_lib.ws_bytes("tm_convkxk_bf16_wgrad_ws", B, h, w, cin, cout, k)
            call("tm_convkxk_bf16_wgrad", B, h, w, cin, cout, k, r["xb"], dyb, dw, ws.get(nb), nb, tm_lib.err_flag(dev),
                 stream())
            nbc = tm_lib.ws_bytes("tm_colsum_ws", npix, cout)
            call("tm_colsum", npix, cout, dy, cout, None, db, 0, tm_lib.workspace(nbc, dev), nbc, stream())
        elif need_wgrad:
            dw, db = _conv_wgrad(ws, r["x"], cin, dy, cout, B, h, w, cin, cout, k, True)
        if need_wgrad:
            grads[r["name"] + ".weight"], grads[r["name"] + ".bias"] = dw, db
        if li > 0:
            dx = _empty(npix, cin, dev=dev)
            if r["tma"]:
                call("tm_convkxk_bf16", B, h, w, cout, cin, k, dyb, r["wd"], None, dx, cin, 0, tm_lib.err_flag(dev),
                     stream())
            else:
                _conv(dy, cout, B, h, w, cout, cin, k, r["wb"], None, dx, cin)
            g = dx
        elif need_dx:
            # encode.0 (Cin = 2) never takes the TMA route (_tma_kxk_ok): its dy is fp32
            dimg = _empty(B, cin, h, w, dev=dev)
            call("tm_conv_dgrad_narrow", B, h, w, cin, cout, k, dy, cout, 0, r["w"], dimg, stream())
    if not need_dx:
        return grads
    return grads, (dimg[0] if st["squeeze"] else dimg)


class LayoutNetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, x, need, *params):
        out, st = layoutnet_forward(net, x, need_bwd=need)
        ctx.net, ctx.st, ctx.x_dtype = net, st, x.dtype
        ctx.names = [k for k, _ in net.named_parameters()]
        return out

    @staticmethod
    def backward(ctx, gout):
        if not ctx.needs_input_grad[1]:
            grads = layoutnet_backward(ctx.net, ctx.st, gout)
            return (None, None, None) + tuple(grads[k] for k in ctx.names)
        wg = any(ctx.needs_input_grad[3:])                 # frozen parameters: the image gradient alone
        grads, dx = layoutnet_backward(ctx.net, ctx.st, gout, need_dx=True, need_wgrad=wg)
        return (None, dx.to(ctx.x_dtype), None) + tuple(grads.get(k) for k in ctx.names)
