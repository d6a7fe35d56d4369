"""Drop-in ``Unet`` module: the reference's U-Net surface on libtm_b200 (sm_100a).

``UNet(pooling, bilinear=False)`` has the reference's sub-module tree, so parameter and buffer
names (``inc.double_conv.0.weight`` ... ``outc.conv.0.bias``) and whole-module pickles are
interchangeable with ``src/Unet.py``.  The sub-modules only HOLD parameters: the forward and
backward passes are the CUDA implicit-GEMM / BatchNorm / pooling kernels driven by
``tm_unet.py``.  Output is (B, 1, H/2, W/2) like Unet.py:74-78,118; a 3-D (C,H,W) input is
accepted (train.py:465 passes one).
"""
import torch
import torch.nn as nn

import tm_unet


def _no_eager(name):
    def forward(self, *a, **k):
        raise RuntimeError(f"{name} only holds parameters here; call UNet.forward (CUDA path)")
    return forward


class DoubleConv(nn.Module):
    forward = _no_eager("DoubleConv")

    def __init__(self, in_channels, out_channels, mid_channels=None):
        super().__init__()
        mid = mid_channels or out_channels
        self.double_conv = nn.Sequential(
            nn.Conv2d(in_channels, mid, kernel_size=3, padding=1, bias=False), nn.BatchNorm2d(mid),
            nn.ReLU(inplace=True),
            nn.Conv2d(mid, out_channels, kernel_size=3, padding=1, bias=False), nn.BatchNorm2d(out_channels),
            nn.ReLU(inplace=True))


class Down(nn.Module):
    forward = _no_eager("Down")

    def __init__(self, pooling, in_channels, out_channels):
        super().__init__()
        self.maxpool_conv = nn.Sequential(pooling, DoubleConv(in_channels, out_channels))


class Up(nn.Module):
    forward = _no_eager("Up")

    def __init__(self, in_channels, out_channels, bilinear=True):
        super().__init__()
        if bilinear:
            raise NotImplementedError("bilinear up-sampling is never constructed by the reference "
                                      "(train.py:70); only ConvTranspose2d(k=2, s=2) is implemented")
        self.up = nn.ConvTranspose2d(in_channels, in_channels // 2, kernel_size=2, stride=2)
        self.conv = DoubleConv(in_channels, out_channels)


class OutConv(nn.Module):
    forward = _no_eager("OutConv")

    def __init__(self, pooling, in_channels, out_channels):
        super(OutConv, self).__init__()
        self.conv = nn.Sequential(nn.Conv2d(in_channels, out_channels, kernel_size=1), pooling,
                                  nn.ReLU(inplace=True))


class UNet(nn.Module):
    def __init__(self, pooling, bilinear=False):
        super(UNet, self).__init__()
        if pooling == 'max':
            pooling_layer = nn.MaxPool2d(2)
        elif pooling == 'avg':
            pooling_layer = nn.AvgPool2d(2)
        else:
            assert False, 'wrong pooling type for layoutnet!'
        self.pooling = pooling
        self.n_channels = 3
        self.bilinear = bilinear
        self.inc = DoubleConv(3, 16)
        self.down1 = Down(pooling_layer, 16, 32)
        self.down2 = Down(pooling_layer, 32, 64)
        self.down3 = Down(pooling_layer, 64, 128)
        self.up1 = Up(128, 64, bilinear)
        self.up2 = Up(64, 32, bilinear)
        self.up3 = Up(32, 16, bilinear)
        self.outc = OutConv(pooling_layer, 16, 1)

    def __setstate__(self, state):                       # pickles written by the reference lack .pooling
        super().__setstate__(state)
        if "pooling" not in self.__dict__:
            self.pooling = "avg" if isinstance(self.outc.conv[1], nn.AvgPool2d) else "max"

    def forward(self, x):
        params = list(self.parameters())
        need = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
        return tm_unet.UNetFn.apply(self, x, need, *params)
