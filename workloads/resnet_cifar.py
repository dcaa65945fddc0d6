"""CIFAR ResNet-(6n+2) layer graph (reference models/resnet.py): a plain 3->16 stem conv, three
stages of n two-conv residual blocks at 16/32/64 channels, stride-2 entry into stages 2 and 3 with
a quantized 1x1 projection shortcut, global average pool, linear head.  Every conv except the stem
is a ``QuantizedConv2d``; every norm is an ``nn.SyncBatchNorm`` as in the reference -- by default the
``FusedSyncBatchNorm`` subclass (same parameters / buffers / state_dict), which takes the residual
add and the ReLU of the block into its own kernels."""
from typing import Callable, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F


def conv_bn_act(conv, bn, x, residual=None, relu=False):
    """relu(bn(conv(x)) + residual).  With this repo's classes (po2_quantization_b200/fold.py): at inference the
    norm, the add and the ReLU are folded into the conv kernel's epilogue (one launch); in training the conv runs,
    then the norm computes its batch statistics and normalises (+ add, + ReLU), in one launch where the tensor fits."""
    if getattr(bn, "fused_residual_relu", False):
        from po2_quantization_b200 import conv_bn_act as fused                # inference: folded; training: conv,
        return fused(conv, bn, x, residual, relu)                             # then the one-launch norm
    return bn_act(bn, conv(x), residual, relu)


def bn_act(bn, x, residual=None, relu=False):
    """relu(bn(x) + residual): one call on a FusedSyncBatchNorm, the three stock ops otherwise."""
    if getattr(bn, "fused_residual_relu", False):
        return bn(x, residual, relu)
    y = bn(x)
    if residual is not None:
        y = y + residual
    return F.relu(y) if relu else y


class _Block(nn.Module):
    def __init__(self, conv_cls, norm_cls, c_in, c_out, stride, quantize_fn, bits):
        super().__init__()
        self.conv1 = conv_cls(c_in, c_out, kernel_size=3, stride=stride, padding=1, quantize_fn=quantize_fn, bits=bits)
        self.bn1 = norm_cls(c_out)
        self.conv2 = conv_cls(c_out, c_out, kernel_size=3, stride=1, padding=1, quantize_fn=quantize_fn, bits=bits)
        self.bn2 = norm_cls(c_out)
        self.downsample = None
        if stride != 1 or c_in != c_out:
            self.downsample = nn.Sequential(
                conv_cls(c_in, c_out, kernel_size=1, stride=stride, padding=0, quantize_fn=quantize_fn, bits=bits),
                norm_cls(c_out))

    def forward(self, x):
        y = conv_bn_act(self.conv1, self.bn1, x, relu=True)
        sc = x if self.downsample is None else conv_bn_act(self.downsample[0], self.downsample[1], x)
        return conv_bn_act(self.conv2, self.bn2, y, residual=sc, relu=True)


class ResNetCifar(nn.Module):
    def __init__(self, conv_cls, norm_cls, n: int, num_classes: int, quantize_fn: Optional[Callable], bits: int,
                 stem_cls=nn.Conv2d):
        super().__init__()
        # never quantized (models/resnet.py:99-102); with this repo's classes StemConv2d = nn.Conv2d with the weight
        # gradient on the small-C kernel
        self.conv1 = stem_cls(3, 16, kernel_size=3, stride=1, padding=1, bias=False)
        self.bn1 = norm_cls(16)
        c_in = 16
        for si, (c_out, stride) in enumerate(((16, 1), (32, 2), (64, 2)), start=1):
            blocks = []
            for bi in range(n):
                blocks.append(_Block(conv_cls, norm_cls, c_in, c_out, stride if bi == 0 else 1, quantize_fn, bits))
                c_in = c_out
            setattr(self, f"layer{si}", nn.Sequential(*blocks))
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))
        self.fc = nn.Linear(64, num_classes)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")

    def forward(self, x):
        x = bn_act(self.bn1, self.conv1(x), relu=True)
        x = self.layer3(self.layer2(self.layer1(x)))
        return self.fc(torch.flatten(self.avgpool(x), 1))

    def quantized_convs(self):
        from po2_quantization_b200 import QuantizedConv2d
        return [m for m in self.modules() if isinstance(m, QuantizedConv2d)]


def resnet_cifar(depth: int, num_classes: int = 10, quantize_fn=None, bits: int = 4, conv_cls=None, norm_cls=None):
    """depth in {20, 32, 44, 56}; conv_cls / norm_cls default to this repo's QuantizedConv2d and
    FusedSyncBatchNorm (tests pass the reference's or the oracle's conv class -- and then get the
    stock nn.SyncBatchNorm -- to build the same graph on another implementation)."""
    assert (depth - 2) % 6 == 0
    if norm_cls is None:
        if conv_cls is None:
            from po2_quantization_b200 import FusedSyncBatchNorm as norm_cls
        else:
            norm_cls = nn.SyncBatchNorm
    stem_cls = nn.Conv2d
    if conv_cls is None:
        from po2_quantization_b200 import QuantizedConv2d as conv_cls
        from po2_quantization_b200 import StemConv2d as stem_cls
    return ResNetCifar(conv_cls, norm_cls, (depth - 2) // 6, num_classes, quantize_fn, bits, stem_cls)
