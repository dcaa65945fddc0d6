"""Inference: eval-mode BatchNorm (+ the block's residual add) (+ its activation) folded into the epilogue of
the quantized conv in front of it -- models/resnet.py:55-71, models/mobilenet.py:29-31, models/mobile_vit.py:20
in ``eval()``: ``act(bn(conv(x)) + shortcut)`` becomes ONE kernel launch, the conv's, with

    out = act(conv(x) * a[k] + b[k] + shortcut),   a = gamma / sqrt(running_var + eps),  b = beta - running_mean * a

(SURVEY.md section 8(f) row 3).  ``conv_bn_act`` is the functional form for model code that applies the norm in
its own ``forward``; ``fold_conv_bn`` rewrites ``nn.Sequential(conv, norm, ...)`` runs in place for inference.
Training, autograd and layers the kernels do not take keep the separate conv and norm calls.
"""
import os
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from .batchnorm import ACT, FusedSyncBatchNorm
from .quantized_conv import QuantizedConv2d


def _affine(bn: nn.modules.batchnorm._BatchNorm):
    """(a, b) of an eval-mode norm, cached on the module until one of its tensors changes"""
    ver = tuple(t._version if t is not None else -1 for t in (bn.weight, bn.bias, bn.running_mean, bn.running_var))
    key = (ver, bn.running_mean.device, float(bn.eps))
    cache = bn.__dict__.get("_po2_affine")
    if cache is None or cache[0] != key:
        with torch.no_grad():
            a = torch.rsqrt(bn.running_var.float() + bn.eps)
            if bn.weight is not None:
                a = a * bn.weight.float()
            b = -bn.running_mean.float() * a
            if bn.bias is not None:
                b = b + bn.bias.float()
        cache = (key, a.contiguous(), b.contiguous())
        bn.__dict__["_po2_affine"] = cache
    return cache[1], cache[2]


def _foldable(conv, bn, x) -> bool:
    return (isinstance(conv, QuantizedConv2d) and isinstance(bn, nn.modules.batchnorm._BatchNorm) and not bn.training
            and bn.running_mean is not None and bn.running_var is not None and x.is_cuda
            and x.dtype in (torch.float32, torch.bfloat16)
            and not (torch.is_grad_enabled() and x.requires_grad))


def conv_bn_act(conv, bn, x: torch.Tensor, residual: Optional[torch.Tensor] = None, relu: bool = False) -> torch.Tensor:
    """act(bn(conv(x)) + residual).  One launch at inference where the layer allows; the separate calls otherwise."""
    act = 1 if relu else ACT[getattr(bn, "act", None)]
    # (SiLU on very large outputs stays a separate pass: measured on MobileViT 224x224 at batch 256, the conv
    # kernels' four epilogue warps per CTA fall behind HBM when they also evaluate exp() per element --
    # 23.6 ms folded against 22.5 ms with the norm kernels -- while the small maps gain)
    big_silu = act == 3 and x.shape[0] * conv.out_channels * x.shape[2] * x.shape[3] // (conv.stride[0] ** 2) > (1 << 24)
    if _foldable(conv, bn, x) and not big_silu and os.environ.get("PO2_FOLD_BN", "1") == "1":
        a, b = _affine(bn)
        out = conv.forward_folded(x, a, b, residual, act)
        if out is not None:
            return out
    y = conv(x)
    if getattr(bn, "fused_residual_relu", False):
        return bn(y, residual, relu)
    y = bn(y)
    if residual is not None:
        y = y + residual
    return F.relu(y) if relu else y


class FoldedConvBN(nn.Module):
    """``norm(conv(x))`` (+ the norm's own activation) as one module, for ``fold_conv_bn``"""

    def __init__(self, conv: QuantizedConv2d, bn: nn.Module):
        super().__init__()
        self.conv, self.bn = conv, bn

    def forward(self, x):
        return conv_bn_act(self.conv, self.bn, x)


def fold_conv_bn(model: nn.Module) -> int:
    """In every ``nn.Sequential`` of ``model``, replace a ``QuantizedConv2d`` directly followed by a
    ``FusedSyncBatchNorm`` with one ``FoldedConvBN`` (the norm's slot becomes ``nn.Identity``, so the indices
    of the other entries do not move).  For inference: the ``state_dict`` keys of the folded pairs change
    (``i.weight`` -> ``i.conv.weight``, ``i+1.*`` -> ``i.bn.*``), so fold AFTER loading weights.  Returns the number
    of folded pairs."""
    n = 0
    for seq in [m for m in model.modules() if isinstance(m, nn.Sequential)]:
        items = list(seq._modules.items())
        for (k0, m0), (k1, m1) in zip(items, items[1:]):
            if isinstance(m0, QuantizedConv2d) and isinstance(m1, FusedSyncBatchNorm):
                seq._modules[k0] = FoldedConvBN(m0, m1)
                seq._modules[k1] = nn.Identity()
                n += 1
    return n


def invalidate_caches(model: nn.Module) -> int:
    """Drop everything this library caches per module keyed on ``Tensor._version``: prefetched / packed weight operands
    (``QuantizedConv2d``) and the folded scale / shift of eval-mode norms.  Needed after REPLAYING a captured training
    step: a CUDA-graph replay runs the optimizer's and the norms' kernels without executing any Python, so version
    counters do not move (true of ``torch.optim`` in-place updates as well) and an eager forward afterwards would meet
    caches that look current but hold the operands of an earlier step.  Returns the number of modules touched."""
    n = 0
    for m in model.modules():
        d = m.__dict__
        hit = False
        for k in ("_po2_prefetch", "_po2_pack_cache", "_po2_affine"):
            if d.pop(k, None) is not None:
                hit = True
        n += int(hit)
    return n


_ACT_OF = {nn.ReLU: "relu", nn.ReLU6: "relu6", nn.SiLU: "silu"}


def fuse_batchnorm(model: nn.Module, fuse_activations: bool = True) -> int:
    """Put the ``nn.SyncBatchNorm`` modules of an UNMODIFIED model (the reference's ``models/resnet.py``,
    ``models/mobilenet.py``, ``models/mobile_vit.py`` construct them directly) on this library's norm kernels, in
    place and after construction: one added line in ``train.py`` / ``test.py`` --
    ``po2_quantization_b200.fuse_batchnorm(model)`` -- instead of an edit of the model files.  Every
    ``nn.SyncBatchNorm`` instance becomes a ``FusedSyncBatchNorm`` (same parameters, buffers and ``state_dict`` keys:
    only the class changes); with ``fuse_activations`` an ``nn.ReLU`` / ``nn.ReLU6`` / ``nn.SiLU`` that directly follows
    a norm inside an ``nn.Sequential`` moves into the norm kernel (its slot becomes ``nn.Identity``).  Activations and
    residual adds that a model applies in its own ``forward`` (``F.relu(self.bn1(...))``) stay torch ops.  Returns the
    number of converted norms."""
    n = 0
    for m in model.modules():
        if type(m) is nn.SyncBatchNorm:
            m.__class__ = FusedSyncBatchNorm
            m.act = None
            n += 1
    if fuse_activations:
        for seq in [m for m in model.modules() if isinstance(m, nn.Sequential)]:
            items = list(seq._modules.items())
            for (k0, m0), (k1, m1) in zip(items, items[1:]):
                if isinstance(m0, FusedSyncBatchNorm) and getattr(m0, "act", None) is None and type(m1) in _ACT_OF:
                    m0.act = _ACT_OF[type(m1)]
                    seq._modules[k1] = nn.Identity()
    return n
