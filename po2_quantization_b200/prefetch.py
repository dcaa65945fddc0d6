"""Weight quantization for all layers at once (QAT).

``QuantizedConv2d.forward`` quantizes its weight on every call (models/quantized_conv.py:34-36):
56 tiny launches per ResNet-56 forward, each sitting in the layer chain in front of its conv.  That
work does not depend on the activations, so ``prefetch_weights(layers)`` does it for ALL PO2/PO2+
layers in ONE multi-tensor launch (``po2_quantize_pack_multi``: one thread-block cluster per weight
tensor, each emitting the quantized weight, its scale and the conv's packed tensor-core operand); a
layer's forward then runs its conv as a single launch from the prefetched operand.
``enable_weight_prefetch(model)`` installs this as a forward pre-hook, so the reference's training
loop needs no change.

Everything runs on the current stream and is CUDA-graph capturable.  Buffers are persistent per
module and keyed by (weight version, input shape, conv mode, bits, quantizer); a layer whose key does
not match takes the ordinary ``po2::qconv2d`` path, which also records the input shape the next
prefetch needs.  Layers the multi-tensor kernel does not take (weights larger than one cluster's
registers, channel counts that need padding) are quantized one by one with ``po2_quantize_pack``.
"""
import os
from typing import Iterable

import torch

from . import _lib, ops
from . import quantizers as _quantizers


class _Slot:
    __slots__ = ("key", "qw", "scale", "packed", "sse", "packed_d")


class _Table:
    """device table of MultiDesc entries for a fixed set of slots"""
    __slots__ = ("ident", "dev", "n", "csize")


def _layer_key(m, xshape, mode):
    fam, plus = _quantizers.quantizer_family(m.quantize_fn)
    return (m.weight._version, tuple(xshape), mode, int(m.bits), plus, m.weight.device, fam)


def _static(key):
    return key[1:]


_tables = {}
_pending_quantize = {}             # device index -> event of a quantizer launch on the side stream not yet waited for


def single_layers(layers) -> bool:
    return any(m.__dict__.get("_po2_prefetch_single") for m, _slot, _key in layers)


def wait_for_quantizer(device) -> None:
    """the current stream waits for a quantizer launch that prefetch_weights put on the side stream (once)"""
    ev = _pending_quantize.pop(device.index, None)
    if ev is not None:
        torch.cuda.current_stream(device).wait_event(ev)


def prefetch_weights(modules: Iterable[torch.nn.Module]) -> int:
    """Quantize + pack the weights of every eligible layer whose weights changed; returns how many
    layers now hold a valid prefetched operand."""
    from .quantized_conv import QuantizedConv2d
    mode = ops.get_conv_mode()
    if mode not in ("tc", "tf32"):
        return 0
    compute = ops.COMPUTE[mode]
    lib = _lib.load()
    layers, stale = {"po2": [], "lin": []}, {"po2": False, "lin": False}
    lin_on = os.environ.get("PO2_LIN", "cuda") == "cuda"
    for m in modules:
        if not isinstance(m, QuantizedConv2d) or m.quantize_fn is None:
            continue
        fam = _quantizers.quantizer_family(m.quantize_fn)
        if fam is None:
            continue
        xshape = m.__dict__.get("_po2_xshape")
        w = m.weight
        if xshape is None or not w.is_cuda or w.dtype != torch.float32 or not w.is_contiguous():
            continue
        if fam[0] == "lin":
            # only weights that are their own exact operand and that the lin quantizer kernel takes (the inline path
            # reports the others)
            K, _, R, S = w.shape
            if not lin_on or not 2 <= int(m.bits) <= ops.LIN_EXACT_BITS[mode] or \
                    K * R * S > lib.po2_lin_max_channel_elems():
                continue
        key = _layer_key(m, xshape, mode)
        slot = m.__dict__.get("_po2_prefetch")
        if slot is False:                                        # known not to run on the tensor-core kernel
            if m.__dict__.get("_po2_prefetch_static") == _static(key):
                continue
            slot = None
        if slot is None or _static(slot.key) != _static(key):
            B, C, H, W_ = xshape
            K, _, R, S = w.shape
            nbytes = int(lib.po2_conv2d_pack_bytes(B, C, H, W_, K, R, S, m.stride[0], m.padding[0], m.groups, compute))
            if nbytes == 0:
                m.__dict__["_po2_prefetch"] = False
                m.__dict__["_po2_prefetch_static"] = _static(key)
                continue
            slot = _Slot()
            slot.qw = torch.empty_like(w, memory_format=torch.contiguous_format)
            slot.packed = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
            if fam[0] == "lin":
                slot.scale = ops.lin_scale(w.device)                        # the lin operand is y itself
                slot.sse = None
            else:
                slot.scale = torch.empty((), dtype=torch.float32, device=w.device)
                slot.sse = torch.zeros((), dtype=torch.float64, device=w.device)   # sum((Q(w)-w)^2), refreshed by every launch
            # the data-gradient conv's operand (stride-1 dense layers), emitted by the same launch
            nd = 0
            if m.stride[0] == 1 and m.groups == 1 and ops._dgrad_mode == "tc":
                nd = int(lib.po2_conv2d_dgrad_pack_bytes(B, C, H, W_, K, R, S, m.padding[0], compute))
            slot.packed_d = torch.empty(nd, dtype=torch.uint8, device=w.device) if nd else None
            slot.key = None
            m.__dict__["_po2_prefetch"] = slot
        if slot.key != key:
            stale[fam[0]] = True
        layers[fam[0]].append((m, slot, key))
    # a model that mixes families gets one launch per family
    if layers["po2"] and stale["po2"]:
        _launch_po2(layers["po2"], lib, compute)
    if layers["lin"] and stale["lin"]:
        _launch_lin(layers["lin"], lib, compute)
    return len(layers["po2"]) + len(layers["lin"])


def _launch_po2(layers, lib, compute) -> None:
    dev = layers[0][0].weight.device
    with torch.cuda.device(dev):
        stream = ops._stream_ptr(dev)
        ident = tuple((id(m), slot.qw.data_ptr(), m.weight.data_ptr(), _static(key)) for m, slot, key in layers)
        tab = _tables.get(id(layers[0][0]))
        if tab is None or tab.ident != ident:
            # (re)build the descriptor table: host fill through the C ABI, one copy to the device
            dbytes = int(lib.po2_multi_desc_bytes())
            host = torch.zeros(len(layers) * dbytes, dtype=torch.uint8)
            multi, single, csize = [], [], 1
            for m, slot, key in layers:
                B, C, H, W_ = key[1]
                K, _, R, S = m.weight.shape
                rc = lib.po2_multi_desc_fill(host.data_ptr(), len(multi), m.weight.data_ptr(), slot.qw.data_ptr(),
                                             slot.scale.data_ptr(), slot.packed.data_ptr(), slot.packed.numel(), B, C, H,
                                             W_, K, R, S, m.stride[0], m.padding[0], m.groups, int(m.bits), 1, int(key[4]),
                                             ops._flavor, compute, slot.sse.data_ptr())
                if rc == -10:
                    single.append(m)
                    slot.sse = None                              # po2_quantize_pack has no fused error output
                    slot.packed_d = None
                    continue
                if rc <= 0:
                    _lib.check(rc if rc < 0 else -6, "po2_multi_desc_fill")
                if slot.packed_d is not None:
                    rd = lib.po2_multi_desc_fill_dgrad(host.data_ptr(), len(multi), slot.packed_d.data_ptr(),
                                                       slot.packed_d.numel(), B, C, H, W_, K, R, S, m.stride[0],
                                                       m.padding[0], m.groups, compute)
                    if rd == -10:
                        slot.packed_d = None
                    else:
                        _lib.check(rd, "po2_multi_desc_fill_dgrad")
                csize = max(csize, rc)
                multi.append(m)
            tab = _Table()
            tab.ident, tab.n, tab.csize = ident, len(multi), csize
            tab.dev = host[:max(len(multi), 1) * dbytes].to(dev)
            _tables[id(layers[0][0])] = tab
            one_by_one = {id(m) for m in single}
            for m, slot, key in layers:
                m.__dict__["_po2_prefetch_single"] = id(m) in one_by_one
        if tab.n:
            ops.LAUNCHES += 1
            if ops.get_wgrad_overlap() and not single_layers(layers) and os.environ.get("PO2_QUANT_STREAM", "0") == "1":
                # opt-in (PO2_QUANT_STREAM=1), measured and not kept: the model's first layers (the full-precision stem
                # conv and its norm) do not need the quantized weights, so the quantizer launch can run beside them on the
                # side stream, the first prefetched conv waiting for it (try_prefetched_forward).  In the captured step the
                # second branch's first kernel starts ~50 us after the stem's, later than it would in line: 2.333 vs
                # 2.317 ms per ResNet-56 step.
                main = torch.cuda.current_stream(dev)
                side = ops.side_stream(dev)
                side.wait_stream(main)                           # the optimizer's update of the weights
                with torch.cuda.stream(side):
                    _lib.check(lib.po2_quantize_pack_multi(tab.dev.data_ptr(), tab.n, tab.csize, ops._stream_ptr(dev)),
                               "po2_quantize_pack_multi")
                    ev = torch.cuda.Event()
                    ev.record(side)
                _pending_quantize[dev.index] = ev
            else:
                _lib.check(lib.po2_quantize_pack_multi(tab.dev.data_ptr(), tab.n, tab.csize, stream), "po2_quantize_pack_multi")
        qws = None
        for m, slot, key in layers:
            if m.__dict__.get("_po2_prefetch_single"):
                if qws is None:
                    qws = ops._workspace(dev).data_ptr()
                B, C, H, W_ = key[1]
                K, _, R, S = m.weight.shape
                ops.LAUNCHES += 2
                _lib.check(lib.po2_quantize_pack(m.weight.data_ptr(), slot.qw.data_ptr(), slot.scale.data_ptr(),
                                                 slot.packed.data_ptr(), slot.packed.numel(), B, C, H, W_, K, R, S,
                                                 m.stride[0], m.padding[0], m.groups, int(m.bits), 1, int(key[4]),
                                                 ops._flavor, compute, qws, stream), "po2_quantize_pack")
            slot.key = key


def _launch_lin(layers, lib, compute) -> None:
    """lin / lin+ layers: y, the forward operand and the stride-1 data-gradient operand of every layer in ONE launch of
    the multi-tensor lin kernel (one CTA per input channel); layers whose operand needs channel padding one by one"""
    dev = layers[0][0].weight.device
    with torch.cuda.device(dev):
        stream = ops._stream_ptr(dev)
        ident = tuple((id(m), slot.qw.data_ptr(), m.weight.data_ptr(), _static(key)) for m, slot, key in layers)
        tkey = (id(layers[0][0]), "lin")
        tab = _tables.get(tkey)
        if tab is None or tab.ident != ident:
            dbytes = int(lib.po2_lin_multi_desc_bytes())
            host = torch.zeros(len(layers) * dbytes, dtype=torch.uint8)
            n, ctas, max_elems, single = 0, 0, 1, set()
            for m, slot, key in layers:
                B, C, H, W_ = key[1]
                K, _, R, S = m.weight.shape
                pd = slot.packed_d
                rc = lib.po2_lin_multi_desc_fill(host.data_ptr(), n, m.weight.data_ptr(), slot.qw.data_ptr(),
                                                 slot.packed.data_ptr(), slot.packed.numel(),
                                                 pd.data_ptr() if pd is not None else None, pd.numel() if pd is not None else 0,
                                                 B, C, H, W_, K, R, S, m.stride[0], m.padding[0], m.groups, int(m.bits),
                                                 ops.LIN_ITERS, int(key[4]), ops._flavor, compute)
                if rc == -10:
                    single.add(id(m))
                    slot.packed_d = None
                    continue
                if rc <= 0:
                    _lib.check(rc if rc < 0 else -6, "po2_lin_multi_desc_fill")
                n += 1
                ctas += rc
                max_elems = max(max_elems, K * R * S)
            tab = _Table()
            tab.ident, tab.n, tab.csize = ident, n, (ctas, max_elems)
            tab.dev = host[:max(n, 1) * dbytes].to(dev)
            _tables[tkey] = tab
            for m, slot, key in layers:
                m.__dict__["_po2_prefetch_single"] = id(m) in single
        if tab.n:
            ops.LAUNCHES += 1
            _lib.check(lib.po2_lin_quantize_pack_multi(tab.dev.data_ptr(), tab.n, tab.csize[0], tab.csize[1], stream),
                       "po2_lin_quantize_pack_multi")
        for m, slot, key in layers:
            if m.__dict__.get("_po2_prefetch_single"):
                B, C, H, W_ = key[1]
                K, _, R, S = m.weight.shape
                ops.LAUNCHES += 2
                _lib.check(lib.po2_lin_quantize_pack(m.weight.data_ptr(), slot.qw.data_ptr(), slot.packed.data_ptr(),
                                                     slot.packed.numel(), None, 0, B, C, H, W_, K, R, S, m.stride[0],
                                                     m.padding[0], m.groups, int(m.bits), ops.LIN_ITERS, int(key[4]),
                                                     ops._flavor, compute, stream), "po2_lin_quantize_pack")
            slot.key = key


class _QConvPrefetched(torch.autograd.Function):
    """conv2d(x, Q(weight)) from a prefetched (qw, scale, packed) triple; straight-through gradient"""

    @staticmethod
    def forward(ctx, x, weight, qw, scale, packed, stride, pad, groups, compute, packed_d):
        K, _, R, S = qw.shape
        out = ops.conv2d_packed(x, packed, scale, K, R, S, stride, pad, groups, compute)
        ctx.save_for_backward(x, qw, scale)
        ctx.packed_d = packed_d          # valid until the next prefetch launch, i.e. through this step's backward
        ctx.weight = weight              # the parameter: backward defers the weight gradient only if it has no .grad
        ctx.cfg = (stride, pad, groups, compute)
        return out

    @staticmethod
    def backward(ctx, g):
        x, qw, scale = ctx.saved_tensors
        stride, pad, groups, compute = ctx.cfg
        wp = ctx.weight
        # ops.set_wgrad_overlap: the weight gradient may run on the side stream when autograd will install it as
        # wp.grad by reference (leaf without a gradient yet, no hooks that would read it during backward)
        defer = (wp.is_leaf and wp.grad is None and not wp._backward_hooks
                 and not getattr(wp, "_post_accumulate_grad_hooks", None))
        gx, gw = ops._conv_backward(g, x, qw, scale, stride, pad, groups, compute, ctx.needs_input_grad[0],
                                    ctx.needs_input_grad[1], packed_d=ctx.packed_d, defer_w=defer)
        return gx, gw, None, None, None, None, None, None, None, None


def try_prefetched_forward(m, x, mode):
    """The layer's forward from its prefetched operand, or None if there is no valid one."""
    slot = m.__dict__.get("_po2_prefetch")
    if not slot or slot.key != _layer_key(m, x.shape, mode):
        return None
    if _pending_quantize:
        wait_for_quantizer(x.device)
    return _QConvPrefetched.apply(x, m.weight, slot.qw, slot.scale, slot.packed, m.stride[0], m.padding[0], m.groups,
                                  ops.COMPUTE[mode], getattr(slot, "packed_d", None))


def enable_weight_prefetch(model: torch.nn.Module) -> torch.nn.Module:
    """Install the prefetch as a forward pre-hook on `model`: before each forward the weights of all its
    PO2/PO2+ QuantizedConv2d layers are quantized in one launch."""
    from .quantized_conv import QuantizedConv2d
    layers = [m for m in model.modules() if isinstance(m, QuantizedConv2d)]

    def pre(_mod, _args):
        prefetch_weights(layers)

    model.register_forward_pre_hook(pre)
    return model
