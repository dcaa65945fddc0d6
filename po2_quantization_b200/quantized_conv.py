"""Host-side mirror of the reference's ``models/quantized_conv.py``.

``QuantizedConv2d`` keeps the reference's constructor (note ``padding=1, bias=False`` defaults),
attributes (``quantize_fn``, ``bits``), ``state_dict`` (``{weight}``) and methods, so the
reference's model files build on it unchanged (SURVEY.md section 8b).
"""
import copy
import os

import torch
import torch.nn as nn

from . import ops


class QuantizedConv2d(nn.Conv2d):
    """reference models/quantized_conv.py:5-45"""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=1, dilation=1,
                 groups=1, bias=False, quantize_fn=None, bits=4):
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias)
        self.quantize_fn = quantize_fn
        self.bits = bits

    def __deepcopy__(self, memo):
        # test.py:120 deep-copies models; a copied Parameter restarts its version counter, so the
        # (non-persistent) PTQ tag is re-keyed to the copy instead of silently going stale
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        new.__dict__ = {k: copy.deepcopy(v, memo) for k, v in self.__dict__.items()
                        if k not in ("_po2_pack_cache", "_po2_prefetch", "_po2_prefetch_single", "_po2_prefetch_static")}
        for name in ("_po2_ptq", "_po2_lin_ptq"):
            tag = self.__dict__.get(name)
            if tag is not None and tag[0] == self.weight._version:
                new.__dict__[name] = (new.weight._version,) + tuple(new.__dict__[name][1:])
        return new

    # ---- which inputs the sm_100a conv kernels take.  Anything else goes to nn.Conv2d's own path
    # (cuDNN) -- never silently: _why_not() names the reason and forward() reports it once per reason
    # (ops.note_library_path; an error under PO2_STRICT=1).  Every QuantizedConv2d the reference's model
    # files construct (bias=False, dilation 1, square stride/padding, fp32) is taken, and so is a bf16 model's layer
    # at inference (no gradient, mode tc / tf32) on the kernels that have a bf16 form.
    def _bf16_inference(self, input) -> bool:
        return (input.dtype == torch.bfloat16 and self.weight.dtype == torch.bfloat16
                and ops.get_conv_mode() in ("tc", "tf32")
                and not (torch.is_grad_enabled() and (input.requires_grad or self.weight.requires_grad)))

    def _why_not(self, input):
        if ops.get_conv_mode() == "cudnn":
            return None                                       # the caller asked for cuDNN: not a fallback
        if not input.is_cuda:
            return "CPU input"
        bf16 = self._bf16_inference(input)
        if (input.dtype != torch.float32 or self.weight.dtype != torch.float32) and not bf16:
            return f"dtype {input.dtype}/{self.weight.dtype} (fp32 NCHW only)"
        if input.dim() != 4:
            return f"{input.dim()}-D input (batched NCHW only)"
        if self.bias is not None:
            return "bias=True"
        if self.dilation != (1, 1):
            return f"dilation {self.dilation}"
        if self.padding_mode != "zeros" or not isinstance(self.padding, tuple):
            return f"padding {self.padding!r} / padding_mode {self.padding_mode!r}"
        if self.stride[0] != self.stride[1] or self.padding[0] != self.padding[1]:
            return f"non-square stride {self.stride} / padding {self.padding}"
        # the planner's answer for this input shape, asked once per shape: PO2_E_SIZE when x or the output has 2^31 or
        # more elements (the kernels index them in 32 bits), PO2_E_UNSUPPORTED for a bf16 shape no bf16 kernel takes
        key = (tuple(input.shape), tuple(self.weight.shape), input.dtype, ops.get_conv_mode())
        kind = self.__dict__.get("_po2_kind")
        if kind is None or kind[0] != key:
            kind = (key, ops.conv_kernel_kind(input.shape, self.weight.shape, self.stride[0], self.padding[0], self.groups,
                                              ops.COMPUTE[key[3]], input.dtype))
            self.__dict__["_po2_kind"] = kind
        if kind[1] == ops.E_SIZE:
            return f"input {list(input.shape)} (x and the output must each have fewer than 2^31 elements)"
        if bf16 and kind[1] < 0:
            return f"bf16 layer {list(self.weight.shape)} groups {self.groups} (no bf16 kernel for this shape)"
        return ""

    def _po2_conv_ok(self, input) -> bool:
        return self._why_not(input) == ""

    def _lin_why_not(self, input, bits, quantizes=True):
        """_why_not for a lin / lin+ weight, which is its own exact operand only up to ops.LIN_EXACT_BITS of the mode
        (quantizes: the lin quantizer kernel runs in this forward and must take the channel size)"""
        why = self._why_not(input)
        if why != "":
            return why
        if input.dtype != torch.float32:
            return f"dtype {input.dtype}/{self.weight.dtype} (fp32 NCHW only)"
        mode = ops.get_conv_mode()
        if not 2 <= bits <= ops.LIN_EXACT_BITS[mode]:
            return f"lin weights of {bits} bits are not exact as {mode} operands (at most {ops.LIN_EXACT_BITS[mode]} bits)"
        if quantizes:
            from . import _lib
            K, _, R, S = self.weight.shape
            if K * R * S > _lib.load().po2_lin_max_channel_elems():
                return f"lin quantizer channel of {K * R * S} weights exceeds the kernel's shared-memory capacity"
        return ""

    def _lin_forward(self, input, plus):
        """QAT forward of a lin / lin+ layer, or None where it keeps nn.Conv2d's own convolution (reported on CUDA)"""
        bits = int(self.bits)
        if os.environ.get("PO2_LIN", "cuda") != "cuda":
            return None                                       # the op-by-op quantizer reports itself
        why = self._lin_why_not(input, bits)
        if why is None or not input.is_cuda:
            return None                                       # cudnn mode / CPU: the stock path, as requested
        if why:
            ops.note_library_path("qconv:" + why, f"QuantizedConv2d runs nn.Conv2d's own convolution (cuDNN) for this "
                                  f"layer: {why}")
            return None
        mode = ops.get_conv_mode()
        if mode in ("tc", "tf32"):
            from . import prefetch
            out = prefetch.try_prefetched_forward(self, input, mode)
            if out is not None:
                return out
            self.__dict__["_po2_xshape"] = tuple(input.shape)
        out, _y = ops.lin_qconv2d(input, self.weight, bits, bool(plus), self.stride[0], self.padding[0], self.groups,
                                  ops.COMPUTE[mode])
        return out

    def _lin_ptq_forward(self, input, tag):
        """forward of a layer quantize_model() wrote lin / lin+ weights into: the weight is its own operand, scale 1.0"""
        why = self._lin_why_not(input, tag[1], quantizes=False)
        if why is None or (why and not input.is_cuda):
            return self._conv_forward(input, self.weight, self.bias)
        if why:
            return self._library_conv(input, self.weight, why)
        mode = ops.get_conv_mode()
        one = ops.lin_scale(input.device)
        if mode in ("tc", "tf32") and not (torch.is_grad_enabled() and (input.requires_grad or self.weight.requires_grad)):
            packed = self._ptq_packed(input, tag[0], one, mode)
            if packed is not None:
                K, _, R, S = self.weight.shape
                return ops.conv2d_packed(input, packed, one, K, R, S, self.stride[0], self.padding[0], self.groups,
                                         ops.COMPUTE[mode])
        return ops.conv2d(input, self.weight, one, self.stride[0], self.padding[0], self.groups, ops.COMPUTE[mode])

    def _ptq_packed(self, input, version, scale, mode):
        """the packed operand of the static weight, built once per (weight version, input shape); None: no such operand"""
        key = (version, tuple(input.shape), input.device, mode)
        cache = self.__dict__.get("_po2_pack_cache")
        if cache is None or cache[0] != key:
            packed = ops.conv2d_pack(self.weight.detach(), scale, tuple(input.shape), self.stride[0], self.padding[0],
                                     self.groups, ops.COMPUTE[mode])
            cache = (key, packed)
            self.__dict__["_po2_pack_cache"] = cache
        return cache[1]

    def _bf16_forward(self, input, family, ep=None):
        """forward of a bf16 PO2 / PO2+ / lin / lin+ layer at inference (PTQ weights, or a QAT layer in eval); family:
        what _bf16_layer returned; ep = (ep_a, ep_b, residual, act) for the folded form.  Cached in _po2_pack_cache per
        (weight version, input shape, device, mode, dtype, family): the packed operand, or the fp32 widening of the bf16
        weight for the depthwise / small-pointwise kernels.  A QAT layer's weight is quantized in bf16 first
        (quantize_full, or the bf16 lin kernel), as the quantizer itself does on a bf16 model.  A lin weight y is a bf16
        tensor, so it is its own exact operand at any bit width, with scale 1.0 (ops.lin_scale)."""
        mode = ops.get_conv_mode()
        compute, w = ops.COMPUTE[mode], self.weight
        stride, pad, groups = self.stride[0], self.padding[0], self.groups
        fam = _quantizers.quantizer_family(self.quantize_fn) if self.quantize_fn is not None else None
        qat = (int(self.bits), fam[1]) if fam is not None else ()
        key = (w._version, tuple(input.shape), input.device, mode, input.dtype, family) + qat
        cache = self.__dict__.get("_po2_pack_cache")
        if cache is None or cache[0] != key:
            if family == "lin":
                y = (_quantizers._lin_forward_cuda(w.detach(), int(self.bits), ops.LIN_ITERS, fam[1]) if qat
                     else w.detach())
                scale = ops.lin_scale(input.device)
            elif qat:
                y, _codes, scale, _zc, _sse = ops.quantize_full(w.detach(), int(self.bits), 1, bool(fam[1]))
            else:
                y, scale = w.detach(), self._po2_ptq[1]
            packed = ops.conv2d_pack(y, scale, tuple(input.shape), stride, pad, groups, compute, input.dtype)
            cache = (key, packed, y.float() if packed is None else None, scale)
            self.__dict__["_po2_pack_cache"] = cache
        _, packed, wf, scale = cache
        K, _, R, S = w.shape
        if ep is None:
            if packed is not None:
                return ops.conv2d_packed(input, packed, scale, K, R, S, stride, pad, groups, compute)
            return ops.conv2d(input, wf, scale, stride, pad, groups, compute)
        ep_a, ep_b, residual, act = ep
        if packed is not None:
            return ops.conv2d_packed_ep(input, packed, scale, K, R, S, stride, pad, groups, compute, ep_a, ep_b, residual,
                                        int(act))
        return ops.conv2d_ep(input, wf, scale, stride, pad, groups, compute, ep_a, ep_b, residual, int(act))

    def _bf16_layer(self, input):
        """"po2" / "lin": the quantizer family of a layer whose bf16 call the kernels take at inference (a PO2 / lin QAT
        quantizer, or a current PTQ tag); None for any other layer or call.  A lin QAT layer also needs the bf16 lin
        quantizer kernel to take its weight."""
        if self.quantize_fn is not None:
            fam = _quantizers.quantizer_family(self.quantize_fn)
            family = fam[0] if fam is not None else None
            if family == "lin":
                from . import _lib
                K, _, R, S = self.weight.shape
                if (os.environ.get("PO2_LIN", "cuda") != "cuda" or not 2 <= int(self.bits) <= 16
                        or K * R * S > _lib.load().po2_lin_max_channel_elems()):
                    family = None
        else:
            family = None
            for name, tagged in (("_po2_ptq", "po2"), ("_po2_lin_ptq", "lin")):
                tag = self.__dict__.get(name)
                if tag is not None and tag[0] == self.weight._version:
                    family = tagged
                    break
        if family is None or input.dtype != torch.bfloat16 or self._why_not(input) != "":
            return None
        return family

    def _library_conv(self, input, weight, why):
        if why:
            ops.note_library_path("qconv:" + why, f"QuantizedConv2d runs nn.Conv2d's own convolution (cuDNN) for this "
                                  f"layer: {why}")
        if input.dim() == 4:
            ops.check_conv_shapes(input.shape, weight.shape, self.groups, self.padding[0] if isinstance(self.padding, tuple) else 0)
        return self._conv_forward(input, weight, self.bias)

    def _po2_conv(self, input, weight, scale):
        return ops.conv2d(input, weight, scale, self.stride[0], self.padding[0], self.groups,
                          ops.COMPUTE[ops.get_conv_mode()])

    def forward(self, input):
        # models/quantized_conv.py:32-38: quantize the weight on every forward (QAT), then conv
        if input.dtype == torch.bfloat16 and input.is_cuda:
            family = self._bf16_layer(input)
            if family is not None:
                return self._bf16_forward(input, family)
        if self.quantize_fn is not None:
            fam = _quantizers.quantizer_family(self.quantize_fn)
            if fam is not None and fam[0] == "lin":
                out = self._lin_forward(input, fam[1])
                if out is not None:
                    return out
            plus = fam[1] if fam is not None and fam[0] == "po2" else None
            if plus is not None and self._po2_conv_ok(input):
                mode = ops.get_conv_mode()
                if mode in ("tc", "tf32"):
                    # weights already quantized by the multi-tensor prefetch (prefetch.py)?  Then the conv
                    # is a single launch; otherwise remember the input shape for the next prefetch
                    from . import prefetch
                    out = prefetch.try_prefetched_forward(self, input, mode)
                    if out is not None:
                        return out
                    self.__dict__["_po2_xshape"] = tuple(input.shape)
                # PO2 / PO2+: one op = quantizer kernel (which also emits the packed +-2^q tensor-core
                # operand) + conv kernel; the straight-through gradient reaches self.weight
                out, _qw, _scale = ops.qconv2d(input, self.weight, int(self.bits), 1, bool(plus), self.stride[0],
                                               self.padding[0], self.groups, ops.COMPUTE[ops.get_conv_mode()])
                return out
            # a lin / lin+ layer the kernels do not take (reported by _lin_forward on CUDA), or a PO2 layer whose
            # configuration the kernels do not take
            quantized_weight = self.quantize_fn.apply(self.weight, self.bits)
            return self._library_conv(input, quantized_weight, self._why_not(input) if plus is not None else None)
        tag = getattr(self, "_po2_ptq", None)
        if tag is not None and tag[0] == self.weight._version:
            why = self._why_not(input)
            if why:
                return self._library_conv(input, self.weight, why)
            # post-training-quantized weights (quantize_model): already on the grid +-scale*2^q
            mode = ops.get_conv_mode()
            if mode in ("tc", "tf32") and not (torch.is_grad_enabled() and (input.requires_grad or self.weight.requires_grad)):
                # static weights, no autograd: pack the tensor-core operand once per (weight version,
                # input shape) and run each forward as a single launch
                key = (tag[0], tuple(input.shape), input.device, mode)
                cache = self.__dict__.get("_po2_pack_cache")
                if cache is None or cache[0] != key:
                    packed = ops.conv2d_pack(self.weight.detach(), tag[1], tuple(input.shape), self.stride[0],
                                             self.padding[0], self.groups, ops.COMPUTE[mode])
                    cache = (key, packed)
                    self.__dict__["_po2_pack_cache"] = cache
                if cache[1] is not None:
                    K, _, R, S = self.weight.shape
                    return ops.conv2d_packed(input, cache[1], tag[1], K, R, S, self.stride[0], self.padding[0], self.groups,
                                             ops.COMPUTE[mode])
            if why is None:
                return self._conv_forward(input, self.weight, self.bias)
            return self._po2_conv(input, self.weight, tag[1])
        tag = self.__dict__.get("_po2_lin_ptq")
        if tag is not None and tag[0] == self.weight._version:
            return self._lin_ptq_forward(input, tag)
        # no quantizer and no PTQ tag: a full-precision layer, i.e. plain nn.Conv2d (models/quantized_conv.py:38)
        return self._conv_forward(input, self.weight, self.bias)

    def forward_folded(self, input, ep_a, ep_b, residual=None, act=0):
        """Inference forward with a per-out-channel affine (an eval-mode BatchNorm folded in), the residual add
        and the activation in the conv kernel's epilogue: act(conv(input) * ep_a + ep_b + residual).  Returns
        None when this layer / call cannot take the folded path (the caller then runs conv and norm separately):
        autograd active, a configuration the kernels do not take, a QAT layer without a prefetched operand."""
        if torch.is_grad_enabled() and (input.requires_grad or self.weight.requires_grad):
            return None
        mode = ops.get_conv_mode()
        if mode == "cudnn" or self._why_not(input) != "":
            return None
        if input.dtype == torch.bfloat16:
            family = self._bf16_layer(input)
            return self._bf16_forward(input, family, (ep_a, ep_b, residual, act)) if family is not None else None
        compute = ops.COMPUTE[mode]
        K, _, R, S = self.weight.shape
        if self.quantize_fn is not None:
            if _quantizers.quantizer_family(self.quantize_fn) is None or mode not in ("tc", "tf32"):
                return None
            from . import prefetch
            slot = self.__dict__.get("_po2_prefetch")
            if not slot or slot.key != prefetch._layer_key(self, input.shape, mode):
                self.__dict__["_po2_xshape"] = tuple(input.shape)
                return None
            prefetch.wait_for_quantizer(input.device)
            return ops.conv2d_packed_ep(input, slot.packed, slot.scale, K, R, S, self.stride[0], self.padding[0], self.groups,
                                        compute, ep_a, ep_b, residual, int(act))
        tag = getattr(self, "_po2_ptq", None)
        if tag is None or tag[0] != self.weight._version:
            tag = self.__dict__.get("_po2_lin_ptq")
            if tag is None or tag[0] != self.weight._version or self._lin_why_not(input, tag[1], quantizes=False) != "":
                return None                                      # a full-precision layer: plain nn.Conv2d
            one = ops.lin_scale(input.device)
            packed = self._ptq_packed(input, tag[0], one, mode) if mode in ("tc", "tf32") else None
            if packed is not None:
                return ops.conv2d_packed_ep(input, packed, one, K, R, S, self.stride[0], self.padding[0], self.groups,
                                            compute, ep_a, ep_b, residual, int(act))
            return ops.conv2d_ep(input, self.weight.detach(), one, self.stride[0], self.padding[0], self.groups, compute,
                                 ep_a, ep_b, residual, int(act))
        if mode in ("tc", "tf32"):
            key = (tag[0], tuple(input.shape), input.device, mode)
            cache = self.__dict__.get("_po2_pack_cache")
            if cache is None or cache[0] != key:
                packed = ops.conv2d_pack(self.weight.detach(), tag[1], tuple(input.shape), self.stride[0],
                                         self.padding[0], self.groups, compute)
                cache = (key, packed)
                self.__dict__["_po2_pack_cache"] = cache
            if cache[1] is not None:
                return ops.conv2d_packed_ep(input, cache[1], tag[1], K, R, S, self.stride[0], self.padding[0], self.groups,
                                            compute, ep_a, ep_b, residual, int(act))
        return ops.conv2d_ep(input, self.weight.detach(), tag[1], self.stride[0], self.padding[0], self.groups, compute,
                             ep_a, ep_b, residual, int(act))

    def get_quantization_error(self):
        """models/quantized_conv.py:40-45: (sum((Q(w) - w)^2), numel); (0, numel) without a quantizer.

        For PO2 / PO2+ on CUDA the sum is the fused fp64 output of the quantizer kernel itself: either the
        value the multi-tensor prefetch already produced for the current weight version (no launch at
        all -- what the models' per-epoch error walkers, train.py:106, then read for all layers), or one
        launch of the single-tensor kernel.  The reference sums in fp32 with 12 ATen launches; the
        value returned here is the fp64 sum rounded once to fp32 (a detached 0-dim tensor)."""
        if self.quantize_fn is not None:
            plus = getattr(self.quantize_fn, "_PLUS", None)
            w = self.weight
            if plus is not None and w.is_cuda and w.dtype in ops._DT and w.numel() > 0:
                slot = self.__dict__.get("_po2_prefetch")
                if (slot and slot.sse is not None and slot.key is not None and slot.key[0] == w._version
                        and slot.key[3] == int(self.bits) and slot.key[4] == bool(plus)):
                    from . import prefetch
                    prefetch.wait_for_quantizer(w.device)
                    return slot.sse.to(torch.float32), w.numel()
                sse = ops.quantize_full(w.detach(), int(self.bits), 1, bool(plus))[4]
                return sse.to(torch.float32), w.numel()
            quantized_weight = self.quantize_fn.apply(self.weight, self.bits)
            return torch.sum((quantized_weight - self.weight) ** 2), self.weight.numel()
        return 0, self.weight.numel()


# quantizers.py imports QuantizedConv2d (quantize_model walks the layers): bound last, read at call time
from . import quantizers as _quantizers  # noqa: E402
