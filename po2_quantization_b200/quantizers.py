"""Host-side mirror of the reference's ``utils/quantizers.py`` public surface.

Same names, signatures and call protocols (``Q.apply(t, bits)``, ``Q.forward(None, t, bits=b)``,
``quantize_model``, ``quantizer_dict``) -- SURVEY.md section 8b -- but PO2 / PO2+ run as
hand-written sm_100a kernels through the C ABI (``po2::quantize``).  CUDA tensors only: there is
no CPU fallback on this path.
"""
from typing import Callable, Optional

import os

import torch

from . import ops
from .quantized_conv import QuantizedConv2d


class _Po2Base(torch.autograd.Function):
    """Shared shell of the two quantizer classes; ``_PLUS`` selects the rounding rule."""
    _PLUS = False

    @classmethod
    def _run(cls, input: torch.Tensor, bits: int, fsr: int) -> torch.Tensor:
        ops._require_cuda(input, cls.__name__)
        return ops.quantize(input, int(bits), int(fsr), cls._PLUS)


class PowerOfTwoQuantizer(_Po2Base):
    """2^round(log2|x/s|), s = max|x|, clamped to ``bits`` -- reference utils/quantizers.py:19-36."""
    _PLUS = False

    @staticmethod
    def forward(ctx, input: torch.Tensor, bits: int = 4, fsr: int = 1):
        return PowerOfTwoQuantizer._run(input, bits, fsr)

    @staticmethod
    def backward(ctx, grad_output):
        # straight-through estimator, utils/quantizers.py:34-36: the same tensor object
        return grad_output, None, None


class PowerOfTwoPlusQuantizer(_Po2Base):
    """2^round(log2(|x/s|/1.5)+0.5) -- reference utils/quantizers.py:39-56."""
    _PLUS = True

    @staticmethod
    def forward(ctx, input: torch.Tensor, bits: int = 4, fsr: int = 1):
        return PowerOfTwoPlusQuantizer._run(input, bits, fsr)

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output, None, None


# ------------------------------------------------------------------------------------------------
# lin / lin+ (SURVEY.md section 8f "next" #1): per-input-channel uniform quantizer whose step is
# constrained to a power of two (utils/quantizers.py:8-16, 59-136).  CUDA fp32 or bf16 4-D weights take the
# single-launch kernel of csrc/po2_lin.cu (bf16: each op rounded to bf16, as the op-by-op form does on bf16 tensors);
# everything else the op-by-op form below.
# ------------------------------------------------------------------------------------------------
def _uniform_per_in_channel(w: torch.Tensor, step: torch.Tensor, bits: int) -> torch.Tensor:
    s = step.view(-1, 1, 1)
    lim = float(2 ** (bits - 1) - 1)
    return s * torch.clamp(torch.round(w / s), min=-lim, max=lim)


def _lin_forward_cuda(w: torch.Tensor, bits: int, num_iters: int, plus: bool):
    """one launch of csrc/po2_lin.cu (one CTA per input channel) for an fp32 or bf16 w, or None if the shape is not
    taken"""
    from . import _lib
    lib = _lib.load()
    K, C = w.shape[0], w.shape[1]
    RS = w.shape[2] * w.shape[3]
    if K * RS > lib.po2_lin_max_channel_elems() or not 2 <= bits <= 16:
        return None
    x = w.contiguous()
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = lib.po2_lin_quantize_dt(x.data_ptr(), y.data_ptr(), K, C, RS, int(bits), int(num_iters), int(plus),
                                     ops._flavor, ops._DT[x.dtype], ops._stream_ptr(x.device))
    if rc == -10:
        return None
    _lib.check(rc, "po2_lin_quantize_dt")
    ops.LAUNCHES += 1
    return y


def _lin_forward(w: torch.Tensor, bits: int, num_iters: int, plus: bool) -> torch.Tensor:
    kernel_dtype = w.dtype in (torch.float32, torch.bfloat16)
    if w.is_cuda and kernel_dtype and w.dim() == 4 and w.numel() > 0 and os.environ.get("PO2_LIN", "cuda") == "cuda":
        y = _lin_forward_cuda(w.detach(), bits, num_iters, plus)
        if y is not None:
            return y
        why = "a channel exceeds the kernel's shared-memory capacity or bits is outside 2..16"
    else:
        why = ("CPU tensor" if not w.is_cuda else f"dtype {w.dtype}" if not kernel_dtype else
               f"{w.dim()}-D tensor" if w.dim() != 4 else "empty tensor" if w.numel() == 0 else "PO2_LIN != cuda")
    # op-by-op ATen form in the reference's order (utils/quantizers.py:59-136) -- a library path, so it is
    # reported (once per reason; an error under PO2_STRICT=1).  lin / lin+ are SURVEY section 8f "next" rows:
    # unlike PO2 / PO2+ they keep this form for the inputs the kernel does not take.
    ops.note_library_path("lin:" + why, f"lin/lin+ quantizer runs as stock ATen ops: {why}")
    hi = torch.amax(w, dim=(0, 2, 3))
    lo = torch.amin(w, dim=(0, 2, 3))
    step = (hi - lo) / (2 ** bits - 1)
    q = _uniform_per_in_channel(w, step, bits) / step.view(-1, 1, 1)
    for _ in range(num_iters):
        step = torch.sum(q * w, dim=[0, 2, 3]) / torch.sum(q * q, dim=[0, 2, 3])
        if plus:
            step = torch.sqrt(torch.tensor(8.0 / 9.0)) * step
        step = 2 ** torch.round(torch.log2(step))
        q = _uniform_per_in_channel(w, step, bits) / step.view(-1, 1, 1)
    return q * step.view(-1, 1, 1)


class LinearPowerOfTwoQuantizer(torch.autograd.Function):
    """reference utils/quantizers.py:59-96"""
    # (family, plus): NOT _PLUS, which the PO2 code paths (checkpoint codes, prefetch) read as "PO2 grid"
    _FAMILY = ("lin", False)

    @staticmethod
    def forward(ctx, input: torch.Tensor, bits: int = 4, num_iters: int = 10):
        return _lin_forward(input, bits, num_iters, plus=False)

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output, None, None


class LinearPowerOfTwoPlusQuantizer(torch.autograd.Function):
    """reference utils/quantizers.py:99-136"""
    _FAMILY = ("lin", True)

    @staticmethod
    def forward(ctx, input: torch.Tensor, bits: int = 4, num_iters: int = 10):
        return _lin_forward(input, bits, num_iters, plus=True)

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output, None, None


def quantizer_family(quantizer):
    """("po2", plus) for PowerOfTwo[Plus]Quantizer, ("lin", plus) for LinearPowerOfTwo[Plus]Quantizer, None for
    anything else (no quantizer, or one this library has no kernel path for)"""
    fam = getattr(quantizer, "_FAMILY", None)
    if fam is not None:
        return fam
    plus = getattr(quantizer, "_PLUS", None)
    return None if plus is None else ("po2", bool(plus))


def quantize_model(model: torch.nn.Module, quantizer: Optional[Callable[..., None]], bits: int) -> float:
    """Post-training quantization in place -- reference utils/quantizers.py:139-153.

    Every parameter of every ``QuantizedConv2d`` is overwritten with its quantized value; returns
    the mean squared quantization error as a Python float.  For the PO2 quantizers the squared
    error comes out of the same kernel pass that quantizes (no extra reads of the weights)."""
    total = None
    numel = 0
    with torch.no_grad():
        for _, module in model.named_modules():
            if not isinstance(module, QuantizedConv2d):
                continue
            for _, param in module.named_parameters():
                scale = None
                if isinstance(quantizer, type) and issubclass(quantizer, _Po2Base) and param.is_cuda:
                    qp, _codes, scale, _zc, sse = ops.quantize_full(param, int(bits), 1, quantizer._PLUS)
                    err = sse
                else:
                    qp = quantizer.forward(None, param, bits=bits)
                    err = torch.sum((qp - param) ** 2).double()
                total = err if total is None else total + err
                numel += param.numel()
                param.copy_(qp)
                if scale is not None and param is module.weight:
                    # non-persistent tag (state_dict stays {weight}): the weight is now on the grid
                    # +-scale*2^q, which lets forward() feed the tensor-core conv an exact operand
                    module._po2_ptq = (param._version, scale, int(bits), bool(quantizer._PLUS))
                fam = quantizer_family(quantizer)
                if (fam is not None and fam[0] == "lin" and param is module.weight and param.is_cuda
                        and os.environ.get("PO2_LIN", "cuda") == "cuda"):
                    # lin / lin+: n * 2^k per input channel, its own exact operand (scale 1.0); a separate tag, since
                    # _po2_ptq means PO2 codes to the checkpoint writer
                    module._po2_lin_ptq = (param._version, int(bits), fam[1])
    if total is None:
        raise ZeroDivisionError("quantize_model: the model has no QuantizedConv2d parameters")
    return float((total / numel).item())


def model_quantization_error(model: torch.nn.Module):
    """(sum over all QuantizedConv2d layers of sum((Q(w) - w)^2), total numel) -- the quantity the
    reference's per-model walkers accumulate layer by layer (models/resnet.py:214-224, train.py:106),
    without their denominator quirks (SURVEY.md section 5).  With `enable_weight_prefetch` every layer's
    term is already on the device from the multi-tensor launch of the last forward; the terms are summed
    in fp64 by ONE stack+sum instead of one add per layer."""
    terms, numel = [], 0
    for m in model.modules():
        if isinstance(m, QuantizedConv2d):
            e, n = m.get_quantization_error()
            numel += n
            if torch.is_tensor(e):
                terms.append(e.double())
    if not terms:
        return 0, numel
    return torch.stack(terms).sum(), numel


quantizer_dict = {
    "lin": LinearPowerOfTwoQuantizer,
    "lin+": LinearPowerOfTwoPlusQuantizer,
    "po2": PowerOfTwoQuantizer,
    "po2+": PowerOfTwoPlusQuantizer,
}
