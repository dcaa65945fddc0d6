"""Packed-code checkpoints (SURVEY.md section 8f "next" #4).

The reference only ever stores fp32 ``state_dict``s (train.py:118-120; test.py:50-55 strips the DDP
``module.`` prefix).  A PO2 / PO2+ quantized conv weight carries ``bits`` bits of information per
element -- sign + exponent level -- plus ONE fp32 scale per tensor, so a deployment checkpoint needs
1/8 (4-bit) or 1/4 (8-bit) of the fp32 bytes for those tensors:

    packed = pack_state_dict(model)             # QuantizedConv2d weights -> codes + scale, the rest as is
    torch.save(packed, path)                    # or save_packed_checkpoint(model, path)
    state = load_packed_checkpoint(path)        # fp32 state_dict again, on the CUDA device
    model.load_state_dict(state, strict=True)

Round trip: for a post-training-quantized model (``quantize_model``) the unpacked ``state_dict`` is
BIT-IDENTICAL to the original; for a QAT model (fp32 master weights + ``quantize_fn``) the unpacked
weights are exactly ``Q(weight)``, i.e. what every forward of that model convolves with and what
``quantize_model`` would have written.  Codes come from the sm_100a quantizer kernel
(``po2::quantize_full``: byte-for-byte the oracle's ``pack_codes(exponent_codes())``) and are decoded
by ``po2::dequantize``; tensors the code format cannot represent exactly are stored as fp32, never
approximated:
  * exact zeros have no code (the reference's sign(0) is 0): their positions travel as a bitmask;
  * a tensor for which ``dequantize(codes) != Q(weight)`` bit for bit (non-finite scale, products that
    underflow at 8 bits) is kept raw and counted in ``meta["raw_fallbacks"]``.
Keys, order and the ``module.`` prefix of the original ``state_dict`` are preserved.
"""
from typing import Dict, Optional

import torch

from . import ops
from .quantized_conv import QuantizedConv2d
from .quantizers import quantizer_family

FORMAT = "po2-packed-v1"


def _qconv_weight_names(model: torch.nn.Module) -> Dict[str, QuantizedConv2d]:
    return {(name + "." if name else "") + "weight": m for name, m in model.named_modules() if isinstance(m, QuantizedConv2d)}


def _layer_quantizer(m: QuantizedConv2d, quantizer, bits):
    """(bits, plus) this layer's weight is quantized with, or None if it is a full-precision layer"""
    # lin / lin+ weights have no PO2 codes: stored as fp32 (their PTQ tag is _po2_lin_ptq, not read here)
    if quantizer is not None:
        fam = quantizer_family(quantizer)
        return (int(bits), fam[1]) if fam is not None and fam[0] == "po2" else None
    if m.quantize_fn is not None:
        fam = quantizer_family(m.quantize_fn)
        return (int(m.bits), fam[1]) if fam is not None and fam[0] == "po2" else None
    tag = m.__dict__.get("_po2_ptq")
    if tag is not None and tag[0] == m.weight._version and len(tag) >= 4:
        return int(tag[2]), bool(tag[3])
    return None


def pack_state_dict(model: torch.nn.Module, quantizer=None, bits: Optional[int] = None) -> dict:
    """``model.state_dict()`` with every PO2/PO2+ ``QuantizedConv2d`` weight replaced by its packed
    sign+exponent codes and scale.  The quantizer of a layer is, in this order: the (quantizer, bits)
    given here; the layer's own ``quantize_fn`` / ``bits`` (QAT); what ``quantize_model`` recorded (PTQ).
    Layers without any (full precision, lin / lin+) are stored as fp32."""
    if quantizer is not None and bits is None:
        raise ValueError("pack_state_dict: bits is required with an explicit quantizer")
    sd = model.state_dict()
    names = _qconv_weight_names(model)
    tensors, packed, raw_fallbacks, fp32_bytes, packed_bytes = {}, {}, [], 0, 0
    for key, t in sd.items():
        m = names.get(key)
        q = _layer_quantizer(m, quantizer, bits) if m is not None else None
        if q is None or not t.is_cuda or t.dtype not in ops._DT or t.numel() == 0:
            tensors[key] = t.detach().cpu()
            continue
        nbits, plus = q
        w = t.detach().contiguous()
        y, codes, scale, zero_count, _ = ops.quantize_full(w, nbits, 1, plus)
        back = ops.dequantize(codes, scale, w.numel(), nbits, 1, w.dtype).view_as(w)
        entry = {"shape": tuple(w.shape), "dtype": str(w.dtype).split(".")[-1], "bits": nbits, "fsr": 1, "plus": plus,
                 "codes": codes.cpu(), "scale": scale.cpu()}
        if int(zero_count.item()) > 0:
            zero = (y == 0)
            back = torch.where(zero, torch.zeros_like(back), back)
            zb = zero.flatten().to(torch.uint8)
            pad = (-zb.numel()) % 8
            if pad:
                zb = torch.cat([zb, zb.new_zeros(pad)])
            entry["zero_mask"] = (zb.view(-1, 8) << torch.arange(8, device=zb.device, dtype=torch.uint8)).sum(1).to(torch.uint8).cpu()
        if not torch.equal(back.view(torch.int32 if w.dtype == torch.float32 else torch.int16),
                           y.view(torch.int32 if w.dtype == torch.float32 else torch.int16)):
            tensors[key] = y.cpu()                          # never approximate: keep Q(w) as fp32
            raw_fallbacks.append(key)
            continue
        packed[key] = entry
        fp32_bytes += w.numel() * w.element_size()
        packed_bytes += entry["codes"].numel() + 4 + (entry["zero_mask"].numel() if "zero_mask" in entry else 0)
    return {"format": FORMAT, "order": list(sd.keys()), "tensors": tensors, "packed": packed,
            "meta": {"raw_fallbacks": raw_fallbacks, "quantized_fp32_bytes": fp32_bytes, "quantized_packed_bytes": packed_bytes}}


def unpack_state_dict(packed: dict, device="cuda") -> "dict[str, torch.Tensor]":
    """the fp32 ``state_dict`` back (packed tensors are decoded on ``device`` by the dequantize kernel)"""
    if not isinstance(packed, dict) or packed.get("format") != FORMAT:
        raise ValueError(f"not a {FORMAT} checkpoint")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError("unpack_state_dict: codes are decoded by the sm_100a dequantize kernel (CUDA device required)")
    out = {}
    for key in packed["order"]:
        if key in packed["tensors"]:
            out[key] = packed["tensors"][key].to(dev)
            continue
        e = packed["packed"][key]
        dtype = getattr(torch, e["dtype"])
        n = 1
        for d in e["shape"]:
            n *= d
        w = ops.dequantize(e["codes"].to(dev), e["scale"].to(dev), n, e["bits"], e["fsr"], dtype)
        if "zero_mask" in e:
            zb = e["zero_mask"].to(dev)
            zero = ((zb.view(-1, 1) >> torch.arange(8, device=dev, dtype=torch.uint8)) & 1).flatten()[:n].bool()
            w = torch.where(zero, torch.zeros_like(w), w)
        out[key] = w.view(e["shape"])
    return out


def save_packed_checkpoint(model: torch.nn.Module, path: str, quantizer=None, bits: Optional[int] = None) -> dict:
    """torch.save(pack_state_dict(model, quantizer, bits), path); returns the size accounting"""
    packed = pack_state_dict(model, quantizer, bits)
    torch.save(packed, path)
    return packed["meta"]


def load_packed_checkpoint(path: str, device="cuda") -> "dict[str, torch.Tensor]":
    return unpack_state_dict(torch.load(path, map_location="cpu", weights_only=False), device)
