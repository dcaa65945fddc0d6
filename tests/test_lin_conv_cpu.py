"""lin / lin+ layers on the conv kernels, the parts that need no GPU: argument errors of the lin quantize+pack entry
points come back as PO2_E_* codes before any launch, CPU lin layers keep the op-by-op quantizer plus nn.Conv2d, and
the quantizer-family helper and the lin PTQ tag behave as the host code relies on."""
import copy
import ctypes

import pytest
import torch
import torch.nn.functional as F

import po2_quantization_b200 as P
from po2_quantization_b200 import _lib
from po2_quantization_b200.quantizers import quantizer_family

E_BITS, E_NULL, E_SIZE, E_SHAPE, E_FLAVOR, E_WORKSPACE, E_UNSUPPORTED = -2, -3, -4, -6, -7, -8, -10
CONV = (128, 16, 32, 32, 16, 3, 3, 1, 1, 1)          # B, C, H, W, K, R, S, stride, pad, groups: ResNet 16->16 3x3


def _pack(lib, *, w=16, y=16, packed=16, pbytes=1 << 20, dgrad=None, dbytes=0, conv=CONV, bits=4, iters=10, plus=0,
          flavor=0, compute=2):
    p = ctypes.c_void_p
    return lib.po2_lin_quantize_pack(p(w) if w else None, p(y) if y else None, p(packed) if packed else None, pbytes,
                                     p(dgrad) if dgrad else None, dbytes, *conv, bits, iters, plus, flavor, compute, None)


def _fill(lib, table, index=0, *, packed=16, pbytes=1 << 20, conv=CONV, bits=4, iters=10, compute=2):
    p = ctypes.c_void_p
    return lib.po2_lin_multi_desc_fill(table, index, p(16), p(16), p(packed) if packed else None, pbytes, None, 0, *conv,
                                       bits, iters, 0, 0, compute)


def test_lin_quantize_pack_argument_errors_are_return_codes():
    lib = _lib.load()
    assert _pack(lib, w=0) == E_NULL
    assert _pack(lib, packed=0) == E_NULL
    assert _pack(lib, bits=1) == E_BITS
    assert _pack(lib, bits=17) == E_BITS
    assert _pack(lib, iters=-1) == E_BITS
    assert _pack(lib, flavor=9) == E_FLAVOR
    assert _pack(lib, pbytes=16) == E_WORKSPACE
    assert _pack(lib, conv=(128, 16, 32, 32, 16, 3, 3, 1, 1, 0)) == E_SIZE                 # groups 0
    assert _pack(lib, conv=(128, 16, 32, 32, 16, 3, 3, 1, 1, 3)) == E_SHAPE                # 16 channels in 3 groups
    # no tensor-core operand: the fp32 mode, a depthwise layer, a channel above the kernel's capacity
    assert _pack(lib, compute=1) == E_UNSUPPORTED
    assert _pack(lib, conv=(128, 32, 16, 16, 32, 3, 3, 1, 1, 32)) == E_UNSUPPORTED
    big = lib.po2_lin_max_channel_elems() // 9 + 16
    assert _pack(lib, conv=(8, 16, 8, 8, big, 3, 3, 1, 1, 1)) == E_UNSUPPORTED
    # the operand would not be exact, or the step not a power of two
    assert _pack(lib, bits=13, compute=2) == E_UNSUPPORTED
    assert _pack(lib, bits=10, compute=0) == E_UNSUPPORTED
    assert _pack(lib, iters=0) == E_UNSUPPORTED
    # the data-gradient operand exists for stride-1 dense layers only
    assert _pack(lib, dgrad=16, dbytes=1 << 20, conv=(128, 16, 32, 32, 32, 3, 3, 2, 1, 1)) == E_UNSUPPORTED
    assert _pack(lib, dgrad=16, dbytes=16) == E_WORKSPACE


def test_lin_multi_desc_fill_and_launch_argument_errors():
    lib = _lib.load()
    dbytes = lib.po2_lin_multi_desc_bytes()
    assert dbytes >= 64
    table = (ctypes.c_uint8 * (4 * dbytes))()
    assert _fill(lib, None) == E_NULL
    assert _fill(lib, table, packed=0) == E_NULL
    assert _fill(lib, table, bits=13) == E_UNSUPPORTED
    assert _fill(lib, table, compute=1) == E_UNSUPPORTED
    assert _fill(lib, table, conv=(4, 48, 14, 9, 40, 3, 3, 1, 1, 1)) == E_UNSUPPORTED      # operand needs padding
    # filled in order, the return value is the tensor's CTA count (one per input channel)
    assert _fill(lib, table, 0) == 16
    assert _fill(lib, table, 1, conv=(128, 16, 32, 32, 32, 3, 3, 2, 1, 1)) == 16
    assert _fill(lib, table, 2, conv=(128, 32, 16, 16, 32, 3, 3, 1, 1, 1)) == 32
    assert lib.po2_lin_quantize_pack_multi(None, 3, 64, 288, None) == E_NULL
    assert lib.po2_lin_quantize_pack_multi(ctypes.c_void_p(16), -1, 64, 288, None) == E_SIZE
    assert lib.po2_lin_quantize_pack_multi(ctypes.c_void_p(16), 3, 64, 0, None) == E_UNSUPPORTED
    assert lib.po2_lin_quantize_pack_multi(ctypes.c_void_p(16), 3, 64, lib.po2_lin_max_channel_elems() + 1,
                                           None) == E_UNSUPPORTED
    assert lib.po2_lin_quantize_pack_multi(ctypes.c_void_p(16), 0, 0, 288, None) == 0      # nothing to do: no launch


def test_quantizer_family_helper():
    assert quantizer_family(P.PowerOfTwoQuantizer) == ("po2", False)
    assert quantizer_family(P.PowerOfTwoPlusQuantizer) == ("po2", True)
    assert quantizer_family(P.LinearPowerOfTwoQuantizer) == ("lin", False)
    assert quantizer_family(P.LinearPowerOfTwoPlusQuantizer) == ("lin", True)
    assert quantizer_family(None) is None
    assert quantizer_family(torch.autograd.Function) is None
    for name, q in P.quantizer_dict.items():
        assert quantizer_family(q) is not None, name
    # the PO2-code readers (checkpoint, prefetch) take _PLUS to mean a PO2 grid: the lin classes must not carry it
    assert not hasattr(P.LinearPowerOfTwoQuantizer, "_PLUS")
    assert not hasattr(P.LinearPowerOfTwoPlusQuantizer, "_PLUS")


def test_cpu_lin_layers_run_op_by_op_and_nn_conv2d(recwarn):
    torch.manual_seed(0)
    x = torch.randn(2, 16, 8, 8)
    for q, plus in ((P.LinearPowerOfTwoQuantizer, False), (P.LinearPowerOfTwoPlusQuantizer, True)):
        for bits in (2, 4, 8):
            conv = P.QuantizedConv2d(16, 32, 3, quantize_fn=q, bits=bits)
            y = P.quantizers._lin_forward(conv.weight.detach(), bits, 10, plus)
            out = conv(x)
            assert torch.equal(out, F.conv2d(x, y, None, 1, 1))
    assert not [w for w in recwarn if "qconv:" in str(w.message) or "nn.Conv2d's own" in str(w.message)]


def test_lin_ptq_tag_is_rekeyed_by_deepcopy_and_not_read_as_po2_codes():
    from po2_quantization_b200 import checkpoint
    conv = P.QuantizedConv2d(16, 32, 3)
    with torch.no_grad():
        conv.weight.add_(1.0)                                  # version > 0, like quantize_model's copy_
    conv._po2_lin_ptq = (conv.weight._version, 4, True)
    dup = copy.deepcopy(conv)
    assert dup._po2_lin_ptq == (dup.weight._version, 4, True)
    # a stale tag is not carried over as current
    with torch.no_grad():
        conv.weight.add_(1.0)
    dup2 = copy.deepcopy(conv)
    assert dup2.__dict__.get("_po2_lin_ptq", (None,))[0] != dup2.weight._version
    # the checkpoint writer sees no PO2 quantizer for lin layers (they stay fp32)
    assert checkpoint._layer_quantizer(dup, None, None) is None
    assert checkpoint._layer_quantizer(dup, P.LinearPowerOfTwoPlusQuantizer, 4) is None
    lin_qat = P.QuantizedConv2d(16, 32, 3, quantize_fn=P.LinearPowerOfTwoQuantizer, bits=4)
    assert checkpoint._layer_quantizer(lin_qat, None, None) is None
    po2_qat = P.QuantizedConv2d(16, 32, 3, quantize_fn=P.PowerOfTwoPlusQuantizer, bits=4)
    assert checkpoint._layer_quantizer(po2_qat, None, None) == (4, True)


def test_quantize_model_on_cpu_sets_no_lin_tag():
    torch.manual_seed(0)
    model = torch.nn.Sequential(P.QuantizedConv2d(16, 32, 3), P.QuantizedConv2d(32, 32, 3))
    ref = copy.deepcopy(model)
    mse = P.quantize_model(model, P.LinearPowerOfTwoPlusQuantizer, 4)
    total, n = 0.0, 0
    for m, r in zip(model, ref):
        y = P.quantizers._lin_forward(r.weight.detach(), 4, 10, True)
        assert torch.equal(m.weight.detach(), y)
        total += torch.sum((y - r.weight.detach()) ** 2).double()
        n += y.numel()
        assert "_po2_lin_ptq" not in m.__dict__                # CPU weights: the stock conv, as before
    assert mse == float((total / n).item())
