"""CPU-side checks of the boundary: the C-ABI library loads without a GPU and exports every symbol
include/po2_b200.h declares; argument errors are reported through return codes."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "po2_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(po2_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_all_exported_abi_v2():
    from po2_quantization_b200 import _lib
    lib = _lib.load()
    syms = _declared_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/po2_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == syms, "ctypes signatures out of sync with the header"
    assert lib.po2_abi_version() == 2
    assert lib.po2_workspace_bytes() >= 16


def test_argument_errors_are_return_codes():
    from po2_quantization_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(16)
    # no launch is attempted on an argument error, so this is safe without a GPU
    assert lib.po2_absmax(one, 0, 0, one, one, None) == -4          # PO2_E_SIZE
    assert lib.po2_absmax(one, 8, 7, one, one, None) == -1          # PO2_E_DTYPE
    assert lib.po2_absmax(None, 8, 0, one, one, None) == -3         # PO2_E_NULL
    assert lib.po2_absmax(one, 8, 0, one, None, None) == -8         # PO2_E_WORKSPACE
    assert lib.po2_quantize(one, one, None, None, None, one, 8, 0, 9, 1, 0, 0, None) == -2   # bits
    assert lib.po2_quantize(one, one, None, None, None, one, 8, 0, 4, 1, 2, 0, None) == -9   # mode
    assert lib.po2_quantize(one, one, None, None, None, one, 8, 0, 4, 1, 0, 5, None) == -7   # flavor
    assert b"bits" in lib.po2_error_string(-2)
    assert lib.po2_error_string(0) == b"success"


def test_argument_errors_of_the_gradient_norm_and_lin_entry_points():
    """wgrad / BatchNorm / lin / multi-tensor entry points: argument errors come back as PO2_E_* codes
    before any launch (so this runs without a GPU), and the planning queries answer on the host."""
    from po2_quantization_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(4096)
    conv = (8, 16, 32, 32, 16, 3, 3)
    assert lib.po2_conv2d_wgrad_workspace(*conv, 2, 1, 1, 0) == 0                      # stride 2: not taken
    assert lib.po2_conv2d_wgrad_workspace(*conv, 1, 1, 1, 0) > 0
    assert lib.po2_conv2d_wgrad(None, one, one, *conv, 1, 1, 1, 0, one, 0, None) == -3            # PO2_E_NULL
    assert lib.po2_conv2d_wgrad(one, one, one, *conv, 2, 1, 1, 0, one, 0, None) == -10            # PO2_E_UNSUPPORTED
    assert lib.po2_conv2d_wgrad(one, one, one, *conv, 1, 1, 1, 0, None, 0, None) == -8            # PO2_E_WORKSPACE
    assert lib.po2_bn_workspace_bytes(64) > 64 * 16 and lib.po2_bn_mailbox_bytes() > 1 << 20
    assert lib.po2_bn_stats(None, 8, 16, 64, one, one, 1 << 20, None, 0, 1, None) == -3
    assert lib.po2_bn_stats(one, 8, 16, 64, one, one, 16, None, 0, 1, None) == -8
    assert lib.po2_bn_apply(one, None, one, one, 1, None, None, None, None, None, None, None, 0.1, 1e-5, 7, 0,
                            None, None, 8, 16, 64, None) == -9                                      # unknown activation
    assert lib.po2_bn_bwd_reduce(one, None, one, one, one, one, one, one, one, None, None, 4, 8, 16, 64, one, 1 << 20, None, 0,
                                 1, None) == -9                                                       # unknown activation
    assert lib.po2_bn_bwd_apply(one, None, one, None, one, one, one, one, one, one, 1, None, one, one, 3, 8, 16, 64,
                                None) == -9                                          # SiLU behind a residual add: not here
    assert lib.po2_lin_quantize(one, one, 4096, 4, 9, 4, 10, 0, 0, None) == -10                      # channel too large
    assert lib.po2_lin_quantize(one, one, 16, 4, 9, 1, 10, 0, 0, None) == -2                         # bits
    assert lib.po2_multi_desc_bytes() >= 64
    assert lib.po2_quantize_pack(one, one, one, one, 1 << 20, *conv, 1, 1, 1, 4, 1, 0, 0, 1, one, None) == -10


def test_cpu_tensors_are_rejected_not_emulated():
    import torch
    import po2_quantization_b200 as P
    with pytest.raises(Exception) as ei:
        P.PowerOfTwoQuantizer.forward(None, torch.randn(8), bits=4)
    assert "no CPU fallback" in str(ei.value)
    with pytest.raises(Exception):
        P.PowerOfTwoPlusQuantizer.apply(torch.randn(8), 4)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "po2_quantization_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b|['\"]oracle/|oracle\.po2_oracle", txt, flags=re.M), f
