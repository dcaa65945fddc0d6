"""The bf16 lin / lin+ quantizer's C ABI, checked on the host: po2_lin_quantize_dt reports its argument errors before any
launch (so this runs without a GPU), the same ones po2_lin_quantize reports, and refuses every storage type but fp32
and bf16."""
import ctypes

import pytest

from po2_quantization_b200 import _lib

PO2_E_DTYPE, PO2_E_BITS, PO2_E_NULL, PO2_E_SIZE, PO2_E_FLAVOR, PO2_E_UNSUPPORTED = -1, -2, -3, -4, -7, -10


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _dt(lib, w, y, K, C, RS, bits, iters, plus, flavor, dtype):
    return lib.po2_lin_quantize_dt(w, y, K, C, RS, bits, iters, plus, flavor, dtype, None)


def test_abi_version_is_unchanged(lib):
    assert lib.po2_abi_version() == 2


@pytest.mark.parametrize("dtype", [_lib.F32, _lib.BF16])
def test_null_pointers(lib, dtype):
    one = ctypes.c_void_p(4096)
    assert _dt(lib, None, one, 16, 4, 9, 4, 10, 0, 0, dtype) == PO2_E_NULL
    assert _dt(lib, one, None, 16, 4, 9, 4, 10, 0, 0, dtype) == PO2_E_NULL


def test_only_fp32_and_bf16_are_taken(lib):
    one = ctypes.c_void_p(4096)
    assert _dt(lib, one, one, 16, 4, 9, 4, 10, 0, 0, _lib.F16) == PO2_E_DTYPE          # fp16 keeps the op-by-op form
    for unknown in (3, -1, 7):
        assert _dt(lib, one, one, 16, 4, 9, 4, 10, 0, 0, unknown) == PO2_E_DTYPE


@pytest.mark.parametrize("dtype", [_lib.F32, _lib.BF16])
def test_argument_errors_are_those_of_po2_lin_quantize(lib, dtype):
    one = ctypes.c_void_p(4096)
    cap = lib.po2_lin_max_channel_elems()
    cases = [
        ((cap // 9 + 1, 4, 9, 4, 10, 0, 0), PO2_E_UNSUPPORTED),          # a channel above the shared-memory capacity
        ((16, 4, 9, 1, 10, 0, 0), PO2_E_BITS),
        ((16, 4, 9, 17, 10, 0, 0), PO2_E_BITS),
        ((16, 4, 9, 4, -1, 0, 0), PO2_E_BITS),                            # num_iters < 0
        ((0, 4, 9, 4, 10, 0, 0), PO2_E_SIZE),
        ((16, 0, 9, 4, 10, 0, 0), PO2_E_SIZE),
        ((16, 4, -9, 4, 10, 0, 0), PO2_E_SIZE),
        ((1 << 16, 1 << 12, 9, 4, 10, 0, 0), PO2_E_SIZE),                # >= 2^31 elements
        ((16, 4, 9, 4, 10, 0, 2), PO2_E_FLAVOR),
        ((16, 4, 9, 4, 10, 0, -1), PO2_E_FLAVOR),
    ]
    for args, want in cases:
        assert lib.po2_lin_quantize(one, one, *args, None) == want, args
        assert _dt(lib, one, one, *args, dtype) == want, args
    # the errors come before the dtype check only for null pointers
    assert _dt(lib, None, one, 0, 4, 9, 4, 10, 0, 0, _lib.F16) == PO2_E_NULL
    assert _dt(lib, one, one, 0, 4, 9, 4, 10, 0, 0, _lib.F16) == PO2_E_DTYPE
