"""po2_dilate2_into, the zero-insertion of the output gradient of a stride-2 layer of any size: its argument checks
answer before any launch, so they run without a device.  po2_dilate2, the even-size form, keeps refusing an odd
output width."""
import ctypes

import pytest

from po2_quantization_b200 import _lib

PO2_E_NULL, PO2_E_SIZE, PO2_E_SHAPE, PO2_E_UNSUPPORTED = -3, -4, -6, -10
ONE = ctypes.c_void_p(4096)
ODD = ctypes.c_void_p(4100)          # 4-byte aligned only


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def test_null_pointers(lib):
    assert lib.po2_dilate2_into(None, ONE, 4, 4, 4, 7, 7, None) == PO2_E_NULL
    assert lib.po2_dilate2_into(ONE, None, 4, 4, 4, 7, 7, None) == PO2_E_NULL


@pytest.mark.parametrize("P, Q, H, W", [(3, 4, 7, 7), (5, 4, 7, 7), (4, 3, 7, 7), (4, 5, 7, 7), (7, 7, 7, 7),
                                        (1, 2, 1, 1), (2, 1, 1, 1), (2, 2, 2, 2), (7, 8, 14, 14), (8, 7, 14, 14)])
def test_mismatched_sizes(lib, P, Q, H, W):
    """P must be (H - 1) // 2 + 1 and Q (W - 1) // 2 + 1, each on its own"""
    assert lib.po2_dilate2_into(ONE, ONE, 4, P, Q, H, W, None) == PO2_E_SHAPE


@pytest.mark.parametrize("planes, P, Q, H, W", [(0, 4, 4, 7, 7), (-1, 4, 4, 7, 7), (4, 0, 4, 0, 7), (4, 4, 0, 7, 0),
                                                (4, 1, 4, -1, 7), (4, 4, 1, 7, -1), (4, -1, 4, -3, 7)])
def test_non_positive_sizes(lib, planes, P, Q, H, W):
    assert lib.po2_dilate2_into(ONE, ONE, planes, P, Q, H, W, None) == PO2_E_SHAPE


def test_index_range(lib):
    """g_up has planes * H * W elements, indexed in 32 bits: refused from 2^31"""
    assert lib.po2_dilate2_into(ONE, ONE, 1 << 17, 64, 64, 128, 128, None) == PO2_E_SIZE                  # 2^31 exactly
    assert lib.po2_dilate2_into(ONE, ONE, 1, 23171, 23171, 46341, 46341, None) == PO2_E_SIZE              # odd, 2^31 + 4633
    assert lib.po2_dilate2_into(ONE, ONE, 4, 1 << 15, 1 << 15, 1 << 16, 1 << 16, None) == PO2_E_SIZE      # 2^34: 0 in 32 bits
    assert lib.po2_dilate2_into(ODD, ODD, 6, 12289, 8193, 24577, 16385, None) == PO2_E_SIZE               # any alignment


def test_dilate2_still_refuses_an_odd_width(lib):
    assert lib.po2_dilate2(ONE, ONE, 4, 8, 7, None) == PO2_E_UNSUPPORTED
    assert lib.po2_dilate2(ONE, ONE, 4, 1, 1, None) == PO2_E_UNSUPPORTED
    assert lib.po2_dilate2(ODD, ONE, 4, 8, 8, None) == PO2_E_UNSUPPORTED         # g 8-byte aligned
    assert lib.po2_dilate2(ONE, ctypes.c_void_p(4104), 4, 8, 8, None) == PO2_E_UNSUPPORTED   # g_up 16-byte aligned
