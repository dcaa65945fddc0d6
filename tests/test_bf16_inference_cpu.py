"""bf16 inference on the forward conv kernels, checked on the host: which kernel the planner picks for a bf16 x
(po2_conv2d_kernel_kind_dt answers without a device), which K3 producer branch it reaches, what it refuses, and that an
x the bf16 producers read with 128-bit loads must start on a 16-byte boundary (PO2_E_ALIGN before any launch)."""
import ctypes

import pytest

from po2_quantization_b200 import _lib
from tests.test_conv_exact_cpu import FWD, k3_branches, k3_plan

PO2_E_DTYPE = -1
PO2_E_ALIGN = -5
PO2_E_UNSUPPORTED = -10


def bf16_kind(kind, compute):
    """the kernel a bf16 x runs on where an fp32 x runs on `kind`: K3 (bf16 operands) for K3 and K3T, the same
    depthwise / small-pointwise kernel, and nothing on the fp32 CUDA cores (compute 1) or the direct kernel"""
    if compute == 1 or kind == 0:
        return PO2_E_UNSUPPORTED
    return 2 if kind in (2, 3) else kind


def bf16_branches(B, C, H, W, K, k, stride):
    """k3_branches for a bf16 x: the 128-bit producer loads carry 8 pixels (vec4: W % 8 == 0) or 8 channels (hw1:
    C % 8 == 0)"""
    plan = k3_plan(B, C, H, W, K, k, stride, 0)
    Wf = H * W if (k == 1 and stride == 1) else W
    plan["vec4"] = stride == 1 and Wf % 8 == 0
    plan["hw1"] = H * W == 1 and C % 8 == 0
    return k3_branches(plan, C, K), plan


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _args(case):
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    return (B, C, H, W, K, k, k, stride, k // 2, groups)


@pytest.mark.parametrize("case", FWD, ids=lambda c: c[0])
def test_bf16_kernel_kind_of_each_forward_case(lib, case):
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    want = bf16_kind(kind, compute)
    assert lib.po2_conv2d_kernel_kind_dt(*_args(case), compute, _lib.BF16) == want, name
    # the fp32 answer of the dtype form is the plain query's
    assert lib.po2_conv2d_kernel_kind_dt(*_args(case), compute, _lib.F32) == lib.po2_conv2d_kernel_kind(*_args(case),
                                                                                                        compute)
    ws = lib.po2_conv2d_workspace_dt(*_args(case), compute, _lib.BF16)
    assert (ws == 0) == (want < 0), name
    if want == 2:
        got, plan = bf16_branches(B, C, H, W, K, k, stride)
        # the bf16-operand packed layout, whatever the compute mode
        assert lib.po2_conv2d_pack_bytes_dt(*_args(case), compute, _lib.BF16) == -(-plan["pack_bytes"] // 256) * 256
        assert lib.po2_conv2d_pack_bytes_dt(*_args(case), compute, _lib.BF16) == lib.po2_conv2d_pack_bytes(*_args(case), 0)
    else:
        assert lib.po2_conv2d_pack_bytes_dt(*_args(case), compute, _lib.BF16) == 0, name


@pytest.mark.parametrize("compute", [0, 2])
def test_bf16_reaches_every_k3_producer_branch(lib, compute):
    """the bf16 producer branches the GPU tests cover: 8-pixel vec path, scalar (W % 8 != 0), hw1, 4-phase stride 2,
    and the flattened 1x1 map"""
    cases = {"vec4": (4, 16, 16, 16, 16, 3, 1), "scalar": (4, 16, 12, 12, 16, 3, 1), "hw1": (16, 32, 1, 1, 32, 3, 1),
             "s2": (4, 16, 16, 16, 32, 3, 2), "flat": (4, 32, 6, 6, 48, 1, 1)}
    for branch, (B, C, H, W, K, k, stride) in cases.items():
        assert lib.po2_conv2d_kernel_kind_dt(B, C, H, W, K, k, k, stride, k // 2, 1, compute, _lib.BF16) == 2
        assert branch in bf16_branches(B, C, H, W, K, k, stride)[0], branch
    # 1x1 on 6x6 flattens to 36 pixels: 4-pixel items for fp32, scalar for bf16
    assert "vec4" not in bf16_branches(4, 32, 6, 6, 48, 1, 1)[0]


def test_bf16_refusals(lib):
    geo = (4, 16, 16, 16, 16, 3, 3, 1, 1, 1)
    assert lib.po2_conv2d_kernel_kind_dt(*geo, 1, _lib.BF16) == PO2_E_UNSUPPORTED          # fp32 CUDA cores
    assert lib.po2_conv2d_kernel_kind_dt(2, 16, 8, 8, 32, 3, 3, 1, 1, 4, 0, _lib.BF16) == PO2_E_UNSUPPORTED  # grouped
    assert lib.po2_conv2d_kernel_kind_dt(2, 8, 12, 12, 8, 5, 5, 1, 2, 1, 2, _lib.BF16) == PO2_E_UNSUPPORTED  # 5x5
    assert lib.po2_conv2d_kernel_kind_dt(*geo, 0, _lib.F16) == PO2_E_DTYPE
    ok, big = ctypes.c_void_p(0x1000), 1 << 30
    assert lib.po2_conv2d_fwd_ep_dt(ok, ok, ok, ok, *geo, 0, 4, 1, 1, ok, big, None, None, None, 0, _lib.BF16,
                                    None) == PO2_E_UNSUPPORTED
    assert lib.po2_conv2d_pack_dt(ok, ok, ok, big, *geo, 0, 4, 1, 1, _lib.BF16, None) == PO2_E_UNSUPPORTED


def test_bf16_x_8_bytes_off_is_refused_before_any_launch(lib):
    """bf16 x at 0x1008: 8-byte aligned, 16-byte misaligned.  Where the bf16 producers read 8 pixels (stride 1,
    W % 8 == 0) or 8 channels (1x1 map, C % 8 == 0) with one 128-bit load, every forward entry point refuses it."""
    ok, bad = ctypes.c_void_p(0x1000), ctypes.c_void_p(0x1008)
    big = 1 << 30
    # 3x3 stride 1 at W 16, 1x1 on an 8x8 map (64 pixels in one row), 3x3 on a 1x1 map with 32 channels
    for geo in ((4, 16, 16, 16, 16, 3, 3, 1, 1, 1), (4, 32, 8, 8, 48, 1, 1, 1, 0, 1), (16, 32, 1, 1, 32, 3, 3, 1, 1, 1)):
        for compute in (0, 2):
            assert lib.po2_conv2d_kernel_kind_dt(*geo, compute, _lib.BF16) == 2, geo
            assert lib.po2_conv2d_fwd_ep_dt(bad, ok, ok, ok, *geo, 0, 4, 1, compute, ok, big, None, None, None, 0,
                                            _lib.BF16, None) == PO2_E_ALIGN, geo
            assert lib.po2_conv2d_fwd_ep_dt(bad, ok, ok, ok, *geo, 0, 4, 1, compute, ok, big, ok, ok, ok, 1, _lib.BF16,
                                            None) == PO2_E_ALIGN, geo
            assert lib.po2_conv2d_fwd_packed_ep_dt(bad, ok, ok, ok, *geo, compute, None, None, None, 0, _lib.BF16,
                                                   None) == PO2_E_ALIGN, geo
            assert lib.po2_conv2d_fwd_packed_ep_dt(bad, ok, ok, ok, *geo, compute, ok, ok, ok, 2, _lib.BF16,
                                                   None) == PO2_E_ALIGN, geo
