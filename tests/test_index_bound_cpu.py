"""The 2^31-element bound of the C ABI, checked on the host: the kernels index activations in 32 bits, so every entry
point refuses a tensor of 2^31 or more elements with PO2_E_SIZE before any launch, and the planning queries
(po2_conv2d_kernel_kind / _dt, po2_conv2d_dgrad_workspace, po2_conv2d_wgrad_kernel_kind) give the same answer as the
launch: a kernel just below the bound, a refusal at it.  The entry points without a query are only asked about sizes
they refuse, so nothing here launches a kernel."""
import ctypes

import pytest

from po2_quantization_b200 import _lib

PO2_E_SIZE = -4
ONE = ctypes.c_void_p(4096)          # never dereferenced: every call below is refused before a launch
BIG = 1 << 40                        # workspace bytes
TF32, BF16_OPS = 2, 0                # compute: tf32 operands (K3T / K5T), bf16 operands (K3 / K5)
F32, BF16 = 0, 1                     # PO2_F32, PO2_BF16

# 16->16 3x3 pad 1 at 32 x 32: x and the output have B * 2^14 elements
RESNET_UNDER = (131071, 16, 32, 32, 16, 3, 3)      # 2^31 - 2^14
RESNET_AT = (131072, 16, 32, 32, 16, 3, 3)         # 2^31
# 1x1 convs whose element counts sit exactly on the bound: x = B * C * H * W, out = B * K * H * W
PW_UNDER = (2**31 - 1, 1, 1, 1, 1, 1, 1)           # both 2^31 - 1
PW_AT = (2**30, 2, 1, 1, 2, 1, 1)                  # both 2^31
PW_OUT_AT = (2**30, 1, 1, 1, 2, 1, 1)              # x 2^30, out 2^31
PW_IN_AT = (2**30, 2, 1, 1, 1, 1, 1)               # x 2^31, out 2^30
# depthwise 576-channel 3x3 at 7 x 7 (the scalar depthwise kernel): 576 * 49 * B elements
DW_UNDER = (76087, 576, 7, 7, 576, 3, 3)           # 2^31 - 4160
DW_AT = (76088, 576, 7, 7, 576, 3, 3)              # 2^31 + 24064


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def kind(lib, shape, compute, groups=1, dtype=F32):
    B, C, H, W, K, R, S = shape
    return lib.po2_conv2d_kernel_kind_dt(B, C, H, W, K, R, S, 1, R // 2, groups, compute, dtype)


def test_shapes_sit_on_the_bound():
    def elems(shape):
        B, C, H, W, K, _, _ = shape
        return B * C * H * W, B * K * H * W
    assert elems(RESNET_UNDER) == (2**31 - 2**14,) * 2 and elems(RESNET_AT) == (2**31,) * 2
    assert elems(PW_UNDER) == (2**31 - 1,) * 2 and elems(PW_AT) == (2**31,) * 2
    assert elems(PW_OUT_AT) == (2**30, 2**31) and elems(PW_IN_AT) == (2**31, 2**30)
    assert elems(DW_UNDER) == (2**31 - 4160,) * 2 and elems(DW_AT)[0] > 2**31


# K3T and K5T need the driver's tensor maps: without a device, the tf32 plans fall back to K3 / K5
@pytest.mark.parametrize("compute, want", [(TF32, (2, 3)), (BF16_OPS, (2,))])
def test_forward_kind_tensor_core(lib, compute, want):
    """K3T (tf32) / K3 (bf16 operands) just below 2^31, PO2_E_SIZE at it -- in fp32 and for a bf16 x"""
    assert kind(lib, RESNET_UNDER, compute) in want
    assert kind(lib, RESNET_AT, compute) == PO2_E_SIZE
    assert kind(lib, RESNET_UNDER, compute, dtype=BF16) == 2
    assert kind(lib, RESNET_AT, compute, dtype=BF16) == PO2_E_SIZE
    B, C, H, W, K, R, S = RESNET_AT
    assert lib.po2_conv2d_kernel_kind(B, C, H, W, K, R, S, 1, 1, 1, compute) == PO2_E_SIZE
    assert lib.po2_conv2d_workspace_dt(B, C, H, W, K, R, S, 1, 1, 1, compute, F32) == 0


def test_forward_kind_at_exactly_two_to_the_31(lib):
    """2^31 - 1 elements run (K3; in fp32, the depthwise kernel, C = K = groups = 1); 2^31 in x, in the output or in
    both is refused"""
    for compute in (TF32, BF16_OPS, 1):
        assert kind(lib, PW_UNDER, compute) == (1 if compute == 1 else 2)
        for shape in (PW_AT, PW_OUT_AT, PW_IN_AT):
            assert kind(lib, shape, compute) == PO2_E_SIZE, (shape, compute)


def test_forward_kind_depthwise(lib):
    assert kind(lib, DW_UNDER, TF32, groups=576) == 1
    assert kind(lib, DW_UNDER, TF32, groups=576, dtype=BF16) == 1
    assert kind(lib, DW_AT, TF32, groups=576) == PO2_E_SIZE


@pytest.mark.parametrize("compute", [TF32, BF16_OPS])
def test_dgrad_workspace(lib, compute):
    """po2_conv2d_dgrad_workspace is 0 for exactly the shapes po2_conv2d_dgrad refuses"""
    B, C, H, W, K, R, S = RESNET_UNDER
    assert lib.po2_conv2d_dgrad_workspace(B, C, H, W, K, R, S, 1, compute) > 0
    B, C, H, W, K, R, S = RESNET_AT
    assert lib.po2_conv2d_dgrad_workspace(B, C, H, W, K, R, S, 1, compute) == 0
    assert lib.po2_conv2d_dgrad(ONE, ONE, None, ONE, B, C, H, W, K, R, S, 1, 1, 1, 0, 4, 1, compute, ONE, BIG,
                                None) == PO2_E_SIZE


@pytest.mark.parametrize("compute, want", [(TF32, (1, 2)), (BF16_OPS, (1,))])
def test_wgrad_kind(lib, compute, want):
    B, C, H, W, K, R, S = RESNET_UNDER
    assert lib.po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, R, S, 1, 1, 1, compute) in want
    B, C, H, W, K, R, S = RESNET_AT
    assert lib.po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, R, S, 1, 1, 1, compute) == 0
    assert lib.po2_conv2d_wgrad_workspace(B, C, H, W, K, R, S, 1, 1, 1, compute) == 0


# ---- entry points without a planning query: refused at 2^31 before any launch --------------------------------------
@pytest.mark.parametrize("B, C, HW", [(2**31 // 64 // 49 + 1, 64, 49), (1 << 25, 64, 1), (1 << 20, 64, 32), (2, 1, 1 << 30)])
def test_bn_refuses_two_to_the_31(lib, B, C, HW):
    assert B * C * HW >= 2**31
    ws = lib.po2_bn_workspace_bytes(C)
    assert lib.po2_bn_stats(ONE, B, C, HW, ONE, ONE, ws, None, 0, 1, None) == PO2_E_SIZE
    assert lib.po2_bn_apply(ONE, None, ONE, ONE, 1, None, None, None, None, None, None, None, 0.1, 1e-5, 1, 0, None, None,
                            B, C, HW, None) == PO2_E_SIZE
    assert lib.po2_bn_fwd_fused(ONE, None, ONE, None, None, None, None, None, 0.1, 1e-5, 1, ONE, ONE, None, B, C, HW, ONE,
                                ws, None, 0, 1, None) == PO2_E_SIZE
    assert lib.po2_bn_bwd_reduce(ONE, None, ONE, ONE, ONE, ONE, None, None, ONE, None, None, 1, B, C, HW, ONE, ws, None,
                                 0, 1, None) == PO2_E_SIZE
    assert lib.po2_bn_bwd_apply(ONE, None, ONE, ONE, ONE, ONE, None, None, ONE, ONE, 1, None, ONE, None, 1, B, C, HW,
                                None) == PO2_E_SIZE
    assert lib.po2_bn_bwd_fused(ONE, None, ONE, ONE, ONE, ONE, None, None, None, None, ONE, None, 1, B, C, HW, ONE, ws,
                                None) in (PO2_E_SIZE, -10)


@pytest.mark.parametrize("B, C, H, W", [(76088, 576, 7, 7), (1 << 14, 1, 1 << 8, 1 << 9), (1, 1, 46341, 46341)])
def test_depthwise_backward_refuses_two_to_the_31(lib, B, C, H, W):
    assert B * C * H * W >= 2**31
    assert lib.po2_conv2d_depthwise_dgrad(ONE, ONE, ONE, B, C, H, W, None) == PO2_E_SIZE
    ws = lib.po2_conv2d_depthwise_wgrad_workspace(C)
    assert lib.po2_conv2d_depthwise_wgrad(ONE, ONE, ONE, B, C, H, W, ONE, ws, None) == PO2_E_SIZE


def test_dilate_refuses_two_to_the_31(lib):
    # g_up (planes, H, W) of 2^31 + 2^14 elements, odd H: the stride-2 backward of a 576-channel 7x7 layer
    assert lib.po2_dilate2_into(ONE, ONE, 76087 * 576 + 335, 4, 4, 7, 7, None) == PO2_E_SIZE
    assert lib.po2_dilate2(ONE, ONE, 1 << 17, 64, 64, None) == PO2_E_SIZE              # g_up 2^31


def test_sgd_refuses_two_to_the_31(lib):
    arr = ctypes.c_void_p * 1
    for n in (2**31, 2**31 + 3, 2**32):
        numel = (ctypes.c_longlong * 1)(n)
        assert lib.po2_sgd_step(arr(ONE), arr(ONE), arr(ONE), numel, 1, 0.1, 0.9, 1e-4, 0, None) == PO2_E_SIZE


@pytest.mark.parametrize("C, K, compute, dtype", [(1792, 600000, TF32, F32), (3584, 300000, BF16_OPS, F32),
                                                  (3584, 300000, BF16_OPS, BF16)])
def test_packed_operand_of_two_to_the_30_leaves_the_tensor_cores(lib, C, K, compute, dtype):
    """a 1x1 layer whose packed weight operand has >= 2^30 elements (pack_weights_kernel's 32-bit loop): no
    tensor-core kind, no packed operand, and no workspace for one -- the query and every launch agree"""
    B, H, W = 2, 32, 32
    assert C * K >= 2**30 and B * C * H * W < 2**31 and B * K * H * W < 2**31
    k = kind(lib, (B, C, H, W, K, 1, 1), compute, dtype=dtype)
    assert k not in (2, 3)
    assert k == (0 if dtype == F32 else -10)                   # the direct kernel; a bf16 x has no direct form
    assert lib.po2_conv2d_pack_bytes(B, C, H, W, K, 1, 1, 1, 0, 1, compute) == 0
    if dtype == F32:
        assert lib.po2_conv2d_workspace_dt(B, C, H, W, K, 1, 1, 1, 0, 1, compute, F32) == \
            (K * C * 4 + 255) // 256 * 256                     # the decoded fp32 weight only
