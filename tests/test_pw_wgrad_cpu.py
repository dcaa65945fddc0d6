"""Which weight gradients the fp32 pointwise GEMM (conv_wgrad_pw_kernel, kernel kind 3) takes: a host-side planning
question, answered without a GPU.  The kernel itself is tested in tests/test_pw_wgrad_gpu.py."""
import ctypes

import pytest

from po2_quantization_b200 import _lib

# (C, K, H == W, batch): the 1x1 stride-1 layers of the workload models that are wider than the tcgen05 weight-gradient
# kernels take (K > 128 or C > 256), all with B*H*W <= 8192 and at most 39.3 M multiply-adds
MOBILENET_V2 = [(24, 144, 8), (32, 192, 4), (64, 384, 2), (384, 64, 2), (384, 96, 2), (96, 576, 2), (576, 96, 2),
                (576, 160, 1), (160, 960, 1), (960, 160, 1), (960, 320, 1)]
MOBILEVIT_XS_32 = [(48, 192, 8), (64, 256, 4), (80, 320, 2), (320, 96, 1), (96, 144, 1)]
SHAPES = [(C, K, HW, 128) for C, K, HW in MOBILENET_V2] + [(C, K, HW, 16) for C, K, HW in MOBILEVIT_XS_32]

PO2_E_NULL, PO2_E_WORKSPACE, PO2_E_UNSUPPORTED = -3, -8, -10


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}to{s[1]}@{s[2]}B{s[3]}")
@pytest.mark.parametrize("compute", [0, 2], ids=["bf16", "tf32"])
def test_wide_pointwise_layers_take_the_fp32_gemm(lib, shape, compute):
    C, K, HW, B = shape
    q = (B, C, HW, HW, K, 1, 1, 1, 0, 1, compute)
    assert lib.po2_conv2d_wgrad_kernel_kind(*q) == 3
    assert lib.po2_conv2d_wgrad_workspace(*q) >= K * C * 4               # the partials of at least one split


def test_bounds_of_the_fp32_gemm(lib):
    kind, ws = lib.po2_conv2d_wgrad_kernel_kind, lib.po2_conv2d_wgrad_workspace
    # two bounds, both where cuDNN's tensor-core kernels start to win: B*H*W <= 8192 and B*H*W*C*K <= 2^26
    assert kind(128, 24, 8, 8, 144, 1, 1, 1, 0, 1, 2) == 3                # B*H*W exactly 8192
    assert kind(8192, 24, 1, 1, 144, 1, 1, 1, 0, 1, 2) == 3               # the same as 8192 images of 1x1
    assert kind(8193, 24, 1, 1, 144, 1, 1, 1, 0, 1, 2) == 0               # one pixel more
    assert ws(8193, 24, 1, 1, 144, 1, 1, 1, 0, 1, 2) == 0
    assert kind(256, 24, 8, 8, 144, 1, 1, 1, 0, 1, 2) == 0                # B*H*W = 16384
    assert kind(128, 64, 4, 4, 512, 1, 1, 1, 0, 1, 2) == 3                # 2048 * 64 * 512 = 2^26 multiply-adds
    assert kind(128, 64, 4, 4, 513, 1, 1, 1, 0, 1, 2) == 0                # one output channel more
    assert kind(128, 160, 8, 8, 960, 1, 1, 1, 0, 1, 2) == 0               # 1.26 G multiply-adds
    assert kind(128, 64, 8, 8, 192, 3, 3, 1, 1, 1, 2) == 0                # 3x3 with K > 128
    assert kind(16, 320, 4, 4, 160, 3, 3, 1, 1, 1, 0) == 0                # 3x3 with C > 256
    assert kind(128, 960, 1, 1, 320, 1, 1, 1, 0, 1, 1) == 0               # the fp32 mode's backward is ATen
    assert kind(128, 64, 4, 4, 384, 1, 1, 2, 0, 1, 2) == 0                # stride 2 goes through po2_dilate2
    assert kind(128, 64, 4, 4, 384, 1, 1, 1, 1, 1, 2) == 0                # padded 1x1
    assert kind(128, 64, 4, 4, 384, 1, 1, 1, 0, 2, 2) == 0                # grouped
    assert kind(0, 64, 4, 4, 384, 1, 1, 1, 0, 1, 2) == 0                  # empty batch
    # C and K need no alignment
    assert kind(3, 20, 3, 3, 200, 1, 1, 1, 0, 1, 2) == 3
    assert ws(3, 20, 3, 3, 200, 1, 1, 1, 0, 1, 2) >= 200 * 20 * 4


def test_shapes_the_tensor_core_kernels_take_keep_their_kind(lib):
    kind, ws = lib.po2_conv2d_wgrad_kernel_kind, lib.po2_conv2d_wgrad_workspace
    assert kind(128, 32, 16, 16, 16, 1, 1, 1, 0, 1, 0) == 1               # K5
    assert kind(128, 32, 16, 16, 16, 1, 1, 1, 0, 1, 2) in (1, 2)          # K5T where the tensor-map encoder exists
    assert kind(128, 144, 4, 4, 32, 1, 1, 1, 0, 1, 0) == 1                # narrow small-map layer: K5
    assert kind(128, 16, 32, 32, 16, 3, 3, 1, 1, 1, 0) == 1
    assert ws(128, 32, 16, 16, 16, 1, 1, 1, 0, 1, 0) > 0


def test_argument_errors_come_back_before_any_launch(lib):
    one = ctypes.c_void_p(4096)
    q = (128, 960, 1, 1, 320, 1, 1, 1, 0, 1, 2)
    need = lib.po2_conv2d_wgrad_workspace(*q)
    assert lib.po2_conv2d_wgrad_z(one, one, one, *q, None, 0, None, None) == PO2_E_WORKSPACE
    assert lib.po2_conv2d_wgrad_z(one, one, one, *q, one, need - 256, None, None) == PO2_E_WORKSPACE
    assert lib.po2_conv2d_wgrad_z(None, one, one, *q, one, need, None, None) == PO2_E_NULL
    assert lib.po2_conv2d_wgrad(one, one, one, 16385, 960, 1, 1, 320, 1, 1, 1, 0, 1, 2, one, 1 << 30, None) == PO2_E_UNSUPPORTED
