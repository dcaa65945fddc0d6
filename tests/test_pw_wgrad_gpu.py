"""Weight gradient of the wide pointwise layers on conv_wgrad_pw_kernel (kernel kind 3, csrc/po2_conv_bwd.cu): an
exact-fp32 CUDA-core GEMM over (image, pixel) with a fixed-order reduction of its splits.  Against fp64: the
fp32-accumulate tolerance; bit-identical from call to call; and in the QAT steps of MobileNetV2 and MobileViT no
dense layer's backward is left on aten.convolution_backward."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import _lib, ops  # noqa: E402

from tests.test_pw_wgrad_cpu import SHAPES  # noqa: E402

TOL_FP32 = 1e-5
TOL_TF32 = 2e-3

# (name, B, C, H, W, K, stride)
CASES = [(f"{C}to{K}@{HW}B{B}", B, C, HW, HW, K, 1) for C, K, HW, B in SHAPES] + [
    ("20to200@3x3 (C, K not multiples of 8)", 3, 20, 3, 3, 200, 1),
    ("37to131@5x5 (odd C, K and HW)", 2, 37, 5, 5, 131, 1),
    ("50to150@4x4 (128-bit loads, C % 4 != 0)", 7, 50, 4, 4, 150, 1),
    ("960to320@1 B=1", 1, 960, 1, 1, 320, 1),
    ("96to576@8 B=1", 1, 96, 8, 8, 576, 1),
    ("24to144@8 B=128 (B*H*W = 8192, the bound)", 128, 24, 8, 8, 144, 1),
    ("64to512@4 B=128 (2^26 multiply-adds, the bound)", 128, 64, 4, 4, 512, 1),
    ("64to192 stride 2 @8 (dilate2)", 32, 64, 8, 8, 192, 2),
]


def _rel(out, ref):
    return ((out.double() - ref).abs().max() / ref.abs().max()).item()


def _operands(B, C, H, W, K, stride, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, C, H, W, device="cuda", generator=gen)
    g = torch.randn(B, K, H // stride, W // stride, device="cuda", generator=gen)
    return x, g


@pytest.mark.parametrize("case", CASES, ids=lambda c: c[0])
def test_pointwise_wgrad_matches_fp64_and_is_deterministic(case):
    name, B, C, H, W, K, stride = case
    assert _lib.load().po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, 1, 1, 1, 0, 1, 2) == 3, name
    x, g = _operands(B, C, H, W, K, stride, B + C + K)
    g_s1 = g
    if stride == 2:                          # the stride-1 problem with the zero-inserted output gradient
        g_s1 = torch.empty(B, K, H, W, device="cuda")
        ops.dilate2_out(g, g_s1)
    ref = torch.nn.grad.conv2d_weight(x.double(), (K, C, 1, 1), g.double(), stride=stride)
    for compute in (2, 0):
        gw = torch.full((K, C, 1, 1), float("nan"), device="cuda")
        assert ops.conv2d_wgrad_out(g_s1, x, gw, 0, compute)
        assert _rel(gw, ref) < TOL_FP32, (name, compute, _rel(gw, ref))
        gw2 = torch.full_like(gw, float("nan"))
        assert ops.conv2d_wgrad_out(g_s1, x, gw2, 0, compute)
        assert torch.equal(gw, gw2), "the weight gradient must be deterministic"


def test_pointwise_wgrad_counts_two_launches():
    x, g = _operands(128, 960, 1, 1, 320, 1, 5)
    gw = torch.empty(320, 960, 1, 1, device="cuda")
    before = ops.LAUNCHES
    assert ops.conv2d_wgrad_out(g, x, gw, 0, 2)
    assert ops.LAUNCHES - before == 2                    # conv_wgrad_pw_kernel + conv_wgrad_reduce_kernel


AUTOGRAD = [c for c in CASES if c[0].startswith(("24to144", "960to320@1B", "384to64", "80to320", "20to200", "64to192"))]


@pytest.mark.parametrize("case", AUTOGRAD, ids=lambda c: c[0])
def test_autograd_of_wide_pointwise_layers_leaves_aten(case):
    name, B, C, H, W, K, stride = case
    gen = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(B, C, H, W, device="cuda", generator=gen).requires_grad_(True)
    w0 = torch.randn(K, C, 1, 1, device="cuda", generator=gen) * 0.1
    y, codes, scale, zc, sse = torch.ops.po2.quantize_full(w0, 4, 1, True)
    w = y.clone().requires_grad_(True)
    ops._noted.discard("conv_backward_aten")
    out = torch.ops.po2.conv2d(x, w, scale, stride, 0, 1, 2)
    g = torch.randn(out.shape, device="cuda", generator=gen)
    out.backward(g)
    assert "conv_backward_aten" not in ops._noted, "the backward fell back to aten.convolution_backward"
    xd, wd = x.detach().double().requires_grad_(True), y.double().requires_grad_(True)
    F.conv2d(xd, wd, None, stride, 0).backward(g.double())
    assert _rel(x.grad, xd.grad) < TOL_TF32, (name, _rel(x.grad, xd.grad))
    assert _rel(w.grad, wd.grad) < TOL_FP32, (name, _rel(w.grad, wd.grad))


# ---- whole QAT steps ---------------------------------------------------------------------------------------------
MODELS = {"mobilenetv2_b128": 25, "mobilevit_xs32_b16": 7}       # quantized convs whose weight gradient is kind 3


def _qat_model(name):
    from workloads import mobilenet_v2_cifar, mobilevit_xs
    torch.manual_seed(0)
    dev = torch.device("cuda:0")
    if name == "mobilenetv2_b128":
        model, batch = mobilenet_v2_cifar(10, P.PowerOfTwoPlusQuantizer, 4), 128
    else:
        model, batch = mobilevit_xs((32, 32), 10, (1, 1), P.PowerOfTwoPlusQuantizer, 4), 16
    model = model.to(dev).train()
    P.enable_weight_prefetch(model)
    x = torch.randn(batch, 3, 32, 32, device=dev)
    t = torch.randint(0, 10, (batch,), device=dev)
    # the layers whose weight gradient the pointwise GEMM computes, from their input shapes
    lib, seen = _lib.load(), []
    convs = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d)]
    hooks = [m.register_forward_hook(lambda m, i, o: seen.append((m, tuple(i[0].shape)))) for m in convs]
    with torch.no_grad():
        model(x)
    for h in hooks:
        h.remove()
    kind3 = [m for m, (B, C, H, W) in seen if m.groups == 1 and
             lib.po2_conv2d_wgrad_kernel_kind(B, C, H, W, m.out_channels, *m.kernel_size, 1, m.padding[0], 1, 2) == 3]
    return model, x, t, convs, kind3


@pytest.fixture
def deterministic_cudnn():
    was = torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic = False, True
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic = was
        ops.set_wgrad_mode("tc")
        ops.set_wgrad_overlap(False)


@pytest.mark.parametrize("name", list(MODELS))
def test_qat_step_weight_gradients_leave_cudnn(name, deterministic_cudnn, monkeypatch):
    """One QAT step (default tf32 conv mode, fused norms, prefetched weights): no dense layer's backward runs on
    aten.convolution_backward, and the kind-3 weight gradients agree with aten.convolution_backward in fp32 on the
    same x and output gradient (the weight gradient is a leaf: switching its kernel changes no other tensor of the
    step).  A depthwise stride-2 layer onto a 1x1 map still takes ATen (po2_dilate2 needs an even output width);
    that is not this kernel's ground."""
    model, x, t, convs, kind3 = _qat_model(name)
    assert len(kind3) == MODELS[name]
    crit = nn.CrossEntropyLoss()
    notes = []
    monkeypatch.setattr(ops, "note_library_path", lambda key, message: notes.append((key, message)))

    def grads():
        model.zero_grad(set_to_none=True)
        crit(model(x), t).backward()
        torch.cuda.synchronize()
        return [m.weight.grad.clone() for m in kind3]

    ours = grads()
    aten = [m for k, m in notes if k == "conv_backward_aten"]
    assert all(" groups 1 " not in m for m in aten), aten
    ops.set_wgrad_mode("aten")
    ref = grads()
    ops.set_wgrad_mode("tc")
    for m, a, b in zip(kind3, ours, ref):
        rms = ((a.double() - b.double()).pow(2).mean().sqrt() / b.double().pow(2).mean().sqrt()).item()
        assert rms <= 1e-5, (tuple(m.weight.shape), rms)


@pytest.mark.parametrize("name", list(MODELS))
def test_qat_step_with_side_stream_weight_gradients_under_graph_replay(name, deterministic_cudnn):
    """The kind-3 weight gradients deferred to the side stream inside a CUDA graph are the in-order eager ones, bit
    for bit."""
    model, x, t, convs, kind3 = _qat_model(name)
    assert len(kind3) == MODELS[name]
    crit = nn.CrossEntropyLoss()

    def step():
        model.zero_grad(set_to_none=True)
        crit(model(x), t).backward()

    ops.set_wgrad_overlap(False)
    step()
    torch.cuda.synchronize()
    want = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
    ops.set_wgrad_overlap(True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
        s.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            step()
        for _ in range(2):
            graph.replay()
        s.synchronize()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    ops.set_wgrad_overlap(False)
    qnames = {id(m.weight) for m in convs}
    for n, p in model.named_parameters():
        if n not in want:
            continue
        if id(p) in qnames:
            assert torch.equal(p.grad, want[n]), n
        else:                                             # stem / head / norms: not this kernel's gradients
            assert torch.allclose(p.grad, want[n], rtol=1e-4, atol=1e-6), n
