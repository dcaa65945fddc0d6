"""Backward of stride-2 layers of any size (3x3 pad 1, 1x1 pad 0): odd H or W, and an odd output width, take the same
route as the even layers -- the output gradient zero-inserted to the input's H x W, then the stride-1 data- and
weight-gradient kernels -- with the zero-insertion of po2_dilate2_into where po2_dilate2 (even sizes, even Q) refuses
the shape.  Checked bit for bit on the zero-insertion and on exactly representable operands, against fp64 on random
operands, and in whole QAT steps of MobileNetV2-CIFAR, MobileViT-xs at 32x32 and ResNet-20 at 28x28, whose odd-size
stride-2 layers used to leave our kernels for aten.convolution_backward."""
import os

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import _lib, ops  # noqa: E402

from tests.test_conv_exact_gpu import _gen, _truncate_tf32, lattice_x, quantized_lattice_w  # noqa: E402

NAN = float("nan")
TOL_TC = 1e-2          # bf16 operands (test_conv_gpu.py)
TOL_TF32 = 2e-3        # tf32 operands
TOL_FP32 = 1e-4        # the CUDA-core kernels (test_conv_gpu.py's depthwise tolerance, TOL_FP32 * 10)


def _out_hw(H, W):
    return (H - 1) // 2 + 1, (W - 1) // 2 + 1


def _offset(t, lo):
    """a contiguous copy of t starting `lo` floats past a 16-byte boundary"""
    buf = torch.empty(t.numel() + 4, device="cuda")
    v = buf[lo:lo + t.numel()].view(t.shape)
    v.copy_(t)
    return v


# ---- the zero-insertion ------------------------------------------------------------------------------------------
SIZES = [(1, 1), (2, 2), (3, 3), (2, 5), (5, 2), (7, 7), (14, 14), (15, 8), (8, 4)]    # 8x4: po2_dilate2's too


@pytest.mark.parametrize("lo", [0, 1], ids=["aligned", "offset4"])
@pytest.mark.parametrize("hw", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_zero_insertion_is_bit_exact(hw, lo):
    """g_up[2p][2q] = g[p][q], zero elsewhere; every element written (g_up starts as NaN), at any 4-byte alignment"""
    H, W = hw
    P_, Q = _out_hw(H, W)
    gen = torch.Generator(device="cuda").manual_seed(H * 100 + W)
    g = _offset(torch.randn(3, 5, P_, Q, device="cuda", generator=gen), lo)
    want = torch.zeros(3, 5, H, W, device="cuda")
    want[..., ::2, ::2] = g
    up = _offset(torch.full((3, 5, H, W), NAN, device="cuda"), lo)
    before = ops.LAUNCHES
    ops.dilate2_into_out(g, up)
    assert ops.LAUNCHES - before == 1
    assert torch.equal(up, want), (hw, lo)
    if H % 2 == 0 and W % 2 == 0 and Q % 2 == 0 and lo == 0:      # both kernels take it: the same bits
        up2 = torch.full_like(up, NAN)
        ops.dilate2_out(g, up2)
        assert torch.equal(up2, up)


def test_zero_insertion_loops_over_a_large_plane_set():
    """more elements than the capped grid has threads (148 SMs x 16 blocks x 256): the grid-stride loop"""
    g = torch.randn(128, 96, 8, 8, device="cuda")
    up = torch.full((128, 96, 15, 15), NAN, device="cuda")
    ops.dilate2_into_out(g, up)
    want = torch.zeros_like(up)
    want[..., ::2, ::2] = g
    assert torch.equal(up, want)


# ---- layer gradients ---------------------------------------------------------------------------------------------
# (name, B, C, H, W, K, k, groups)
DEPTHWISE = [("dw 320 @2x2", 16, 320, 2, 2), ("dw 576 @2x2", 128, 576, 2, 2), ("dw 32 @7x7", 8, 32, 7, 7),
             ("dw 48 @14x14", 8, 48, 14, 14), ("dw 24 @5x8", 8, 24, 5, 8)]
LAYERS = [(n, B, C, H, W, C, 3, C) for n, B, C, H, W in DEPTHWISE] + [
    (f"{k}x{k} {C}->{K} @{H}x{W}", 8, C, H, W, K, k, 1)
    for C, K in ((16, 32), (32, 64)) for k in (3, 1) for H, W in ((14, 14), (7, 7), (15, 15))]


def _expected_launches(case, compute):
    """the zero-insertion + the data gradient + the weight gradient (each with its reduce kernel where it has one)"""
    name, B, C, H, W, K, k, groups = case
    if groups > 1:
        return 1 + 1 + 1
    kind = _lib.load().po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, k, k, 1, k // 2, 1, compute)
    fused = kind == 2 and os.environ.get("PO2_WGRAD_FUSED_REDUCE", "0") == "1"
    return 1 + 2 + (1 if fused else 2)


def _backward(case, x, w, scale, g, compute, monkeypatch):
    """x.grad, w.grad of torch.ops.po2.conv2d; asserts our kernels only, the launch count and the zero-insertion used"""
    name, B, C, H, W, K, k, groups = case
    calls = []
    for fn in ("dilate2_out", "dilate2_into_out"):
        real = getattr(ops, fn)
        monkeypatch.setattr(ops, fn, lambda a, b, real=real, fn=fn: (calls.append(fn), real(a, b))[1])
    xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ops._noted.discard("conv_backward_aten")
    out = torch.ops.po2.conv2d(xr, wr, scale, 2, k // 2, groups, compute)
    assert out.shape[2:] == _out_hw(H, W)
    before = ops.LAUNCHES
    out.backward(g)
    assert "conv_backward_aten" not in ops._noted, (name, "the backward fell back to aten.convolution_backward")
    assert ops.LAUNCHES - before == _expected_launches(case, compute), (name, ops.LAUNCHES - before)
    even = H % 2 == 0 and W % 2 == 0 and out.shape[3] % 2 == 0
    assert calls == ["dilate2_out" if even else "dilate2_into_out"], (name, calls)
    monkeypatch.undo()
    return xr.grad, wr.grad


def _fp64(x, w, g, k, groups):
    xd, wd = x.double().requires_grad_(True), w.double().requires_grad_(True)
    F.conv2d(xd, wd, None, 2, k // 2, 1, groups).backward(g.double())
    return xd.grad, wd.grad


@pytest.mark.parametrize("compute", [0, 2], ids=["bf16", "tf32"])
@pytest.mark.parametrize("case", LAYERS, ids=lambda c: c[0])
def test_layer_gradients_are_bit_exact_on_lattice_operands(case, compute, monkeypatch):
    """x, g integers in [-4, 4], PO2 weights (tests/test_conv_exact_gpu.py): every sum is exact, so both gradients are
    fp64 autograd of F.conv2d rounded once to fp32, bit for bit"""
    name, B, C, H, W, K, k, groups = case
    gen = _gen("s2 any size", name, compute)
    x = lattice_x((B, C, H, W), gen)
    w, scale = quantized_lattice_w((K, C // groups, k, k), gen)
    g = lattice_x((B, K) + _out_hw(H, W), gen)
    assert 16 * B * H * W < 2 ** 23 and 4 * k * k * K * 2 ** 7 < 2 ** 23          # the exactness bounds
    gx, gw = _backward(case, x, w, scale, g, compute, monkeypatch)
    rx, rw = _fp64(x, w, g, k, groups)
    assert torch.equal(gx, rx.float()), (name, "dx", (gx != rx.float()).sum().item())
    assert torch.equal(gw, rw.float()), (name, "dw", (gw != rw.float()).sum().item())


def _rel(out, ref):
    return ((out.double() - ref).abs().max() / ref.abs().max()).item()


@pytest.mark.parametrize("compute", [0, 2], ids=["bf16", "tf32"])
@pytest.mark.parametrize("case", LAYERS, ids=lambda c: c[0])
def test_layer_gradients_match_fp64_on_random_operands(case, compute, monkeypatch):
    name, B, C, H, W, K, k, groups = case
    gen = torch.Generator(device="cuda").manual_seed(B + C + H * W + K + k + compute)
    x = torch.randn(B, C, H, W, device="cuda", generator=gen)
    w0 = torch.randn(K, C // groups, k, k, device="cuda", generator=gen) * 0.1
    w, codes, scale, zc, sse = torch.ops.po2.quantize_full(w0, 4, 1, True)
    g = torch.randn((B, K) + _out_hw(H, W), device="cuda", generator=gen)
    gx, gw = _backward(case, x, w, scale, g, compute, monkeypatch)
    rx, rw = _fp64(x, w, g, k, groups)
    if groups > 1:
        tol_x = tol_w = TOL_FP32
    else:
        tol_x = TOL_TF32 if compute == 2 else TOL_TC
        kind = _lib.load().po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, k, k, 1, k // 2, 1, compute)
        tol_w = {1: TOL_TC, 2: TOL_TF32, 3: TOL_FP32}[kind]
    assert _rel(gx, rx) < tol_x, (name, _rel(gx, rx))
    assert _rel(gw, rw) < tol_w, (name, _rel(gw, rw))


# ---- whole QAT steps ---------------------------------------------------------------------------------------------
MODELS = {"mobilenetv2_b128": 576, "mobilevit_xs32_b16": 320, "resnet20_28x28_b64": None}


def _qat_model(name):
    """default tf32 conv mode, fused norms, weight prefetch (as _qat_model in tests/test_pw_wgrad_gpu.py)"""
    from workloads import mobilenet_v2_cifar, mobilevit_xs, resnet_cifar
    torch.manual_seed(0)
    dev = torch.device("cuda:0")
    hw = 32
    if name == "mobilenetv2_b128":
        model, batch = mobilenet_v2_cifar(10, P.PowerOfTwoPlusQuantizer, 4), 128
    elif name == "mobilevit_xs32_b16":
        model, batch = mobilevit_xs((32, 32), 10, (1, 1), P.PowerOfTwoPlusQuantizer, 4), 16
    else:
        model, batch, hw = resnet_cifar(20, 10, P.PowerOfTwoPlusQuantizer, 4), 64, 28
    model = model.to(dev).train()
    P.enable_weight_prefetch(model)
    x = torch.randn(batch, 3, hw, hw, device=dev)
    t = torch.randint(0, 10, (batch,), device=dev)
    return model, x, t


@pytest.fixture
def deterministic_cudnn():
    was = torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic = False, True
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic = was


def _bf16(t):
    return t.bfloat16().float()


def _aten_route(g, x, w, pad, groups, compute):
    """(gx, gw) of aten.convolution_backward -- what ops._conv_backward runs when our kernels do not take a layer --
    on the operands our kernels read: the tensor-core kernels take g (and x for the weight gradient) as bf16 (compute
    0, round to nearest even) or tf32 (compute 2, truncated), or fp32 for the CUDA-core weight-gradient GEMM (kind 3);
    the depthwise kernels are fp32.  Then the two routes differ only in fp32 summation order."""
    B, C, H, W = x.shape
    K, _, R, S = w.shape
    gd = gw_g = g
    xw = x
    if groups == 1:
        gd = _truncate_tf32(g) if compute == 2 else _bf16(g)
        kind = _lib.load().po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, R, S, 1, pad, 1, compute)
        rnd = {1: _bf16, 2: _truncate_tf32, 3: lambda t: t}[kind]
        gw_g, xw = rnd(g), rnd(x)
    args = (None, [2, 2], [pad, pad], [1, 1], False, [0, 0], groups)
    gx = torch.ops.aten.convolution_backward(gd.contiguous(), x, w, *args, [True, False, False])[0]
    gw = torch.ops.aten.convolution_backward(gw_g.contiguous(), xw.contiguous(), w, *args, [False, True, False])[1]
    return gx, gw


def _rms(a, b):
    return ((a.double() - b.double()).pow(2).mean().sqrt() / b.double().pow(2).mean().sqrt()).item()


@pytest.mark.parametrize("name", list(MODELS))
def test_qat_step_runs_every_stride2_backward_on_our_kernels(name, deterministic_cudnn, monkeypatch):
    """One QAT step: no convolution backward takes aten.convolution_backward, and the gradients of the stride-2 layers
    that po2_dilate2 refuses (for ResNet-20 at 28x28: all of its stride-2 layers) are within rms 1e-5 of the aten
    route on the same output gradient, input and weight"""
    model, x, t = _qat_model(name)
    notes = []
    monkeypatch.setattr(ops, "note_library_path", lambda key, message: notes.append((key, message)))
    seen = []
    real = ops._conv_backward

    def recording(g, x, w, scale, stride, pad, groups, compute, need_x, need_w, *args, **kw):
        gx, gw = real(g, x, w, scale, stride, pad, groups, compute, need_x, need_w, *args, **kw)
        H, W = x.shape[2:]
        odd = H % 2 or W % 2 or g.shape[3] % 2
        if stride == 2 and (odd or MODELS[name] is None):
            seen.append((g.detach().clone(), x.detach().clone(), w.detach().clone(), pad, groups, compute,
                         gx.clone() if gx is not None else None, gw.clone()))
        return gx, gw

    monkeypatch.setattr(ops, "_conv_backward", recording)
    model.zero_grad(set_to_none=True)
    nn.CrossEntropyLoss()(model(x), t).backward()
    torch.cuda.synchronize()
    monkeypatch.undo()
    assert not [m for k, m in notes if k == "conv_backward_aten"], notes
    assert seen, name
    if MODELS[name] is not None:
        assert any(gr[4] == MODELS[name] for gr in seen), [tuple(s[1].shape) for s in seen]
    else:
        assert len(seen) == 4 and sum(s[1].shape[2] == 14 for s in seen) == 2      # 28 -> 14 and 14 -> 7, 3x3 + 1x1
    for g, xx, w, pad, groups, compute, gx, gw in seen:
        rx, rw = _aten_route(g, xx, w, pad, groups, compute)
        what = (tuple(xx.shape), tuple(w.shape), groups)
        if gx is not None:                     # the first layer after the stem needs no data gradient
            assert _rms(gx, rx) <= 1e-5, (what, "dx", _rms(gx, rx))
        assert _rms(gw, rw) <= 1e-5, (what, "dw", _rms(gw, rw))


@pytest.mark.parametrize("name", [n for n in MODELS if MODELS[n] is not None])
def test_qat_step_under_graph_replay(name, deterministic_cudnn):
    """Two replays of the captured step give the eager step's gradients of every quantized conv bit for bit"""
    model, x, t = _qat_model(name)
    crit = nn.CrossEntropyLoss()
    convs = {id(m.weight) for m in model.modules() if isinstance(m, P.QuantizedConv2d)}

    def step():
        model.zero_grad(set_to_none=True)
        crit(model(x), t).backward()

    step()
    torch.cuda.synchronize()
    want = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
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
    for n, p in model.named_parameters():
        if n not in want:
            continue
        if id(p) in convs:
            assert torch.equal(p.grad, want[n]), n
        else:                                             # stem / head / norms / attention: not these kernels
            assert torch.allclose(p.grad, want[n], rtol=1e-4, atol=1e-6), n
