"""bf16 models at inference on our kernels: the K3 / depthwise / small-pointwise forward with bf16 activations.

Lattice cases (the operands of tests/test_conv_exact_gpu.py: integer x in [-4, 4], weights +-2^-3 * 2^q) are exact as
bf16 values and every partial sum is exact in fp32, so a correct kernel returns the fp64 conv rounded ONCE to bf16, bit
for bit.  Each case also checks the kernel kind it names, that a NaN-filled output is completely written and that a
second call gives the same bits.  Then whole bf16 models, post-training quantized, against the same bf16 model on
cuDNN."""
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import _lib, ops  # noqa: E402

from tests.test_bf16_inference_cpu import bf16_kind  # noqa: E402
from tests.test_conv_exact_cpu import FWD, fwd_exact  # noqa: E402

S_W = 2.0 ** -3
BF = torch.bfloat16


def _gen(*key):
    return torch.Generator(device="cuda").manual_seed(zlib.crc32(repr(("bf16",) + key).encode()))


def _lattice(shape, gen):
    return torch.randint(-4, 5, shape, generator=gen, device="cuda").float()


def _lattice_w(shape, gen):
    q = torch.randint(-7, 1, shape, generator=gen, device="cuda").float()
    sign = torch.randint(0, 2, shape, generator=gen, device="cuda").float() * 2 - 1
    keep = (torch.randint(0, 8, shape, generator=gen, device="cuda") != 0).float()
    w = sign * torch.exp2(q) * keep * S_W
    w.view(-1)[0] = S_W
    return w


def _ref(x, w, stride, pad, groups):
    """fp64 conv; exact in fp32 on the lattice, so .float().to(bf16) rounds once"""
    return F.conv2d(x.double(), w.double(), None, stride, pad, 1, groups).float()


# every forward case a bf16 x runs on (K3 branches vec4 / scalar / hw1 / s2 / flat, depthwise vec / scalar, small-pw),
# plus bf16-only producer shapes: W % 8 != 0 with W % 4 == 0 (scalar for bf16, vec4 for fp32), and hw1 with C % 8 != 0
BF16_FWD = [c for c in FWD if bf16_kind(c[10], c[9]) > 0] + [
    ("k3 bf16 3x3 16->16 @12 (W % 8 = 4)", 4, 16, 12, 12, 16, 3, 1, 1, 0, 2, ()),
    ("k3 bf16 3x3 20->16 @1x1 (C % 8 = 4)", 16, 20, 1, 1, 16, 3, 1, 1, 2, 2, ()),
    ("k3 bf16 3x3 s2 24->32 @15x9", 3, 24, 15, 9, 32, 3, 2, 1, 0, 2, ()),
]


@pytest.mark.parametrize("case", BF16_FWD, ids=lambda c: c[0])
def test_bf16_forward_is_the_fp64_conv_rounded_once(case):
    name, B, C, H, W, K, k, stride, groups, compute, kind, _ = case
    pad = k // 2
    assert fwd_exact(C, k, groups)
    want = bf16_kind(kind, compute)
    assert ops.conv_kernel_kind((B, C, H, W), (K, C // groups, k, k), stride, pad, groups, compute, BF) == want, name
    gen = _gen(name)
    x = _lattice((B, C, H, W), gen)
    w = _lattice_w((K, C // groups, k, k), gen)
    scale = torch.full((), S_W, device="cuda")
    ref = _ref(x, w, stride, pad, groups).to(BF)
    xb = x.to(BF)
    outs = []
    for _ in range(2):
        out = torch.full(ref.shape, float("nan"), dtype=BF, device="cuda")
        ops.conv2d_out(xb, w, scale, out, stride, pad, groups, compute)
        outs.append(out)
    assert not outs[0].isnan().any(), name
    assert torch.equal(outs[0], ref), (name, (outs[0] != ref).sum().item())
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16)), name
    with torch.no_grad():
        assert torch.equal(torch.ops.po2.conv2d(xb, w.to(BF), scale, stride, pad, groups, compute), ref), (name, "op")
        packed = ops.conv2d_pack(w.to(BF), scale, x.shape, stride, pad, groups, compute, BF)
        assert (packed is not None) == (want == 2), name
        if packed is not None:
            out = torch.ops.po2.conv2d_packed(xb, packed, scale, K, k, k, stride, pad, groups, compute)
            assert torch.equal(out, ref), (name, "packed")


EP_CASES = [c for c in BF16_FWD if c[0] in (
    "dw vec s1 32 @16", "dw vec s2 24 @16", "dw scalar 7 @9x7", "k3 3x3 s1 16->16 @16", "k3 3x3 s1 24->40 @14x9",
    "k3 3x3 s2 16->32 @16", "k3 1x1 s1 32->48 @6", "k3 3x3 32->32 @1x1 (hw1)", "k3 3x3 256->32 @8 (chunks)",
    "k3t mode0 16->16 @32", "pw split 576->160 @1", "pw single 24->40 @4x4")]


def _bf16_ulp(t):
    a = t.abs().to(BF)
    return (torch.nextafter(a.float(), torch.full_like(a.float(), float("inf"))).to(BF).float() - a.float()).clamp_min(2.0 ** -133)


@pytest.mark.parametrize("act", [0, 1, 2, 3], ids=["none", "relu", "relu6", "silu"])
@pytest.mark.parametrize("case", EP_CASES, ids=lambda c: c[0])
def test_bf16_folded_epilogue(case, act):
    """act(conv * a[k] + b[k] + residual), a = +-2^j, b on the 2^-8 grid, a bf16 integer residual: the pre-activation is
    exact in fp32, so the bf16 output is it rounded once -- bit for bit, except SiLU (the kernel's __expf), which is
    within one bf16 ulp of the fp64 SiLU rounded to bf16 (the fp32 error of a few fp32 ulps can move the rounding by one)"""
    name, B, C, H, W, K, k, stride, groups, compute, kind, _ = case
    pad = k // 2
    gen = _gen(name, act)
    x = _lattice((B, C, H, W), gen)
    w = _lattice_w((K, C // groups, k, k), gen)
    scale = torch.full((), S_W, device="cuda")
    a = torch.exp2(torch.randint(-2, 3, (K,), generator=gen, device="cuda").float())
    a = a * (torch.randint(0, 2, (K,), generator=gen, device="cuda").float() * 2 - 1)
    b = torch.randint(-512, 513, (K,), generator=gen, device="cuda").float() * 2.0 ** -8
    conv = F.conv2d(x.double(), w.double(), None, stride, pad, 1, groups)
    res = _lattice(conv.shape, gen) if act != 2 else None
    pre = conv * a.double().view(1, -1, 1, 1) + b.double().view(1, -1, 1, 1)
    if res is not None:
        pre = pre + res.double()
    assert pre.abs().max().item() < 2 ** 12
    xb, resb = x.to(BF), (res.to(BF) if res is not None else None)
    with torch.no_grad():
        out = torch.ops.po2.conv2d_ep(xb, w.to(BF), scale, stride, pad, groups, compute, a, b, resb, act)
        out2 = torch.ops.po2.conv2d_ep(xb, w.to(BF), scale, stride, pad, groups, compute, a, b, resb, act)
    assert out.dtype == BF and not out.isnan().any()
    assert torch.equal(out.view(torch.int16), out2.view(torch.int16)), name
    if act == 3:
        ref = F.silu(pre).float().to(BF)
        assert ((out.float() - ref.float()).abs() <= _bf16_ulp(ref)).all(), name
    else:
        ref = [lambda t: t, torch.relu, lambda t: t.clamp(0, 6)][act](pre).float().to(BF)
        assert torch.equal(out, ref), (name, (out != ref).sum().item())
    packed = ops.conv2d_pack(w.to(BF), scale, x.shape, stride, pad, groups, compute, BF)
    if packed is not None:
        with torch.no_grad():
            out3 = torch.ops.po2.conv2d_packed_ep(xb, packed, scale, K, k, k, stride, pad, groups, compute, a, b, resb, act)
        assert torch.equal(out.view(torch.int16), out3.view(torch.int16)), (name, "packed")


@pytest.mark.parametrize("shape", [(4, 16, 16, 16, 16, 3, 1), (4, 16, 12, 12, 24, 3, 2), (4, 24, 16, 16, 24, 3, 1, 24),
                                   (8, 64, 2, 2, 96, 1, 1)], ids=["k3", "k3-s2", "dw", "pw"])
def test_bf16_subnormal_levels_are_exact(shape):
    """8-bit PO2 levels reach 2^-127 * scale: with scale 1 the smallest weights are bf16 subnormals.  Out channels
    other than 0 hold only levels 2^-127 .. 2^-125, so their outputs consist of those products alone; they must equal
    the fp64 conv (rounded once), i.e. nothing is flushed to zero on the way."""
    B, C, H, W, K, k, stride = shape[:7]
    groups = shape[7] if len(shape) > 7 else 1
    pad = k // 2
    gen = _gen("subnormal", shape)
    x = _lattice((B, C, H, W), gen)
    q = torch.randint(-127, -124, (K, C // groups, k, k), generator=gen, device="cuda").double()
    sign = torch.randint(0, 2, q.shape, generator=gen, device="cuda").double() * 2 - 1
    w64 = sign * torch.exp2(q)
    w64[0] = 0.5
    w64.view(-1)[0] = 1.0
    w = w64.to(BF)
    assert torch.equal(w.double(), w64) and (w.float().abs() < 2.0 ** -126).sum() > 0
    scale = torch.ones((), device="cuda")
    assert ops.conv_kernel_kind(x.shape, w.shape, stride, pad, groups, 0, BF) > 0
    ref = F.conv2d(x.double(), w64, None, stride, pad, 1, groups).float().to(BF)
    assert (ref[:, 1:] != 0).any()
    with torch.no_grad():
        out = torch.ops.po2.conv2d(x.to(BF), w, scale, stride, pad, groups, 0)
    assert torch.equal(out, ref), (shape, (out != ref).sum().item(), (ref[:, 1:] != 0).sum().item())


def test_bf16_conv_refuses_autograd():
    x = torch.randn(2, 16, 8, 8, device="cuda", dtype=BF, requires_grad=True)
    w = torch.randn(16, 16, 3, 3, device="cuda", dtype=BF)
    with pytest.raises(RuntimeError, match="inference only"):
        torch.ops.po2.conv2d(x, w, None, 1, 1, 1, 0)


def _model(family):
    from workloads.mobilenet_cifar import mobilenet_v2_cifar
    from workloads.mobilevit import mobilevit_xs
    from workloads.resnet_cifar import resnet_cifar
    torch.manual_seed(5)
    if family == "resnet20":
        return resnet_cifar(20, 10, None, 4), torch.randn(64, 3, 32, 32), 4
    if family == "mobilenet":
        return mobilenet_v2_cifar(10, None, 4), torch.randn(64, 3, 32, 32), 4
    return mobilevit_xs((64, 64), 10, (2, 2), None, 8), torch.randn(8, 3, 64, 64), 8


@pytest.mark.parametrize("fold", [False, True], ids=["separate", "folded"])
@pytest.mark.parametrize("family", ["resnet20", "mobilenet", "mobilevit"])
def test_bf16_ptq_models_run_on_our_kernels(family, fold, monkeypatch):
    """bf16 PTQ inference: cast to bf16 FIRST, then quantize_model (a cast afterwards makes new parameters and the PTQ
    tag goes stale).  No QuantizedConv2d leaves our kernels; the logits match the same bf16 model on cuDNN; the forward
    replays in a CUDA graph with the same bits.

    Tolerance: both paths round each conv output to bf16 (relative error <= 2^-8), and the reference also rounds the
    norm's output and the residual sum separately, where the folded epilogue rounds once.  Counting up to three bf16
    roundings per quantized layer on the deepest path, a worst-case linear bound is 3 * n_layers * 2^-8 of the logit
    scale (max |logit|); top-1 must agree wherever the reference's margin exceeds that bound."""
    m, x, bits = _model(family)
    m, x = m.cuda().to(BF).eval(), x.cuda().to(BF)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
                mod.running_mean.normal_(0, 0.2); mod.running_var.uniform_(0.5, 1.5)
                mod.weight.uniform_(0.7, 1.3); mod.bias.normal_(0, 0.1)
    P.quantize_model(m, P.PowerOfTwoPlusQuantizer, bits)
    n_layers = sum(isinstance(mod, P.QuantizedConv2d) for mod in m.modules())
    if fold:
        assert P.fold_conv_bn(m) > 0 or family == "resnet20"
    monkeypatch.setenv("PO2_FOLD_BN", "1" if fold else "0")
    monkeypatch.delenv("PO2_STRICT", raising=False)
    notes = []
    real_note = ops.note_library_path
    monkeypatch.setattr(ops, "note_library_path", lambda key, msg: (notes.append(key), real_note(key, msg)))
    mode = ops.get_conv_mode()
    try:
        with torch.no_grad():
            ops.set_conv_mode("cudnn")
            ref = m(x).float()
            ops.set_conv_mode("tf32")
            out = m(x)
            ops.set_conv_mode("tc")
            out_tc = m(x)
            ops.set_conv_mode("tf32")
            n0 = ops.LAUNCHES
            again = m(x)
            launches = ops.LAUNCHES - n0
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                m(x)
            torch.cuda.current_stream().wait_stream(s)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                captured = m(x)
            g.replay()
            torch.cuda.synchronize()
    finally:
        ops.set_conv_mode(mode)
    assert not [k for k in notes if k.startswith("qconv:")], notes
    assert out.dtype == BF and launches >= n_layers // 2
    assert torch.equal(out.view(torch.int16), again.view(torch.int16))
    assert torch.equal(out.view(torch.int16), out_tc.view(torch.int16))           # bf16 operands in both modes
    assert torch.equal(captured.view(torch.int16), out.view(torch.int16))
    tol = 3 * n_layers * 2.0 ** -8
    scale = ref.abs().max()
    rel = ((out.float() - ref).abs().max() / scale).item()
    assert rel <= tol, (rel, tol)
    top = ref.topk(2, dim=1).values
    decisive = (top[:, 0] - top[:, 1]) > tol * scale
    assert torch.equal(out.float().argmax(1)[decisive], ref.argmax(1)[decisive])
    print(f"{family} fold={fold}: rel {rel:.3e} (bound {tol:.3e}), {launches} launches")


@pytest.mark.parametrize("k,stride,groups", [(3, 1, 1), (3, 2, 1), (3, 1, 32), (1, 1, 1)], ids=["k3", "k3-s2", "dw", "pw"])
def test_bf16_qat_layer_in_eval_quantizes_in_bf16(k, stride, groups):
    """A QAT layer (quantize_fn set) of a bf16 model under no_grad: its bf16 weight is quantized by quantize_full in
    bf16 and the conv runs on our kernels -- the same bits as the layer post-training quantized with quantize_model;
    a changed weight is re-quantized (the cache follows the weight's version)."""
    torch.manual_seed(11)
    H = 2 if k == 1 else 16                            # 1x1 on a 2x2 map: the small-pointwise GEMM
    qat = P.QuantizedConv2d(32, 32, k, stride=stride, padding=k // 2, groups=groups,
                            quantize_fn=P.PowerOfTwoPlusQuantizer, bits=4).cuda().to(BF)
    ptq = P.QuantizedConv2d(32, 32, k, stride=stride, padding=k // 2, groups=groups, bits=4).cuda().to(BF)
    x = torch.randn(8, 32, H, H, device="cuda").to(BF)
    for step in range(2):
        with torch.no_grad():
            ptq.weight.copy_(qat.weight)
        P.quantize_model(ptq, P.PowerOfTwoPlusQuantizer, 4)
        n0 = ops.LAUNCHES
        with torch.no_grad():
            out, ref = qat(x), ptq(x)
        assert ops.LAUNCHES > n0 and out.dtype == BF
        y = ops.quantize_full(qat.weight.detach(), 4, 1, True)[0]
        assert torch.equal(y, ptq.weight)
        assert torch.equal(out.view(torch.int16), ref.view(torch.int16)), step
        with torch.no_grad():
            qat.weight.mul_(-0.5)
