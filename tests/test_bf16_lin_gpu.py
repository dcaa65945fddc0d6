"""lin / lin+ layers of bf16 models at inference on our kernels, and the bf16 lin quantizer kernel.

The quantizer (po2_lin_quantize_dt with PO2_BF16) evaluates the reference's op sequence with every op rounded to bf16,
as torch does on bf16 tensors; it is held to the op-by-op form the way the fp32 kernel is
(tests/test_quantizer_gpu.py::test_lin_cuda_kernel_vs_op_by_op_form).  Its output y is a bf16 tensor, so y is its own
exact tensor-core operand at any bit width (scale 1.0): on lattice activations a bf16 lin layer equals the fp64 conv of
the same y rounded once to bf16, bit for bit, on every kernel a bf16 x runs on.  Then whole bf16 models, post-training
quantized with lin and lin+, against the same bf16 model on cuDNN."""
import copy
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import _lib, ops  # noqa: E402
from po2_quantization_b200 import quantizers as Q  # noqa: E402

BF = torch.bfloat16
LIN = [(P.LinearPowerOfTwoQuantizer, False), (P.LinearPowerOfTwoPlusQuantizer, True)]
LIN_IDS = ["lin", "lin+"]
SHAPES = [(16, 16, 3, 3), (64, 32, 3, 3), (96, 16, 1, 1), (320, 960, 1, 1), (64, 128, 3, 3), (8, 3, 5, 5)]


def _gen(*key, device="cuda"):
    return torch.Generator(device=device).manual_seed(zlib.crc32(repr(("bf16 lin",) + key).encode()))


def _record_notes(monkeypatch):
    notes = []
    real_note = ops.note_library_path
    monkeypatch.setattr(ops, "note_library_path", lambda key, msg: (notes.append(key), real_note(key, msg)))
    monkeypatch.delenv("PO2_STRICT", raising=False)
    return notes


def _op_by_op(w, bits, plus, monkeypatch):
    """the reference's op sequence (quantizers._lin_forward, aten branch) on w's device and dtype"""
    monkeypatch.setenv("PO2_LIN", "aten")
    try:
        return Q._lin_forward(w, bits, ops.LIN_ITERS, plus)
    finally:
        monkeypatch.setenv("PO2_LIN", "cuda")


def _check_channels(got, ref, what):
    """>= 97 % of the input channels bit-identical; each other channel's step exactly one binade away (a ratio
    <q,w>/<q,q> within rounding of a power-of-two tie may go either way with another summation order)"""
    got, ref = got.cpu().float(), ref.cpu().float()
    same = (got.view(torch.int32) == ref.view(torch.int32)).all(dim=3).all(dim=2).all(dim=0)
    assert same.float().mean().item() >= 0.97, (what, same.float().mean().item())
    for c in (~same).nonzero().flatten().tolist():
        sg = got[:, c][got[:, c] != 0].abs().min().item()
        sr = ref[:, c][ref[:, c] != 0].abs().min().item()
        assert sg in (2 * sr, sr / 2), (what, c, sg, sr)
    return same.float().mean().item()


# ---- 1. the kernel against the op-by-op bf16 form ------------------------------------------------------------------
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_bf16_lin_kernel_vs_op_by_op_form(shape, q, monkeypatch):
    cls, plus = q
    monkeypatch.delenv("PO2_STRICT", raising=False)
    g = torch.Generator().manual_seed(sum(shape) + int(plus))
    w = (torch.randn(shape, generator=g) * 0.07).to(BF)
    wd = w.cuda()
    for bits in (2, 4, 8):
        n0 = ops.LAUNCHES
        got = cls.forward(None, wd, bits=bits)
        assert ops.LAUNCHES == n0 + 1 and got.dtype == BF and got.shape == w.shape
        _check_channels(got, _op_by_op(w, bits, plus, monkeypatch), ("cpu", bits))
    # the op-by-op form on CUDA bf16 tensors, against the kernel under the torch_cuda flavor
    old = ops.get_log2_flavor()
    ops.set_log2_flavor("torch_cuda")
    try:
        for bits in (2, 4, 8):
            got = cls.forward(None, wd, bits=bits)
            _check_channels(got, _op_by_op(wd, bits, plus, monkeypatch), ("cuda", bits))
    finally:
        ops.set_log2_flavor(old)


def test_bf16_lin_quantizer_is_one_launch():
    from torch.profiler import ProfilerActivity, profile
    w = (torch.randn(64, 32, 3, 3, device="cuda") * 0.07).to(BF)
    P.LinearPowerOfTwoPlusQuantizer.forward(None, w, bits=4)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        P.LinearPowerOfTwoPlusQuantizer.forward(None, w, bits=4)
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert len(kernels) == 1 and "lin_quantize_kernel" in kernels[0], kernels


# ---- 2. NaN and constant channels ----------------------------------------------------------------------------------
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_bf16_lin_nan_and_constant_channels(q, monkeypatch):
    cls, plus = q
    w = (torch.randn(8, 4, 3, 3, generator=torch.Generator().manual_seed(2)) * 0.1).to(BF)
    w[:, 1] = 0.25                      # constant channel: step 0 -> 0/0 -> NaN in the reference too
    w[2, 2, 1, 1] = float("nan")        # NaN poisons its channel
    for bits in (2, 4, 8):
        ref = _op_by_op(w, bits, plus, monkeypatch)
        got = cls.forward(None, w.cuda(), bits=bits).cpu()
        assert torch.isnan(ref[:, 1]).all() and torch.isnan(ref[:, 2]).all()
        assert torch.equal(torch.isnan(got), torch.isnan(ref)), bits
        ok = ~torch.isnan(ref)
        assert torch.equal(got[ok].view(torch.int16), ref[ok].view(torch.int16)), bits


# ---- 3. fp32 is unchanged ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("plus", [0, 1], ids=LIN_IDS)
def test_lin_quantize_dt_f32_is_po2_lin_quantize(plus):
    lib = _lib.load()
    st = ops._stream_ptr(torch.device("cuda"))
    for K, C, R, S in SHAPES:
        w = torch.randn(K, C, R, S, device="cuda", generator=_gen("f32", K, C, R, S)) * 0.07
        for bits in (2, 4, 8, 16):
            a, b = torch.full_like(w, float("nan")), torch.full_like(w, float("nan"))
            _lib.check(lib.po2_lin_quantize(w.data_ptr(), a.data_ptr(), K, C, R * S, bits, 10, plus, ops._flavor, st),
                       "po2_lin_quantize")
            _lib.check(lib.po2_lin_quantize_dt(w.data_ptr(), b.data_ptr(), K, C, R * S, bits, 10, plus, ops._flavor,
                                               _lib.F32, st), "po2_lin_quantize_dt")
            torch.cuda.synchronize()
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (K, C, R, S, bits)


# ---- 4. conv exactness on lattice activations ---------------------------------------------------------------------
# (name, B, C, H, W, K, k, stride, groups, bf16 kernel kind): K3 3x3 s1 / s2 and 1x1, depthwise s1 / s2, small pointwise
CONV = [
    ("k3 3x3 s1", 4, 16, 16, 16, 32, 3, 1, 1, 2),
    ("k3 3x3 s2", 4, 16, 16, 16, 32, 3, 2, 1, 2),
    ("k3 1x1", 4, 32, 6, 6, 48, 1, 1, 1, 2),
    ("dw s1", 4, 32, 16, 16, 32, 3, 1, 32, 1),
    ("dw s2", 4, 24, 16, 16, 24, 3, 2, 24, 1),
    ("small pw", 4, 24, 4, 4, 40, 1, 1, 1, 4),
]


def _lin_ptq_layer(case, cls, bits):
    """a bf16 QuantizedConv2d post-training quantized with cls, and integer lattice activations in [-4, 4]"""
    name, B, C, H, W, K, k, stride, groups, kind = case
    gen = _gen(name, cls.__name__, bits)
    layer = P.QuantizedConv2d(C, K, k, stride=stride, padding=k // 2, groups=groups, bits=bits).cuda().to(BF)
    with torch.no_grad():
        layer.weight.copy_(torch.randn(layer.weight.shape, generator=gen, device="cuda") * 0.1)
    P.quantize_model(layer, cls, bits)
    assert layer.__dict__["_po2_lin_ptq"][0] == layer.weight._version
    x = torch.randint(-4, 5, (B, C, H, W), generator=gen, device="cuda").float()
    return layer, x


@pytest.mark.parametrize("bits", [4, 8])
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
@pytest.mark.parametrize("case", CONV, ids=lambda c: c[0])
def test_bf16_lin_layer_is_the_fp64_conv_rounded_once(case, q, bits, monkeypatch):
    """the products of a lattice x and a bf16 y are exact in fp32 and so is every partial sum (the steps of the input
    channels are a few binades apart at most): a correct kernel returns the fp64 conv rounded once to bf16"""
    cls, plus = q
    name, B, C, H, W, K, k, stride, groups, kind = case
    layer, x = _lin_ptq_layer(case, cls, bits)
    y = layer.weight.detach()
    assert y.dtype == BF
    ref = F.conv2d(x.double(), y.double(), None, stride, k // 2, 1, groups).float().to(BF)
    notes = _record_notes(monkeypatch)
    try:
        for mode in ("tc", "tf32"):
            ops.set_conv_mode(mode)
            assert ops.conv_kernel_kind(x.shape, y.shape, stride, k // 2, groups, ops.COMPUTE[mode], BF) == kind
            n0 = ops.LAUNCHES
            with torch.no_grad():
                out = layer(x.to(BF))
                again = layer(x.to(BF))
            assert ops.LAUNCHES > n0 and out.dtype == BF
            assert torch.equal(out, ref), (name, mode, (out != ref).sum().item())
            assert torch.equal(out.view(torch.int16), again.view(torch.int16))
            assert layer.__dict__["_po2_pack_cache"][0][5] == "lin"
    finally:
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
    assert not notes, notes


def _bf16_ulp(t):
    a = t.abs().to(BF)
    return (torch.nextafter(a.float(), torch.full_like(a.float(), float("inf"))).to(BF).float() - a.float()).clamp_min(2.0 ** -133)


@pytest.mark.parametrize("act", [0, 1, 2, 3], ids=["none", "relu", "relu6", "silu"])
@pytest.mark.parametrize("case", CONV, ids=lambda c: c[0])
def test_bf16_lin_layer_folded_epilogue(case, act, monkeypatch):
    """act(conv * a[k] + b[k] + residual), a = +-2^j, b on the 2^-8 grid, a bf16 integer residual: the pre-activation is
    exact in fp32, so the output is it rounded once to bf16 -- bit for bit, except SiLU (the kernel's __expf), within
    one bf16 ulp of the fp64 SiLU rounded to bf16"""
    name, B, C, H, W, K, k, stride, groups, kind = case
    layer, x = _lin_ptq_layer(case, P.LinearPowerOfTwoPlusQuantizer, 4)
    y = layer.weight.detach()
    gen = _gen(name, act)
    a = torch.exp2(torch.randint(-2, 3, (K,), generator=gen, device="cuda").float())
    a = a * (torch.randint(0, 2, (K,), generator=gen, device="cuda").float() * 2 - 1)
    b = torch.randint(-512, 513, (K,), generator=gen, device="cuda").float() * 2.0 ** -8
    conv = F.conv2d(x.double(), y.double(), None, stride, k // 2, 1, groups)
    res = torch.randint(-4, 5, conv.shape, generator=gen, device="cuda").double() if act != 2 else None
    pre = conv * a.double().view(1, -1, 1, 1) + b.double().view(1, -1, 1, 1)
    if res is not None:
        pre = pre + res
    assert pre.abs().max().item() < 2 ** 12
    if act == 3:
        ref = F.silu(pre).float().to(BF)
    else:
        ref = [lambda t: t, torch.relu, lambda t: t.clamp(0, 6)][act](pre).float().to(BF)
    resb = res.to(BF) if res is not None else None
    notes = _record_notes(monkeypatch)
    try:
        for mode in ("tc", "tf32"):
            ops.set_conv_mode(mode)
            with torch.no_grad():
                out = layer.forward_folded(x.to(BF), a, b, resb, act)
            assert out is not None and out.dtype == BF and not out.isnan().any(), (name, mode)
            if act == 3:
                assert ((out.float() - ref.float()).abs() <= _bf16_ulp(ref)).all(), (name, mode)
            else:
                assert torch.equal(out, ref), (name, mode, (out != ref).sum().item())
    finally:
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
    assert not notes, notes


# ---- 5. whole models -----------------------------------------------------------------------------------------------
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


@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
@pytest.mark.parametrize("fold", [False, True], ids=["separate", "folded"])
@pytest.mark.parametrize("family", ["resnet20", "mobilenet", "mobilevit"])
def test_bf16_lin_ptq_models_run_on_our_kernels(family, fold, q, monkeypatch):
    """bf16 lin / lin+ PTQ inference, as tests/test_bf16_inference_gpu.py holds PO2+: cast to bf16 first, then
    quantize_model.  No QuantizedConv2d and no quantizer leaves our kernels; the logits are within 3 * n_layers * 2^-8
    of the logit scale of the same bf16 model on cuDNN and top-1 agrees where the reference's margin exceeds that; tc
    and tf32 give the same bits (bf16 operands in both), and so do a CUDA-graph replay and a deep copy of the model."""
    cls, plus = q
    m, x, bits = _model(family)
    m, x = m.cuda().to(BF).eval(), x.cuda().to(BF)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
                mod.running_mean.normal_(0, 0.2); mod.running_var.uniform_(0.5, 1.5)
                mod.weight.uniform_(0.7, 1.3); mod.bias.normal_(0, 0.1)
    notes = _record_notes(monkeypatch)
    P.quantize_model(m, cls, bits)
    n_layers = sum(isinstance(mod, P.QuantizedConv2d) for mod in m.modules())
    if fold:
        assert P.fold_conv_bn(m) > 0 or family == "resnet20"
    monkeypatch.setenv("PO2_FOLD_BN", "1" if fold else "0")
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
            mc = copy.deepcopy(m)
            copied = mc(x)
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
    assert not [k for k in notes if k.startswith(("qconv:", "lin:"))], notes
    assert out.dtype == BF and launches >= n_layers // 2
    for c in (m, mc):
        lin = [mod for mod in c.modules() if isinstance(mod, P.QuantizedConv2d)]
        assert all(mod.__dict__["_po2_pack_cache"][0][5] == "lin" for mod in lin)
    assert torch.equal(out.view(torch.int16), again.view(torch.int16))
    assert torch.equal(out.view(torch.int16), out_tc.view(torch.int16))
    assert torch.equal(captured.view(torch.int16), out.view(torch.int16))
    assert torch.equal(copied.view(torch.int16), out.view(torch.int16))
    tol = 3 * n_layers * 2.0 ** -8
    scale = ref.abs().max()
    rel = ((out.float() - ref).abs().max() / scale).item()
    assert rel <= tol, (rel, tol)
    top = ref.topk(2, dim=1).values
    decisive = (top[:, 0] - top[:, 1]) > tol * scale
    assert torch.equal(out.float().argmax(1)[decisive], ref.argmax(1)[decisive])
    print(f"{family} {LIN_IDS[plus]} fold={fold}: rel {rel:.3e} (bound {tol:.3e}), {launches} launches")


# ---- 6. a QAT layer in eval ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
@pytest.mark.parametrize("k,stride,groups", [(3, 1, 1), (3, 2, 1), (3, 1, 32), (1, 1, 1)], ids=["k3", "k3-s2", "dw", "pw"])
def test_bf16_lin_qat_layer_in_eval_quantizes_in_bf16(k, stride, groups, q, monkeypatch):
    """A lin / lin+ QAT layer of a bf16 model under no_grad: its bf16 weight is quantized by the bf16 lin kernel and
    the conv runs on our kernels -- the same bits as the layer post-training quantized with quantize_model; a changed
    weight is re-quantized (the cache follows the weight's version)."""
    cls, plus = q
    torch.manual_seed(11)
    H = 2 if k == 1 else 16                            # 1x1 on a 2x2 map: the small-pointwise GEMM
    qat = P.QuantizedConv2d(32, 32, k, stride=stride, padding=k // 2, groups=groups, quantize_fn=cls, bits=4).cuda().to(BF)
    ptq = P.QuantizedConv2d(32, 32, k, stride=stride, padding=k // 2, groups=groups, bits=4).cuda().to(BF)
    x = torch.randn(8, 32, H, H, device="cuda").to(BF)
    notes = _record_notes(monkeypatch)
    for step in range(2):
        with torch.no_grad():
            ptq.weight.copy_(qat.weight)
        P.quantize_model(ptq, cls, 4)
        n0 = ops.LAUNCHES
        with torch.no_grad():
            out, ref = qat(x), ptq(x)
        assert ops.LAUNCHES > n0 and out.dtype == BF
        assert torch.equal(cls.forward(None, qat.weight.detach(), bits=4), ptq.weight)
        assert torch.equal(out.view(torch.int16), ref.view(torch.int16)), step
        with torch.no_grad():
            qat.weight.mul_(-0.5)
    assert not notes, notes


# ---- 7. a bf16 lin layer that needs a gradient ---------------------------------------------------------------------
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_bf16_lin_layer_with_a_gradient_keeps_the_stock_conv(q, monkeypatch):
    cls, plus = q
    notes = _record_notes(monkeypatch)
    torch.backends.cudnn.deterministic = True
    try:
        torch.manual_seed(13)
        qat = P.QuantizedConv2d(16, 32, 3, quantize_fn=cls, bits=4).cuda().to(BF)
        ptq = copy.deepcopy(qat)
        ptq.quantize_fn = None
        P.quantize_model(ptq, cls, 4)
        x = torch.randn(4, 16, 16, 16, device="cuda").to(BF)
        for layer in (qat, ptq):
            notes.clear()
            xa = x.clone().requires_grad_(True)
            out = layer(xa)
            assert any(key.startswith("qconv:dtype") for key in notes), notes
            y = cls.forward(None, qat.weight.detach(), bits=4)
            assert torch.equal(out, F.conv2d(x, y, None, 1, 1))
            out.float().square().mean().backward()
            assert xa.grad is not None and layer.weight.grad is not None
            assert torch.isfinite(layer.weight.grad).all()
    finally:
        torch.backends.cudnn.deterministic = False
