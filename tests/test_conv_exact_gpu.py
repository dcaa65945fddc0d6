"""Every conv kernel, bit for bit, on operands whose sums are exact.

x and the output gradient are small integers in [-4, 4]; weights are +-s * 2^q with s = 2^-3 and q on the 4-bit PO2 grid
(fsr 1: q in [-7, 0]), with exact zeros -- what po2::quantize_scaled returns for them.  Every product and partial sum is
then a multiple of 2^-10 below 2^23 such steps (tests/test_conv_exact_cpu.py checks the bound for each case), exact in
fp32 and in the bf16 / tf32 operand formats, so a correct kernel returns F.conv2d in fp64, rounded once to fp32, bit for
bit, whatever its summation order or tiling.  A dropped, duplicated or misplaced term shows at any single output.
Each case also checks the kernel kind the case names, a bit-identical second call, and (output pre-filled with NaN)
that every output element is written.  The case table lives in tests/test_conv_exact_cpu.py."""
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import po2_quantization_b200  # noqa: E402,F401  (registers torch.ops.po2.*)
from po2_quantization_b200 import _lib, ops  # noqa: E402

from tests.test_conv_exact_cpu import (DEPTHWISE, DGRAD, FWD, STEM, STRIDE2, WGRAD, dgrad_exact, fwd_exact,  # noqa: E402
                                       out_hw, wgrad_exact)

S_W = 2.0 ** -3
NAN = float("nan")


def _gen(*key):
    return torch.Generator(device="cuda").manual_seed(zlib.crc32(repr(key).encode()))


def lattice_x(shape, gen):
    return torch.randint(-4, 5, shape, generator=gen, device="cuda").float()


def lattice_w(shape, gen, s=S_W):
    """+-s * 2^q, q in [-7, 0], about one in eight exactly zero, the first entry s (so that max |w| = s)"""
    q = torch.randint(-7, 1, shape, generator=gen, device="cuda").float()
    sign = torch.randint(0, 2, shape, generator=gen, device="cuda").float() * 2 - 1
    keep = (torch.randint(0, 8, shape, generator=gen, device="cuda") != 0).float()
    w = sign * torch.exp2(q) * keep * s
    w.view(-1)[0] = s
    return w


def quantized_lattice_w(shape, gen):
    """lattice weights and their scale, checked to be a fixed point of the 4-bit PO2 quantizer"""
    w = lattice_w(shape, gen)
    y, scale = torch.ops.po2.quantize_scaled(w, 4, 1, False)
    assert torch.equal(y, w) and scale.item() == S_W
    return w, scale


def nan_like(shape):
    return torch.full(shape, NAN, device="cuda")


def _fwd_ref(x, w, stride, pad, groups):
    return F.conv2d(x.double(), w.double(), None, stride, pad, 1, groups).float()


def _fwd_operands(case):
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    gen = _gen(name)
    x = lattice_x((B, C, H, W), gen)
    w, scale = quantized_lattice_w((K, C // groups, k, k), gen)
    return x, w, scale


# ---- forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", FWD, ids=lambda c: c[0])
def test_forward_is_bit_exact_through_every_entry_point(case):
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    pad = k // 2
    assert fwd_exact(C, k, groups)
    lib = _lib.load()
    assert lib.po2_conv2d_kernel_kind(B, C, H, W, K, k, k, stride, pad, groups, compute) == kind, name
    x, w, scale = _fwd_operands(case)
    ref = _fwd_ref(x, w, stride, pad, groups)
    outs = {}
    for run in range(2):
        out = nan_like(ref.shape)
        ops.conv2d_out(x, w, scale, out, stride, pad, groups, compute)
        outs[run] = out
    assert torch.equal(outs[0], ref), (name, (outs[0] != ref).sum().item())
    assert torch.equal(outs[0], outs[1]), name
    # packed sign + exponent codes: the decode kernel (kinds 0, 1, 4) or the pack kernel (2, 3) rebuilds the weight.
    # A zero has no code of its own and is emitted as (+, lowest level) (include/po2_b200.h, po2_quantize)
    y, codes, sc, zc, sse = torch.ops.po2.quantize_full(w, 4, 1, False)
    assert torch.equal(y, w) and zc.item() == (w == 0).sum().item()
    out = nan_like(ref.shape)
    ops.conv2d_out(x, codes, sc, out, stride, pad, groups, compute, w_format=_lib.W_CODES, bits=4, fsr=1,
                   wshape=tuple(w.shape))
    ref_codes = _fwd_ref(x, torch.where(w == 0, S_W * 2.0 ** -7, w), stride, pad, groups)
    assert torch.equal(out, ref_codes), (name, "codes", (out != ref_codes).sum().item())
    assert torch.equal(torch.ops.po2.conv2d(x, w, scale, stride, pad, groups, compute), ref), (name, "op")
    # the fused quantize (+ pack) + conv
    out, qw, qs = torch.ops.po2.qconv2d(x, w, 4, 1, False, stride, pad, groups, compute)
    assert torch.equal(qw, w) and torch.equal(out, ref), (name, "qconv2d")
    packed = ops.conv2d_pack(w, scale, x.shape, stride, pad, groups, compute)
    assert (packed is not None) == (kind in (2, 3)), name
    if packed is not None:
        out = torch.ops.po2.conv2d_packed(x, packed, scale, K, k, k, stride, pad, groups, compute)
        assert torch.equal(out, ref), (name, "packed")


EP_CASES = [c for c in FWD if c[0] in (
    "direct grouped 16->32 g4 @8", "dw vec s1 32 @16", "dw scalar 7 @9x7", "k3 3x3 s1 24->40 @14x9",
    "k3 3x3 s2 16->32 @16", "k3 1x1 s1 32->48 @6", "k3 3x3 32->300 @8 (N tiles)", "k3 3x3 256->32 @8 (chunks)",
    "k3 resnet 16->16 @32 B=128", "k3t mode0 16->16 @32", "k3t mode4 32->32 @8", "k3t 1x1 32->64 @8",
    "pw split 576->160 @1", "pw single 24->40 @4x4")]


def _ulp(t):
    a = t.abs()
    return torch.nextafter(a, torch.full_like(a, float("inf"))) - a


@pytest.mark.parametrize("act", [0, 1, 2, 3], ids=["none", "relu", "relu6", "silu"])
@pytest.mark.parametrize("compute", [0, 2], ids=["bf16", "tf32"])
@pytest.mark.parametrize("case", EP_CASES, ids=lambda c: c[0])
def test_epilogue_is_bit_exact(case, compute, act):
    """act(conv * a[k] + b[k] + residual) with a = +-2^j, b on the 2^-8 grid and an integer residual: exact in fp32, so
    bit for bit -- except SiLU, the one inexact activation, against torch's fp32 SiLU of the exact pre-activation"""
    name, B, C, H, W, K, k, stride, groups, _, kind, branches = case
    pad = k // 2
    x, w, scale = _fwd_operands(case)
    gen = _gen(name, compute, act)
    a = torch.exp2(torch.randint(-2, 3, (K,), generator=gen, device="cuda").float())
    a = a * (torch.randint(0, 2, (K,), generator=gen, device="cuda").float() * 2 - 1)
    b = torch.randint(-512, 513, (K,), generator=gen, device="cuda").float() * 2.0 ** -8
    conv = F.conv2d(x.double(), w.double(), None, stride, pad, 1, groups)
    res = lattice_x(conv.shape, gen) if act != 2 else None
    pre = conv * a.double().view(1, -1, 1, 1) + b.double().view(1, -1, 1, 1)
    if res is not None:
        pre = pre + res.double()
    assert pre.abs().max().item() < 2 ** 12       # a multiple of 2^-12: exact in fp32 at every step
    pre = pre.float()
    out = torch.ops.po2.conv2d_ep(x, w, scale, stride, pad, groups, compute, a, b, res, act)
    if act == 3:
        ref = F.silu(pre)
        # __expf is within 2 + floor(1.173 |v|) ulp (CUDA C Programming Guide); one more for 1 + e and the division,
        # one for torch's own SiLU
        tol = (4 + torch.floor(1.173 * pre.abs())) * _ulp(ref)
        assert ((out - ref).abs() <= tol).all(), (name, ((out - ref).abs() / _ulp(ref)).max().item())
    else:
        ref = [lambda t: t, torch.relu, lambda t: t.clamp(0, 6)][act](pre)
        assert torch.equal(out, ref), (name, (out != ref).sum().item())
    packed = ops.conv2d_pack(w, scale, x.shape, stride, pad, groups, compute)
    if packed is not None:
        out2 = torch.ops.po2.conv2d_packed_ep(x, packed, scale, K, k, k, stride, pad, groups, compute, a, b, res, act)
        assert torch.equal(out, out2), (name, "packed")


SCALE_CASES = [c for c in FWD if c[0] in (
    "direct 5x5 8->8 @12", "dw vec s1 32 @16", "k3 3x3 s2 16->32 @16", "k3 3x3 256->32 @8 (chunks)",
    "k3 tf32 3x3 16->16 @12", "k3t mode0 24->40 @20x24", "k3t 1x1 32->64 @8", "pw split 576->160 @1")]


@pytest.mark.parametrize("case", SCALE_CASES, ids=lambda c: c[0])
def test_non_dyadic_scale_is_applied_once_after_accumulation(case):
    """w = +-1.337 * 2^q: the tensor-core kernels (2, 3) convolve with +-2^q and multiply the fp32 sum by the scale once,
    so out == fp32(exact sum) * 1.337f bit for bit.  Kinds 0, 1 and 4 multiply by the fp32 weight itself (products
    rounded in fp32): there the fp32-accumulate tolerance."""
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    pad = k // 2
    x, w, _ = _fwd_operands(case)
    s = torch.tensor(1.337, dtype=torch.float32, device="cuda")
    unit = w / S_W                                  # +-2^q, exact
    ws = unit * s                                   # +-1.337f * 2^q, exact
    out = torch.ops.po2.conv2d(x, ws, s, stride, pad, groups, compute)
    if kind in (2, 3):
        ref = _fwd_ref(x, unit, stride, pad, groups) * s
        assert torch.equal(out, ref), (name, (out != ref).sum().item())
    else:
        ref = F.conv2d(x.double(), ws.double(), None, stride, pad, 1, groups)
        assert ((out.double() - ref).abs().max() / ref.abs().max()).item() < 1e-5, name


# ---- backward --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", DGRAD, ids=lambda c: c[0])
def test_dgrad_is_bit_exact(case):
    name, B, C, H, W, K, k, compute, packed = case
    pad = k // 2
    assert dgrad_exact(K, k)
    lib = _lib.load()
    gen = _gen(name)
    g = lattice_x((B, K, H, W), gen)
    w, scale = quantized_lattice_w((K, C, k, k), gen)
    ref = torch.nn.grad.conv2d_input((B, C, H, W), w.double(), g.double(), stride=1, padding=pad).float()
    gx = nan_like(ref.shape)
    assert ops.conv2d_dgrad_out(g, w, scale, gx, pad, compute)
    assert torch.equal(gx, ref), (name, (gx != ref).sum().item())
    gx2 = nan_like(ref.shape)
    assert ops.conv2d_dgrad_out(g, w, scale, gx2, pad, compute)
    assert torch.equal(gx, gx2), name
    if not packed:
        return
    # the operand the multi-descriptor quantizer (weight prefetch) emits for the data gradient
    qw, qs = torch.empty_like(w), torch.empty((), device="cuda")
    fwd = torch.empty(int(lib.po2_conv2d_pack_bytes(B, C, H, W, K, k, k, 1, pad, 1, compute)), dtype=torch.uint8,
                      device="cuda")
    pd = torch.empty(int(lib.po2_conv2d_dgrad_pack_bytes(B, C, H, W, K, k, k, pad, compute)), dtype=torch.uint8,
                     device="cuda")
    sse = torch.zeros((), dtype=torch.float64, device="cuda")
    host = torch.zeros(int(lib.po2_multi_desc_bytes()), dtype=torch.uint8)
    csize = lib.po2_multi_desc_fill(host.data_ptr(), 0, w.data_ptr(), qw.data_ptr(), qs.data_ptr(), fwd.data_ptr(),
                                    fwd.numel(), B, C, H, W, K, k, k, 1, pad, 1, 4, 1, 0, ops._flavor, compute,
                                    sse.data_ptr())
    assert csize > 0, (name, csize)
    assert lib.po2_multi_desc_fill_dgrad(host.data_ptr(), 0, pd.data_ptr(), pd.numel(), B, C, H, W, K, k, k, 1, pad, 1,
                                         compute) == 0
    table = host.cuda()
    _lib.check(lib.po2_quantize_pack_multi(table.data_ptr(), 1, csize, ops._stream_ptr(table.device)), "multi")
    gx3 = nan_like(ref.shape)
    ops.conv2d_dgrad_packed_out(g, pd, qs, gx3, w.shape, pad, compute)
    assert torch.equal(qw, w) and torch.equal(gx3, gx), (name, "multi-descriptor operand")
    x = lattice_x((B, C, H, W), gen)               # and the forward operand of the same launch
    out = torch.ops.po2.conv2d_packed(x, fwd, qs, K, k, k, 1, pad, 1, compute)
    assert torch.equal(out, _fwd_ref(x, w, 1, pad, 1)), (name, "multi-descriptor forward operand")


@pytest.mark.parametrize("case", WGRAD, ids=lambda c: c[0])
def test_wgrad_is_bit_exact(case):
    name, B, C, H, W, K, k, compute, kind, branches = case
    pad = k // 2
    assert wgrad_exact(B, H, W)
    assert _lib.load().po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, k, k, 1, pad, 1, compute) == kind, name
    gen = _gen(name)
    x = lattice_x((B, C, H, W), gen)
    g = lattice_x((B, K, H, W), gen)
    ref = torch.nn.grad.conv2d_weight(x.double(), (K, C, k, k), g.double(), stride=1, padding=pad).float()
    gw = nan_like(ref.shape)
    assert ops.conv2d_wgrad_out(g, x, gw, pad, compute)
    assert torch.equal(gw, ref), (name, (gw != ref).sum().item())
    gw2 = nan_like(ref.shape)
    assert ops.conv2d_wgrad_out(g, x, gw2, pad, compute)
    assert torch.equal(gw, gw2), name


@pytest.mark.parametrize("shape", STEM, ids=lambda s: "x".join(map(str, s)))
def test_stem_wgrad_is_bit_exact(shape):
    B, C, H, W, K = shape
    lib = _lib.load()
    gen = _gen("stem", shape)
    x = lattice_x((B, C, H, W), gen)
    g = lattice_x((B, K, H, W), gen)
    ref = torch.nn.grad.conv2d_weight(x.double(), (K, C, 3, 3), g.double(), stride=1, padding=1).float()
    ws = torch.empty(int(lib.po2_conv2d_stem_wgrad_workspace(B, C, H, W, K, 3, 3, 1, 1, 1)), dtype=torch.uint8,
                     device="cuda")
    assert ws.numel() > 0
    for _ in range(2):
        gw = nan_like(ref.shape)
        _lib.check(lib.po2_conv2d_stem_wgrad(g.data_ptr(), x.data_ptr(), gw.data_ptr(), B, C, H, W, K, 3, 3, 1, 1, 1,
                                             ws.data_ptr(), ws.numel(), ops._stream_ptr(x.device)), "stem wgrad")
        assert torch.equal(gw, ref), shape


def _autograd_exact(name, x, w, scale, stride, pad, groups, compute, g, offset=False):
    """x.grad and w.grad of torch.ops.po2.conv2d against fp64 autograd, bit for bit, on our kernels only.
    offset: x and the output gradient are contiguous views 4 bytes past a 16-byte boundary"""
    n = x.numel()
    buf = torch.zeros(n + 4, device="cuda")
    lo = 1 if offset else 0
    buf[lo:lo + n] = x.reshape(-1)
    buf.requires_grad_(True)
    xr, wr = buf[lo:lo + n].view(x.shape), w.detach().clone().requires_grad_(True)
    if offset:
        g = _offset_view(g)
        assert xr.data_ptr() % 16 == 4
    ops._noted.discard("conv_backward_aten")
    out = torch.ops.po2.conv2d(xr, wr, scale, stride, pad, groups, compute)
    out.backward(g)
    assert "conv_backward_aten" not in ops._noted, (name, "the backward fell back to aten.convolution_backward")
    gx = buf.grad[lo:lo + n].view(x.shape)
    xd, wd = x.detach().double().requires_grad_(True), w.detach().double().requires_grad_(True)
    ref = F.conv2d(xd, wd, None, stride, pad, 1, groups)
    ref.backward(g.double())
    assert torch.equal(out, ref.float()), (name, "forward")
    assert torch.equal(gx, xd.grad.float()), (name, "dx", (gx != xd.grad.float()).sum().item())
    assert torch.equal(wr.grad, wd.grad.float()), (name, "dw", (wr.grad != wd.grad.float()).sum().item())
    return out, gx, wr.grad


@pytest.mark.parametrize("case", DEPTHWISE, ids=lambda c: c[0])
def test_depthwise_backward_is_bit_exact(case):
    name, B, C, H, W, stride = case
    gen = _gen(name)
    x = lattice_x((B, C, H, W), gen)
    w, scale = quantized_lattice_w((C, 1, 3, 3), gen)
    P, Q = out_hw(H, W, 3, stride)
    _autograd_exact(name, x, w, scale, stride, 1, C, 2, lattice_x((B, C, P, Q), gen))


@pytest.mark.parametrize("compute", [0, 2], ids=["bf16", "tf32"])
@pytest.mark.parametrize("case", STRIDE2, ids=lambda c: c[0])
def test_stride2_backward_through_dilate2_is_bit_exact(case, compute):
    name, B, C, H, W, K, k = case
    gen = _gen(name, compute)
    x = lattice_x((B, C, H, W), gen)
    w, scale = quantized_lattice_w((K, C, k, k), gen)
    P, Q = out_hw(H, W, k, 2)
    _autograd_exact(name, x, w, scale, 2, k // 2, 1, compute, lattice_x((B, K, P, Q), gen))


# ---- operand rounding ------------------------------------------------------------------------------------------------
def _off_lattice(shape, gen, mant_bits):
    """+-(n + 0.75 ulp(n)), n in 1..4 (ulp with `mant_bits` explicit mantissa bits), and zeros: exactly representable in
    fp32, rounded up in magnitude by round-to-nearest, down by truncation"""
    n = torch.randint(0, 5, shape, generator=gen, device="cuda").float()
    sign = torch.randint(0, 2, shape, generator=gen, device="cuda").float() * 2 - 1
    ulp = torch.exp2(torch.floor(torch.log2(n.clamp(min=1))) - mant_bits)
    return sign * torch.where(n > 0, n + 0.75 * ulp, n)


def _truncate_tf32(t):
    return (t.view(torch.int32) & ~0x1FFF).view(torch.float32)


def _round_tf32(t):
    return ((t.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


ROUND_CASES = {c[0]: c for c in FWD}


@pytest.mark.parametrize("name", ["k3 3x3 s1 16->16 @16", "k3 3x3 s1 24->40 @14x9", "k3 1x1 s1 32->48 @6",
                                  "k3 3x3 s2 16->32 @16"])
def test_bf16_operands_round_to_nearest_even(name):
    """compute 0: the producers convert x with __floats2bfloat162_rn, so the output is the conv of x.bfloat16()"""
    _, B, C, H, W, K, k, stride, groups, compute, kind, branches = ROUND_CASES[name]
    gen = _gen("bf16", name)
    x = _off_lattice((B, C, H, W), gen, 7)
    w = S_W * (torch.randint(0, 2, (K, C, k, k), generator=gen, device="cuda").float() * 2 - 1)
    assert k * k * C * 2 ** 9 < 2 ** 23          # products below 2^-1 in steps of 2^-10
    xb = x.bfloat16().float()
    assert not torch.equal(xb, (x.view(torch.int32) & ~0xFFFF).view(torch.float32))
    out = torch.ops.po2.conv2d(x, w, torch.tensor(S_W, device="cuda"), stride, k // 2, 1, 0)
    assert torch.equal(out, _fwd_ref(xb, w, stride, k // 2, 1)), name


@pytest.mark.parametrize("name", ["k3 tf32 3x3 16->16 @12", "k3 tf32 3x3 s2 16->32 @16", "k3t mode4 16->32 @16",
                                  "k3t mode0 16->16 @32", "k3t 1x1 32->64 @8"])
def test_tf32_operands_are_truncated(name):
    """compute 2: x reaches the tensor core as fp32 bits (registers or TMA) and the tensor core ignores the low 13
    mantissa bits, so the output is the conv of x truncated to tf32 -- not rounded"""
    _, B, C, H, W, K, k, stride, groups, compute, kind, branches = ROUND_CASES[name]
    assert _lib.load().po2_conv2d_kernel_kind(B, C, H, W, K, k, k, stride, k // 2, 1, 2) == kind
    gen = _gen("tf32", name)
    x = _off_lattice((B, C, H, W), gen, 10)
    w = S_W * (torch.randint(0, 2, (K, C, k, k), generator=gen, device="cuda").float() * 2 - 1)
    assert k * k * C * 2 ** 12 < 2 ** 23         # products below 2^-1 in steps of 2^-13
    out = torch.ops.po2.conv2d(x, w, torch.tensor(S_W, device="cuda"), stride, k // 2, 1, 2)
    trunc, rn = _fwd_ref(_truncate_tf32(x), w, stride, k // 2, 1), _fwd_ref(_round_tf32(x), w, stride, k // 2, 1)
    assert not torch.equal(trunc, rn)
    assert torch.equal(out, trunc), (name, "matches round-to-nearest" if torch.equal(out, rn) else "matches neither")


def test_tf32_weight_gradient_operands_are_truncated():
    """K5T reads x and the output gradient as fp32 through tensor maps: the same truncation"""
    B, C, H, W, K = 2, 8, 8, 8, 16
    assert _lib.load().po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, 3, 3, 1, 1, 1, 2) == 2
    gen = _gen("tf32 wgrad")
    x = _off_lattice((B, C, H, W), gen, 10)
    g = lattice_x((B, K, H, W), gen)
    assert 16 * 2 ** 10 * B * H * W < 2 ** 23     # products below 2^4 in steps of 2^-10
    gw = nan_like((K, C, 3, 3))
    assert ops.conv2d_wgrad_out(g, x, gw, 1, 2)
    wref = lambda xx: torch.nn.grad.conv2d_weight(xx.double(), (K, C, 3, 3), g.double(), stride=1, padding=1).float()
    trunc, rn = wref(_truncate_tf32(x)), wref(_round_tf32(x))
    assert not torch.equal(trunc, rn)
    assert torch.equal(gw, trunc), "matches round-to-nearest" if torch.equal(gw, rn) else "matches neither"


# ---- storage offsets -------------------------------------------------------------------------------------------------
def _offset_view(t):
    """a contiguous copy of t that starts 4 bytes past a 16-byte boundary"""
    buf = torch.empty(t.numel() + 4, device="cuda")
    assert buf.data_ptr() % 16 == 0
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v


OFFSET_FWD = [c for c in FWD if c[0] in (
    "direct grouped 16->32 g4 @8", "dw vec s1 32 @16", "dw scalar 7 @9x7", "k3 3x3 s1 16->16 @16",
    "k3 1x1 s1 32->48 @6", "k3 3x3 32->32 @1x1 (hw1)", "k3 tf32 3x3 16->16 @12", "k3t mode0 16->16 @32",
    "k3t mode4 32->32 @8", "k3t 1x1 32->64 @8", "pw split 576->160 @1", "pw single 24->40 @4x4")]


@pytest.mark.parametrize("case", OFFSET_FWD, ids=lambda c: c[0])
def test_forward_takes_inputs_at_any_storage_offset(case):
    """x (and, for the pointwise GEMM, w) as contiguous views 4 bytes past a 16-byte boundary give the aligned result
    through every op; the raw library call refuses such an x where its kernel reads x with 128-bit loads"""
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    pad = k // 2
    x, w, scale = _fwd_operands(case)
    xv, wv = _offset_view(x), _offset_view(w)
    ref = torch.ops.po2.conv2d(x, w, scale, stride, pad, groups, compute)
    assert torch.equal(torch.ops.po2.conv2d(xv, wv, scale, stride, pad, groups, compute), ref), name
    assert torch.equal(torch.ops.po2.qconv2d(xv, wv, 4, 1, False, stride, pad, groups, compute)[0], ref), name
    a, b = torch.ones(K, device="cuda"), torch.zeros(K, device="cuda")
    assert torch.equal(torch.ops.po2.conv2d_ep(xv, wv, scale, stride, pad, groups, compute, a, b, None, 0), ref), name
    if kind in (2, 3):
        packed = ops.conv2d_pack(w, scale, x.shape, stride, pad, groups, compute)
        assert torch.equal(torch.ops.po2.conv2d_packed(xv, packed, scale, K, k, k, stride, pad, groups, compute), ref)
        assert torch.equal(torch.ops.po2.conv2d_packed_ep(xv, packed, scale, K, k, k, stride, pad, groups, compute, a, b,
                                                          None, 0), ref)
        if "scalar" not in branches:
            with pytest.raises(_lib.Po2Error):
                ops.conv2d_out(xv, w, scale, torch.empty_like(ref), stride, pad, groups, compute)


# (name, B, C, H, W, K, k, stride, compute): dgrad on K3 transposed; wgrad on K5 (bf16), K5T (tf32), the pointwise
# GEMM (1x1 wide); the stride-2 route through po2_dilate2; a depthwise layer
OFFSET_BWD = [("k3 / k5 3x3 16->16 @16", 4, 16, 16, 16, 16, 3, 1, 0), ("k3t / k5t 3x3 16->16 @16", 4, 16, 16, 16, 16, 3, 1, 2),
              ("pw wgrad 64->384 @2", 16, 64, 2, 2, 384, 1, 1, 2), ("s2 3x3 16->32 @16", 4, 16, 16, 16, 32, 3, 2, 2),
              ("dw 32 @16", 4, 32, 16, 16, 32, 3, 1, 2)]


@pytest.mark.parametrize("case", OFFSET_BWD, ids=lambda c: c[0])
def test_backward_takes_inputs_at_any_storage_offset(case):
    name, B, C, H, W, K, k, stride, compute = case
    groups = C if name.startswith("dw") else 1
    gen = _gen(name)
    x = lattice_x((B, C, H, W), gen)
    w, scale = quantized_lattice_w((K, C // groups, k, k), gen)
    P, Q = out_hw(H, W, k, stride)
    g = lattice_x((B, K, P, Q), gen)
    aligned = _autograd_exact(name, x, w, scale, stride, k // 2, groups, compute, g)
    offset = _autograd_exact(name, x, w, scale, stride, k // 2, groups, compute, g, offset=True)
    for a, b in zip(aligned, offset):
        assert torch.equal(a, b), name


# ---- coverage --------------------------------------------------------------------------------------------------------
K3_BRANCHES = {"vec4", "scalar", "hw1", "s2", "flat", "cpad", "nchunk", "ntiles", "ntail", "mloop"}


def test_case_table_covers_every_kernel_kind_and_k3_branch():
    """A later edit of the case table cannot quietly drop a kernel or a K3 branch: every forward kind 0-4, every
    weight-gradient kind 1-3, each K3 branch in bf16, K3 in tf32, the three K3T forms and both forms of the depthwise and
    pointwise kernels have a case (each case asserts its kind on the device)."""
    seen = sorted({(kind, compute, br) for _, _, _, _, _, _, _, _, _, compute, kind, brs in FWD for br in brs or ("-",)})
    print("\nforward (kind, compute, branch):", seen)
    print("wgrad (kind, compute, branch):",
          sorted({(kind, compute, br) for _, _, _, _, _, _, _, compute, kind, brs in WGRAD for br in brs or ("-",)}))
    assert {c[10] for c in FWD} == {0, 1, 2, 3, 4}
    assert {c[8] for c in WGRAD} == {1, 2, 3}
    k3_bf16 = {br for c in FWD if c[10] == 2 and c[9] == 0 for br in c[11]}
    assert K3_BRANCHES <= k3_bf16, K3_BRANCHES - k3_bf16
    assert any(c[10] == 2 and c[9] == 2 for c in FWD)
    assert {br for c in FWD if c[10] == 3 for br in c[11]} == {"mode0", "mode4", "mode1"}
    assert {br for c in FWD if c[10] == 1 for br in c[11]} == {"vec", "scalar"}
    assert {br for c in FWD if c[10] == 4 for br in c[11]} == {"split", "single"}
    assert {br for c in WGRAD if c[8] == 2 for br in c[9]} >= {"merged", "runs", "rsplit"}
    assert any(c[7] == 0 for c in DGRAD) and any(c[7] == 2 for c in DGRAD) and any(c[8] for c in DGRAD)
    assert {c[6] for c in DGRAD} == {1, 3}
